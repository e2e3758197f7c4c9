"""fk_system_batch_solve_single_pass (System.batch_solve_single_pass) on one B200: System::solve with Decomposer::SinglePass
over n variants of one drawing in one call, against the per-variant System.solve_single_pass loop a design-table sweep runs
without it, and the oracle's SinglePass on one core.

    python tools/bench_system_batch_single_pass.py [--out FILE] [--passes K] [--quick]

Drawings: (a) 16 hinged chains of 4 triangles + 4 circle_triangle_line + one 20-point truss, 65,536 variants; (b) a 30x20
lattice + 8 triangles, 1,024 variants; (c) an 80x60 lattice, 256 variants (fk_system_batch_solve refuses it with LM: its
largest supernodal front has 260 rows).  Variants as in tools/bench_system_batch.py.  Per drawing:
- the plan: sets, waves, structures, and launches per chunk (one prepare, one gather / scatter per wave and one more, one LM
  launch per structure present in a wave);
- end to end: the host clock around the call, from pageable numpy arrays and from pinned buffers (fk_host_alloc), one
  warm-up call first, medians of --passes passes;
- device time split: one extra call under torch.profiler (CUDA activity): prepare kernel, gather / scatter kernel, solve
  launches (everything else), and the gaps between kernels on the stream;
- the per-variant loop (set the variant's numbers, System.solve_single_pass, read the variables) over a sample;
- the oracle's System.solve_single_pass on one core over a sample;
- for context, fk_system_batch_solve (Decomposer::None, LM) on (a) and (b): a different algorithm with different results.
The card's name and power limit are read in the same call.  Anything not run is written as "not measured".
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
from bench_system_batch import _add_ppd, _recording, call, drawing_a, drawing_b, pinned, timed, variants  # noqa: E402

import fiksi_b200 as fk  # noqa: E402
from fiksi_b200 import workloads as wl  # noqa: E402
from fiksi_b200._lib import FkReport, lib  # noqa: E402

REPO = os.path.dirname(ROOT)


def drawing_c(S):
    s = _recording(S)()
    _add_ppd(s, wl.lattice(80, 60))
    return s


def call_sp(s, vars_, params, out, reps):
    got = C.c_uint32(0)
    fk._lib.check(lib().fk_system_batch_solve_single_pass(
        s._h, 1, len(vars_), vars_.ctypes.data_as(C.POINTER(C.c_double)), params.ctypes.data_as(C.POINTER(C.c_double)),
        out.ctypes.data_as(C.POINTER(C.c_double)), reps.ctypes.data_as(C.POINTER(FkReport)), reps.shape[1], C.byref(got), 1))


def device_split(fn):
    import torch
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.init()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    kernels, spans = {}, []
    for e in prof.events():
        if e.device_type.name != "CUDA" or "Memcpy" in e.name or "Memset" in e.name:
            continue
        k = kernels.setdefault(e.name, [0, 0.0])
        k[0] += 1
        k[1] += e.device_time / 1e3  # us -> ms
        spans.append((e.time_range.start, e.time_range.end))
    prep = sum(v[1] for k, v in kernels.items() if "fk_system_batch_prepare_kernel" in k)
    gs = sum(v[1] for k, v in kernels.items() if "fk_system_sp_gather_scatter_kernel" in k)
    solve = sum(v[1] for k, v in kernels.items() if "fk_system_batch_prepare_kernel" not in k and "fk_system_sp_gather_scatter_kernel" not in k)
    spans.sort()
    gaps = sum(max(0.0, b[0] - a[1]) for a, b in zip(spans, spans[1:])) / 1e3
    wall = (spans[-1][1] - spans[0][0]) / 1e3 if spans else 0.0
    total = prep + gs + solve
    return {"prepare_ms": prep, "gather_scatter_ms": gs, "solve_ms": solve, "device_ms": total, "kernel_span_ms": wall,
            "gaps_between_kernels_ms": gaps, "launches": sum(v[0] for v in kernels.values()),
            "kernels": {k: {"launches": v[0], "ms": v[1]} for k, v in sorted(kernels.items(), key=lambda kv: -kv[1][1])}}


def loop_rate(s, vars_, params):
    """variants/s of the per-variant System.solve_single_pass loop"""
    s.solve_single_pass()  # warm-up: topologies, device tables
    t0 = time.perf_counter()
    for k in range(len(vars_)):
        for i, x in enumerate(vars_[k]):
            s.set_variable(i, float(x))
        for c, x in enumerate(params[k]):
            s.set_parameter(c, float(x))
        s.solve_single_pass()
        s.variables
    return len(vars_) / (time.perf_counter() - t0)


def oracle_rate(builder, vars_, params):
    import oracle
    oracle.build()
    cores = os.sched_getaffinity(0)
    os.sched_setaffinity(0, {min(cores)})
    t = 0.0
    for k in range(len(vars_)):
        so = builder(oracle.System)
        for i, x in enumerate(vars_[k]):
            so.set_variable(i, float(x))
        for c, x in enumerate(params[k]):
            so.set_parameter(c, float(x))
        t0 = time.perf_counter()
        so.solve_single_pass()
        t += time.perf_counter() - t0
    os.sched_setaffinity(0, cores)
    return len(vars_) / t


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(REPO, "profiles", "r07_system_batch_single_pass_1gpu.json"))
    ap.add_argument("--passes", type=int, default=5)
    ap.add_argument("--quick", action="store_true", help="small n, for a rehearsal of the script")
    a = ap.parse_args()
    if fk.device_count() < 1:
        raise SystemExit("no CUDA device: nothing to measure")
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()
    res = {"card": smi[0] if smi else "not measured", "passes": a.passes, "drawings": {}}
    # name: (builder, variants, loop sample, oracle sample, None batch for context)
    drawings = {"a_chains_ctl_truss": (drawing_a, 65536, 64, 8, True), "b_lattice30x20_triangles": (drawing_b, 1024, 16, 2, True),
                "c_lattice80x60": (drawing_c, 256, 3, 1, False)}
    for name, (builder, n, n_loop, n_oracle, with_none) in drawings.items():
        if a.quick:
            n = min(n, 64)
        s = builder(fk.System)
        n_sets, n_waves, n_struct, wave, struct = s.single_pass_batch_layout()
        groups = len(set(zip(wave, struct)))
        vars_, params = variants(s, n, seed=0xF1C5)
        d = {"variants": n, "variables": int(len(s.variables)), "constraints": s.num_constraints(), "sets": n_sets,
             "waves": n_waves, "structures": n_struct, "sets_per_structure": np.bincount(struct).tolist() if struct else [],
             "launches_per_chunk": {"prepare": 1, "gather_scatter": n_waves + 1, "solve": groups, "total": 2 + n_waves + groups}}
        out = np.zeros((n, len(s.variables)))
        reps = np.zeros((n, n_sets), dtype=fk.REPORT_DTYPE)
        med, ts = timed(lambda: call_sp(s, vars_, params, out, reps), a.passes)
        d["pageable"] = {"s_per_call": med, "variants_per_s": n / med, "passes_s": ts}
        pv, bv = pinned(vars_)
        pp, bp = pinned(params)
        po, bo = pinned(out)
        pr, br = pinned(reps)
        med, ts = timed(lambda: call_sp(s, pv, pp, po, pr), a.passes)
        d["pinned"] = {"s_per_call": med, "variants_per_s": n / med, "passes_s": ts}
        assert np.array_equal(po, out, equal_nan=True), "pinned and pageable calls differ"
        d["device"] = device_split(lambda: call_sp(s, pv, pp, po, pr))
        for b in (bv, bp, bo, br):
            lib().fk_host_free(C.c_void_p(b))
        m = min(n_loop, n)
        ref = builder(fk.System)
        loop = loop_rate(ref, vars_[:m], params[:m])
        d["per_variant_loop"] = {"variants": m, "variants_per_s": loop}
        d["speedup_vs_loop_pinned"] = d["pinned"]["variants_per_s"] / loop
        if n_oracle:
            try:
                k = min(n_oracle, n)
                d["oracle_one_core"] = {"variants": k, "variants_per_s": oracle_rate(builder, vars_[:k], params[:k])}
            except Exception as e:  # noqa: BLE001
                d["oracle_one_core"] = f"not measured ({type(e).__name__}: {e})"
        else:
            d["oracle_one_core"] = "not measured"
        if with_none:
            nc = s.batch_layout()[0]
            o2 = np.zeros((n, len(s.variables)))
            r2 = np.zeros((n, nc), dtype=fk.REPORT_DTYPE)
            pv, bv = pinned(vars_)
            pp, bp = pinned(params)
            med, _ = timed(lambda: call(s, "lm", pv, pp, o2, r2), a.passes)
            d["decomposer_none_batch_lm"] = {"s_per_call": med, "variants_per_s": n / med, "buffers": "pinned inputs, pageable outputs"}
            for b in (bv, bp):
                lib().fk_host_free(C.c_void_p(b))
        else:
            d["decomposer_none_batch_lm"] = "not measured (refused: FK_ERR_TOO_LARGE)"
        res["drawings"][name] = d
        print(name, json.dumps({k: v for k, v in d.items() if k != "device"}, default=str)[:900], flush=True)
        print("   device split", {k: v for k, v in d["device"].items() if k != "kernels"}, flush=True)
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(res, f, indent=1)
    print("wrote", a.out)


if __name__ == "__main__":
    main()
