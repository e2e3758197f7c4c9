"""fk_system_batch_solve_recursive_assembly (System.batch_solve_recursive_assembly) on one B200: System::solve with
Decomposer::RecursiveAssembly over n variants of one drawing in one call, against the per-variant
System.solve_recursive_assembly loop a design-table sweep runs without it, and the oracle's RecursiveAssembly on one core.

    python tools/bench_system_batch_recursive_assembly.py [--out FILE] [--passes K] [--quick]

Drawings: (a) 16 hinged chains of 4 triangles + 8 single triangles + 4 triangle_inscribed_circle (28 components, 240 steps),
65,536 variants; (b) one hinged chain of 8 triangles (24 steps; its plan is the planner's exhaustive search at its costliest
here), 4,096 variants.  Variants as in tools/bench_system_batch.py.  Per drawing:
- the plan: steps, waves, structures, the host time of building it once, and launches per chunk (one prepare, one gather /
  scatter per wave and one more, one LM launch per structure present in a wave);
- end to end: the host clock around the call, from pageable numpy arrays and from pinned buffers (fk_host_alloc), one
  warm-up call first, medians of --passes passes;
- device time split: one extra call under torch.profiler (CUDA activity): prepare kernel, gather / scatter kernel (with the
  owned-point moves), solve launches, and the gaps between kernels on the stream;
- the per-variant loop (set the variant's numbers, System.solve_recursive_assembly, read the variables) over a sample, and
  the fraction of that sample whose batch result is bit-identical to the loop's (moves use CUDA's sincos in the batch and
  glibc's sin / cos in the loop);
- the oracle's System.solve_recursive_assembly on one core over a sample.
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
from bench_system_batch import _recording, pinned, timed, variants  # noqa: E402
from bench_system_batch_single_pass import device_split  # noqa: E402

import fiksi_b200 as fk  # noqa: E402
from fiksi_b200._lib import FkReport, lib  # noqa: E402
import scenarios as sc  # noqa: E402

REPO = os.path.dirname(ROOT)


def drawing_a(S):
    s = _recording(S)()
    for _ in range(16):
        sc.hinged_triangles_bench(lambda: s, 4)
    for _ in range(8):
        sc.single_triangle(lambda: s)
    for _ in range(4):
        sc.triangle_inscribed_circle(lambda: s)
    return s


def drawing_b(S):
    s = _recording(S)()
    sc.hinged_triangles_bench(lambda: s, 8)
    return s


def call_ra(s, vars_, params, out, reps):
    got = C.c_uint32(0)
    fk._lib.check(lib().fk_system_batch_solve_recursive_assembly(
        s._h, 1, len(vars_), vars_.ctypes.data_as(C.POINTER(C.c_double)), params.ctypes.data_as(C.POINTER(C.c_double)),
        out.ctypes.data_as(C.POINTER(C.c_double)), reps.ctypes.data_as(C.POINTER(FkReport)), reps.shape[1], C.byref(got), 1))


def loop(s, vars_, params):
    """(variants/s, outputs, reports) of the per-variant System.solve_recursive_assembly loop"""
    s.solve_recursive_assembly()  # warm-up: topologies, device tables
    outs, reps = [], []
    t0 = time.perf_counter()
    for k in range(len(vars_)):
        for i, x in enumerate(vars_[k]):
            s.set_variable(i, float(x))
        for c, x in enumerate(params[k]):
            s.set_parameter(c, float(x))
        s.solve_recursive_assembly()
        outs.append(s.variables)
        reps.append(s._reports.copy())
    return len(vars_) / (time.perf_counter() - t0), np.array(outs), np.array(reps)


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
        so.solve_recursive_assembly()
        t += time.perf_counter() - t0
    os.sched_setaffinity(0, cores)
    return len(vars_) / t


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(REPO, "profiles", "r08_system_batch_recursive_assembly_1gpu.json"))
    ap.add_argument("--passes", type=int, default=5)
    ap.add_argument("--quick", action="store_true", help="small n, for a rehearsal of the script")
    a = ap.parse_args()
    if fk.device_count() < 1:
        raise SystemExit("no CUDA device: nothing to measure")
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()
    res = {"card": smi[0] if smi else "not measured", "passes": a.passes, "drawings": {}}
    # name: (builder, variants, loop sample, oracle sample)
    drawings = {"a_chains_triangles_circles": (drawing_a, 65536, 16, 4), "b_chain8": (drawing_b, 4096, 16, 4)}
    for name, (builder, n, n_loop, n_oracle) in drawings.items():
        if a.quick:
            n = min(n, 64)
        s = builder(fk.System)
        t0 = time.perf_counter()
        n_steps, n_waves, n_struct, wave, struct = s.recursive_assembly_batch_layout()
        plan_s = time.perf_counter() - t0
        groups = len(set(zip(wave, struct)))
        vars_, params = variants(s, n, seed=0xF1C5)
        d = {"variants": n, "variables": int(len(s.variables)), "constraints": s.num_constraints(), "steps": n_steps,
             "waves": n_waves, "structures": n_struct, "steps_per_structure": np.bincount(struct).tolist() if struct else [],
             "plan_host_s": plan_s,
             "launches_per_chunk": {"prepare": 1, "gather_scatter": n_waves + 1, "solve": groups, "total": 2 + n_waves + groups}}
        out = np.zeros((n, len(s.variables)))
        reps = np.zeros((n, n_steps), dtype=fk.REPORT_DTYPE)
        med, ts = timed(lambda: call_ra(s, vars_, params, out, reps), a.passes)
        d["pageable"] = {"s_per_call": med, "variants_per_s": n / med, "passes_s": ts}
        pv, bv = pinned(vars_)
        pp, bp = pinned(params)
        po, bo = pinned(out)
        pr, br = pinned(reps)
        med, ts = timed(lambda: call_ra(s, pv, pp, po, pr), a.passes)
        d["pinned"] = {"s_per_call": med, "variants_per_s": n / med, "passes_s": ts}
        assert np.array_equal(po, out, equal_nan=True), "pinned and pageable calls differ"
        d["device"] = device_split(lambda: call_ra(s, pv, pp, po, pr))
        for b in (bv, bp, bo, br):
            lib().fk_host_free(C.c_void_p(b))
        m = min(n_loop, n)
        rate, ref_out, ref_reps = loop(builder(fk.System), vars_[:m], params[:m])
        d["per_variant_loop"] = {"variants": m, "variants_per_s": rate}
        d["speedup_vs_loop_pinned"] = d["pinned"]["variants_per_s"] / rate
        decisions = all(np.array_equal(reps[f][:m], ref_reps[f]) for f in ("exit_reason", "outer_iters", "factorizations", "trace_hash"))
        scale = np.max(np.abs(ref_out), axis=1, keepdims=True)
        d["vs_loop_sample"] = {"variants": m, "bit_identical_fraction": float(np.mean(np.all(out[:m] == ref_out, axis=1))),
                               "decisions_equal": bool(decisions),
                               "max_rel_diff": float(np.max(np.abs(out[:m] - ref_out) / scale))}
        try:
            k = min(n_oracle, n)
            d["oracle_one_core"] = {"variants": k, "variants_per_s": oracle_rate(builder, vars_[:k], params[:k])}
        except Exception as e:  # noqa: BLE001
            d["oracle_one_core"] = f"not measured ({type(e).__name__}: {e})"
        res["drawings"][name] = d
        print(name, json.dumps({k: v for k, v in d.items() if k != "device"}, default=str)[:1200], flush=True)
        print("   device split", {k: v for k, v in d["device"].items() if k != "kernels"}, flush=True)
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(res, f, indent=1)
    print("wrote", a.out)


if __name__ == "__main__":
    main()
