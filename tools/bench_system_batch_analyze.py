"""fk_system_batch_analyze / fk_system_batch_residuals (System.batch_analyze / batch_residuals) on one B200: n variants of a
drawing in one call, against the per-variant loop a design-table sweep runs without them, and the oracle on one core.

    python tools/bench_system_batch_analyze.py [--out FILE] [--passes K] [--quick]

Drawings (those of tools/bench_system_batch.py plus one on the warp kernel):
- (a) 16 hinged chains of 4 triangles + 4 circle_triangle_line + a 20-point truss (372 variables: the analyze matrix leaves
  shared memory), 8,192 variants for analyze, 65,536 for residuals;
- (b) a 30x20 lattice + 8 triangles (1,248 variables; System.residuals() runs fk_topology_eval there), 256 variants for
  analyze, 4,096 for residuals;
- (c) 4 hinged chains of 4 triangles (72 variables, 48 distances), whose matrix fits the warp kernel, 65,536 variants for
  both;
- (d) 16 such chains (288 variables, 192 distances): 442 KB of matrix, one CTA per sketch, 65,536 variants for both.
Variants carry seeded relative noise of 1e-3 on the variables and on the distance / angle parameters.  Per call:
- end to end: the host clock around the call (it returns with the results in host memory), from pageable numpy arrays and
  from pinned buffers (fk_host_alloc), one warm-up call first, medians of --passes passes;
- device time split: one extra call under torch.profiler (CUDA activity): the expand kernel, the analyze kernel, the reduce
  kernel, the residual kernel;
- the per-variant loop: set the variant's variables and parameters, System.analyze() / System.residuals(), on a sample;
- the oracle (CPU restatement) on one core: System.analyze() / calculate_residual of every constraint, on a sample.
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

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
sys.path.insert(0, os.path.join(ROOT, "tools"))

import fiksi_b200 as fk  # noqa: E402
from fiksi_b200._lib import check, lib  # noqa: E402
import scenarios as sc  # noqa: E402
from bench_system_batch import _recording, drawing_a, drawing_b, pinned, timed, variants  # noqa: E402


def chains(k):
    def build(S):
        s = _recording(S)()
        for _ in range(k):
            sc.hinged_triangles_bench(lambda: s, 4)
        return s
    return build


def call(s, op, vars_, params, out):
    f64 = C.POINTER(C.c_double)
    if op == "analyze":
        check(lib().fk_system_batch_analyze(s._h, len(vars_), vars_.ctypes.data_as(f64), params.ctypes.data_as(f64),
                                            out.ctypes.data_as(C.POINTER(C.c_uint8)), 1))
    else:
        check(lib().fk_system_batch_residuals(s._h, len(vars_), vars_.ctypes.data_as(f64), params.ctypes.data_as(f64),
                                              out.ctypes.data_as(f64), 1))


def device_split(fn):
    import torch
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.init()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    kernels = {}
    for e in prof.events():
        if e.device_type.name != "CUDA" or "Memcpy" in e.name or "Memset" in e.name:
            continue
        k = kernels.setdefault(e.name, [0, 0.0])
        k[0] += 1
        k[1] += e.device_time / 1e3  # us -> ms

    def ms(tag):
        return sum(v[1] for k, v in kernels.items() if tag in k)
    # "analyze": fk_batch_analyze_kernel (warp) or fk_analyze_cta_kernel (cta / group)
    r = {"expand_ms": ms("fk_system_an_expand_kernel"), "analyze_ms": ms("analyze"), "reduce_ms": ms("fk_system_an_reduce_kernel"),
         "residual_ms": ms("fk_system_residuals_kernel")}
    r["device_ms"] = sum(v[1] for v in kernels.values())
    r["kernels"] = {k: {"launches": v[0], "ms": v[1]} for k, v in sorted(kernels.items(), key=lambda kv: -kv[1][1])}
    return r


def loop_rate(s, op, vars_, params):
    """(variants/s of the whole loop, variants/s counting the analyze / residuals calls alone)"""
    getattr(s, op)()  # warm-up
    t_call = 0.0
    t0 = time.perf_counter()
    for k in range(len(vars_)):
        for i, x in enumerate(vars_[k]):
            s.set_variable(i, float(x))
        for c, x in enumerate(params[k]):
            s.set_parameter(c, float(x))
        t1 = time.perf_counter()
        getattr(s, op)()
        t_call += time.perf_counter() - t1
    return len(vars_) / (time.perf_counter() - t0), len(vars_) / t_call


def oracle_rate(builder, op, vars_, params):
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
        if op == "analyze":
            so.analyze()
        else:
            [so.calculate_residual(c) for c in range(len(so.params))]
        t += time.perf_counter() - t0
    os.sched_setaffinity(0, cores)
    return len(vars_) / t


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r09_system_batch_analyze_1gpu.json"))
    ap.add_argument("--passes", type=int, default=5)
    ap.add_argument("--quick", action="store_true", help="small n, for a rehearsal of the script")
    a = ap.parse_args()
    if fk.device_count() < 1:
        raise SystemExit("no CUDA device: nothing to measure")
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()
    res = {"card": smi[0] if smi else "not measured", "passes": a.passes, "workloads": {}}
    # drawing -> (builder, {op: (variants, loop sample, oracle sample)})
    drawings = {
        "a_chains_ctl_truss": (drawing_a, {"analyze": (8192, 32, 4), "residuals": (65536, 256, 64)}),
        "b_lattice30x20_triangles": (drawing_b, {"analyze": (256, 4, 1), "residuals": (4096, 64, 8)}),
        "c_chains4x4": (chains(4), {"analyze": (65536, 256, 64), "residuals": (65536, 256, 64)}),
        "d_chains16x4": (chains(16), {"analyze": (65536, 64, 8), "residuals": (65536, 256, 64)}),
    }
    for name, (builder, ops) in drawings.items():
        s = builder(fk.System)
        for op, (n, n_loop, n_oracle) in ops.items():
            if a.quick:
                n = min(n, 256)
            vars_, params = variants(s, n, seed=0xF1C5)
            r = {"variants": n, "variables": int(len(s.variables)), "constraints": s.num_constraints()}
            out = np.zeros((n, s.num_constraints()), np.uint8 if op == "analyze" else np.float64)
            med, ts = timed(lambda: call(s, op, vars_, params, out), a.passes)
            r["pageable"] = {"s_per_call": med, "variants_per_s": n / med, "passes_s": ts}
            pv, bv = pinned(vars_)
            pp, bp = pinned(params)
            po, bo = pinned(out)
            med, ts = timed(lambda: call(s, op, pv, pp, po), a.passes)
            r["pinned"] = {"s_per_call": med, "variants_per_s": n / med, "passes_s": ts}
            assert np.array_equal(po, out, equal_nan=True), "pinned and pageable calls differ"
            r["device"] = device_split(lambda: call(s, op, pv, pp, po))
            for b in (bv, bp, bo):
                lib().fk_host_free(C.c_void_p(b))
            m = min(n_loop, n)
            ref = builder(fk.System)
            loop, loop_call = loop_rate(ref, op, vars_[:m], params[:m])
            r["per_variant_loop"] = {"variants": m, "variants_per_s": loop, "variants_per_s_calls_only": loop_call}
            r["speedup_vs_loop_pinned"] = r["pinned"]["variants_per_s"] / loop
            # the sample agrees with the loop (analyze as lists, residuals bit for bit)
            got = []
            for k in range(m):
                for i, x in enumerate(vars_[k]):
                    ref.set_variable(i, float(x))
                for c, x in enumerate(params[k]):
                    ref.set_parameter(c, float(x))
                got.append(ref.analyze() == np.repeat(np.arange(out.shape[1]), out[k]).tolist() if op == "analyze"
                           else np.array_equal(ref.residuals(), out[k], equal_nan=True))
            r["loop_sample_identical"] = bool(all(got))
            try:
                k = min(n_oracle, n)
                r["oracle_one_core"] = {"variants": k, "variants_per_s": oracle_rate(builder, op, vars_[:k], params[:k])}
            except Exception as e:  # noqa: BLE001
                r["oracle_one_core"] = f"not measured ({type(e).__name__}: {e})"
            res["workloads"][f"{name}/{op}"] = r
            print(name, op, json.dumps({k: v for k, v in r.items() if k != "device"}, default=str)[:700], flush=True)
            print("   device split", {k: v for k, v in r["device"].items() if k != "kernels"}, flush=True)
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(res, f, indent=1)
    print("wrote", a.out)


if __name__ == "__main__":
    main()
