"""fk_system_batch_solve (System.batch_solve) on one B200: n variants of a drawing with several components in one call,
against the per-variant System.solve loop a design-table sweep runs without it, and the oracle on one core.

    python tools/bench_system_batch.py [--out FILE] [--passes K] [--quick]

Drawings: (a) 16 hinged chains of 4 triangles + 4 circle_triangle_line + one 20-point truss (21 components, 3 structures),
65,536 variants; (b) a 30x20 lattice + 8 triangles (the lattice on the global sparse path), 1,024 variants.  Variants carry
seeded relative noise of 1e-3 on the variables and on the distance / angle parameters.  For LM and L-BFGS:
- end to end: the host clock around the call (which returns with the results in host memory), from pageable numpy arrays
  and from pinned buffers (fk_host_alloc), one warm-up call first, medians of --passes passes;
- device time split: one extra call under torch.profiler (CUDA activity), kernel times summed by kernel: the prepare /
  gather kernel, the solve launches (one per structure and chunk) and the scatter kernel;
- the per-variant loop: set the variant's variables and parameters, System.solve, read the variables, over 256 variants;
- the oracle (CPU restatement) on one core: System.solve per variant on a sample (LM; L-BFGS through the composition of
  tests/oracle_system.py).
The card's name and power limit are read in the same call.  Anything not run is written as "not measured".
"""
import argparse
import ctypes as C
import json
import os
import statistics
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import fiksi_b200 as fk  # noqa: E402
from fiksi_b200 import workloads as wl  # noqa: E402
from fiksi_b200._lib import FkReport, FkSolvingOptions, lib  # noqa: E402
import scenarios as sc  # noqa: E402

_PARAM_TAGS = (1, 2, 4, 7)


def _recording(S):
    """S whose constraint calls are recorded (tag, parameter) in construction order; works for fk.System and oracle.System
    alike by wrapping the constraint methods."""
    methods = {"point_point_distance": 1, "point_point_point_angle": 2, "point_line_distance": 4, "line_line_angle": 7,
               "point_point_coincidence": 0, "point_line_incidence": 3, "point_circle_incidence": 5,
               "segment_segment_length_equality": 6, "line_line_parallelism": 8, "line_line_perpendicularity": 9,
               "line_circle_tangency": 10}

    class R(S):
        def __init__(self):
            super().__init__()
            self.tags, self.params = [], []

    def wrap(name, tag):
        base = getattr(S, name)

        def f(self, *args):
            self.tags.append(tag)
            self.params.append(float(args[-1]) if tag in _PARAM_TAGS else 0.0)
            return base(self, *args)
        return f
    for name, tag in methods.items():
        setattr(R, name, wrap(name, tag))
    return R


def _add_ppd(s, w):
    raw = w.raw_vars[0]
    pts = [s.add_point(float(raw[2 * i]), float(raw[2 * i + 1])) for i in range(len(raw) // 2)]
    for e in range(len(w.kind)):
        s.point_point_distance(pts[int(w.idx[e][0]) // 2], pts[int(w.idx[e][1]) // 2], float(w.raw_param[0][e]))


def drawing_a(S):
    s = _recording(S)()
    for _ in range(16):
        sc.hinged_triangles_bench(lambda: s, 4)
    for _ in range(4):
        sc.circle_triangle_line(lambda: s)
    _add_ppd(s, wl.truss(1, 20))
    return s


def drawing_b(S):
    s = _recording(S)()
    _add_ppd(s, wl.lattice(30, 20))
    for _ in range(8):
        sc.single_triangle(lambda: s)
    return s


def variants(s, n, seed):
    rng = np.random.default_rng(seed)
    v0 = s.variables.copy()
    p0 = np.array(s.params)
    vars_ = v0[None, :] * (1.0 + 1e-3 * rng.standard_normal((n, len(v0))))
    params = np.tile(p0, (n, 1))
    noisy = np.array([t in _PARAM_TAGS for t in s.tags])
    params[:, noisy] *= 1.0 + 1e-3 * rng.standard_normal((n, int(noisy.sum())))
    return vars_, params


def pinned(a):
    a = np.ascontiguousarray(a)
    buf = lib().fk_host_alloc(C.c_size_t(max(a.nbytes, 1)))
    h = np.ctypeslib.as_array((C.c_uint8 * max(a.nbytes, 1)).from_address(buf))[:a.nbytes].view(a.dtype).reshape(a.shape)
    h[...] = a
    return h, buf


def call(s, optimizer, vars_, params, out, reps):
    opts = FkSolvingOptions({"lm": 0, "lbfgs": 1}[optimizer], 0, 1, 0)
    got = C.c_uint32(0)
    fk._lib.check(lib().fk_system_batch_solve(s._h, C.byref(opts), len(vars_), vars_.ctypes.data_as(C.POINTER(C.c_double)),
                                              params.ctypes.data_as(C.POINTER(C.c_double)), out.ctypes.data_as(C.POINTER(C.c_double)),
                                              reps.ctypes.data_as(C.POINTER(FkReport)), reps.shape[1], C.byref(got), 1))


def timed(fn, passes):
    fn()  # warm-up: plan, topologies, device tables, buffers
    ts = []
    for _ in range(passes):
        t0 = time.perf_counter()
        fn()
        ts.append(time.perf_counter() - t0)
    return statistics.median(ts), ts


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
    prep = sum(v[1] for k, v in kernels.items() if "fk_system_batch_prepare_kernel" in k)
    scat = sum(v[1] for k, v in kernels.items() if "fk_system_batch_scatter_kernel" in k)
    solve = sum(v[1] for k, v in kernels.items() if "fk_system_batch" not in k)
    total = prep + scat + solve
    return {"prepare_ms": prep, "solve_ms": solve, "scatter_ms": scat, "device_ms": total,
            "outside_solve_share": (prep + scat) / total if total else None,
            "kernels": {k: {"launches": v[0], "ms": v[1]} for k, v in sorted(kernels.items(), key=lambda kv: -kv[1][1])}}


def loop_rate(s, vars_, params, optimizer):
    """(variants/s of the whole loop, variants/s counting the System.solve calls alone)"""
    s.solve(optimizer=optimizer)  # warm-up: topologies, device tables
    t_solve = 0.0
    t0 = time.perf_counter()
    for k in range(len(vars_)):
        for i, x in enumerate(vars_[k]):
            s.set_variable(i, float(x))
        for c, x in enumerate(params[k]):
            s.set_parameter(c, float(x))
        t1 = time.perf_counter()
        s.solve(optimizer=optimizer)
        t_solve += time.perf_counter() - t1
        s.variables
    return len(vars_) / (time.perf_counter() - t0), len(vars_) / t_solve


def oracle_rate(builder, vars_, params, optimizer):
    import oracle
    import oracle_system
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
        if optimizer == "lm":
            so.solve()
        else:
            oracle_system.solve(oracle, so, optimizer="lbfgs")
        t += time.perf_counter() - t0
    os.sched_setaffinity(0, cores)
    return len(vars_) / t


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r06_system_batch_1gpu.json"))
    ap.add_argument("--passes", type=int, default=5)
    ap.add_argument("--quick", action="store_true", help="small n, for a rehearsal of the script")
    a = ap.parse_args()
    if fk.device_count() < 1:
        raise SystemExit("no CUDA device: nothing to measure")
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()
    res = {"card": smi[0] if smi else "not measured", "passes": a.passes, "drawings": {}}
    drawings = {"a_chains_ctl_truss": (drawing_a, 65536, 8), "b_lattice30x20_triangles": (drawing_b, 1024, 2)}
    for name, (builder, n, n_oracle) in drawings.items():
        if a.quick:
            n = min(n, 256)
        s = builder(fk.System)
        nc, ns, mult = s.batch_layout()
        vars_, params = variants(s, n, seed=0xF1C5)
        d = {"variants": n, "variables": int(len(s.variables)), "constraints": s.num_constraints(), "components": nc,
             "structures": ns, "multiplicity": mult, "optimizers": {}}
        for opt in ("lm", "lbfgs"):
            r = {}
            out = np.zeros((n, len(s.variables)))
            reps = np.zeros((n, nc), dtype=fk.REPORT_DTYPE)
            med, ts = timed(lambda: call(s, opt, vars_, params, out, reps), a.passes)
            r["pageable"] = {"s_per_call": med, "variants_per_s": n / med, "passes_s": ts}
            pv, bv = pinned(vars_)
            pp, bp = pinned(params)
            po, bo = pinned(out)
            pr, br = pinned(reps)
            med, ts = timed(lambda: call(s, opt, pv, pp, po, pr), a.passes)
            r["pinned"] = {"s_per_call": med, "variants_per_s": n / med, "passes_s": ts}
            assert np.array_equal(po, out, equal_nan=True), "pinned and pageable calls differ"
            r["device"] = device_split(lambda: call(s, opt, pv, pp, po, pr))
            for b in (bv, bp, bo, br):
                lib().fk_host_free(C.c_void_p(b))
            m = min(256, n)
            loop, loop_solve = loop_rate(builder(fk.System), vars_[:m], params[:m], opt)
            r["per_variant_loop"] = {"variants": m, "variants_per_s": loop, "variants_per_s_solve_calls_only": loop_solve}
            r["speedup_vs_loop_pinned"] = r["pinned"]["variants_per_s"] / loop
            try:
                k = min(n_oracle, n)
                r["oracle_one_core"] = {"variants": k, "variants_per_s": oracle_rate(builder, vars_[:k], params[:k], opt)}
            except Exception as e:  # noqa: BLE001
                r["oracle_one_core"] = f"not measured ({type(e).__name__}: {e})"
            d["optimizers"][opt] = r
            print(name, opt, json.dumps({k: v for k, v in r.items() if k != "device"}, default=str)[:600], flush=True)
            print("   device split", {k: v for k, v in r["device"].items() if k != "kernels"}, flush=True)
        res["drawings"][name] = d
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(res, f, indent=1)
    print("wrote", a.out)


if __name__ == "__main__":
    main()
