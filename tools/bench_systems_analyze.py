"""fk_systems_analyze / fk_systems_residuals (fiksi_b200.analyze_systems / systems_residuals) on one B200: System::analyze and
calculate_residual over many different drawings in one call, against the per-drawing loop.

    python tools/bench_systems_analyze.py [--out FILE] [--passes K] [--quick]

Workloads: (a), (b), (c) are tools/bench_systems_solve.py's (65,536 small mixed drawings, 8,192 Henneberg drawings of nearly
all distinct structures, 1,024 mid-size drawings: 30x20 lattices, 8x7 cad_grids, 200-point trusses), unsolved; and
(u) 65,536 copies of one drawing of 4 hinged 4-triangle chains: one structure, so fk_systems_analyze's heterogeneous warp
    launch runs next to fk_system_batch_analyze's uniform warp kernel (System.batch_analyze on the same drawing, n = 65,536) in
    the same run, alternating.
For analyze and for residuals:
- first call: systems freshly built, so the call builds every drawing's plan; steady call: the plans built beforehand.  Host
  clock around the call, which returns with the outputs on the host; medians of --passes passes after one warm-up call;
- the per-drawing loop (System.analyze() / System.residuals()) on a sample, and the steady call's ratio to it;
- device split: one call under torch.profiler in a process of its own (after a warm-up call there), kernel and copy times summed.
The card's name and power limit are read in the same run.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
sys.path.insert(0, os.path.join(ROOT, "tools"))

import numpy as np  # noqa: E402

import fiksi_b200 as fk  # noqa: E402
from bench_systems_solve import workload_a, workload_b, workload_c  # noqa: E402

CALLS = {"analyze": fk.analyze_systems, "residuals": fk.systems_residuals}


def four_chains(S):
    """4 hinged chains of 4 triangles each (hinged_triangles_bench's shape), fixed offsets."""
    s = S()
    for c in range(4):
        hinge = s.add_point(10.0 * c, 0.0)
        for k in range(4):
            p1, p2 = s.add_point(10.0 * c - 1.0 + 0.01 * k, k + 0.1), s.add_point(10.0 * c + 1.0, k - 0.1)
            s.point_point_distance(hinge, p1, 2.0)
            s.point_point_distance(hinge, p2, 2.0)
            s.point_point_distance(p1, p2, 3.0)
    return s


def workload_u(n):
    return [four_chains] * n


def build(builders):
    return [b(fk.System) for b in builders]


def timed(fn, passes, fresh):
    ts = []
    for _ in range(passes):
        args = fresh()
        t0 = time.perf_counter()
        fn(*args)
        ts.append(time.perf_counter() - t0)
    return statistics.median(ts), ts


def device_split(fns):
    import torch
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.init()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for f in fns:
            f()
        torch.cuda.synchronize()
    split = {"hetero_ms": 0.0, "uniform_ms": 0.0, "reduce_ms": 0.0, "residual_ms": 0.0, "copy_ms": 0.0}
    kernels = {}
    for e in prof.events():
        if e.device_type.name != "CUDA":
            continue
        ms = e.device_time / 1e3
        k = kernels.setdefault(e.name, [0, 0.0])
        k[0] += 1
        k[1] += ms
        key = ("copy_ms" if "Memcpy" in e.name or "Memset" in e.name else "hetero_ms" if "fk_systems_analyze" in e.name
               else "reduce_ms" if "an_reduce" in e.name else "residual_ms" if "residuals" in e.name else "uniform_ms")
        split[key] += ms
    split["device_ms"] = sum(split.values())
    split["kernels"] = {k: {"launches": v[0], "ms": v[1]} for k, v in sorted(kernels.items(), key=lambda kv: -kv[1][1])[:12]}
    return split


def loop_rate(systems, op):
    f = (lambda s: s.analyze()) if op == "analyze" else (lambda s: s.residuals())
    f(systems[0])  # warm-up
    t0 = time.perf_counter()
    for s in systems[1:]:
        f(s)
    return (len(systems) - 1) / (time.perf_counter() - t0)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r14_systems_analyze_1gpu.json"))
    ap.add_argument("--passes", type=int, default=5)
    ap.add_argument("--quick", action="store_true", help="small workloads, for a rehearsal of the script")
    ap.add_argument("--split", nargs=2, metavar=("WORKLOAD", "OP"), help="print the device split of one call (internal)")
    a = ap.parse_args()
    if fk.device_count() < 1:
        raise SystemExit("no CUDA device: nothing to measure")
    sizes = {"a_small_mixed": (workload_a, 65536, 256), "b_distinct": (workload_b, 8192, 256), "c_mid_size": (workload_c, 1024, 32),
             "u_one_structure": (workload_u, 65536, 256)}
    if a.split:
        make, n, _ = sizes[a.split[0]]
        systems = build(make(min(n, 512) if a.quick else n))
        CALLS[a.split[1]](systems)  # warm-up, plans built
        fns = [lambda: CALLS[a.split[1]](systems)]
        if a.split[0] == "u_one_structure" and a.split[1] == "analyze":
            tmpl = systems[0]
            tmpl.batch_analyze(n=len(systems))
            fns.append(lambda: tmpl.batch_analyze(n=len(systems)))
        print(json.dumps(device_split(fns)))
        return
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()
    res = {"card": smi[0] if smi else "not measured", "passes": a.passes, "workloads": {}}
    for name, (make, n, n_loop) in sizes.items():
        if a.quick:
            n, n_loop = min(n, 512), min(n_loop, 16)
        builders = make(n)
        t0 = time.perf_counter()
        probe = build(builders)
        ns, inst, kind = fk.systems_analyze_layout(probe)
        d = {"drawings": n, "build_s": time.perf_counter() - t0, "constraints": int(sum(s.num_constraints() for s in probe)),
             "structures": ns, "launch_kinds": {str(k): kind.count(k) for k in (0, 1)}, "ops": {}}
        for op, fn in CALLS.items():
            fn(build(builders))  # warm-up: modules, buffers
            r = {}
            med, ts = timed(fn, a.passes, lambda: (build(builders),))
            r["first_call"] = {"s_per_call": med, "drawings_per_s": n / med, "passes_s": ts}
            med, ts = timed(fn, a.passes, lambda: (probe,))
            r["steady_call"] = {"s_per_call": med, "drawings_per_s": n / med, "passes_s": ts}
            if name == "u_one_structure" and op == "analyze":  # the uniform warp kernel on the same drawing, alternating
                tmpl = probe[0]
                tmpl.batch_analyze(n=n)
                same = np.array_equal(np.stack(fn(probe)), tmpl.batch_analyze(n=n))
                hs, us = [], []
                for _ in range(a.passes):
                    hs.append(timed(fn, 1, lambda: (probe,))[0])
                    us.append(timed(lambda: tmpl.batch_analyze(n=n), 1, lambda: ())[0])
                r["vs_fk_system_batch_analyze"] = {"systems_analyze_s": statistics.median(hs), "systems_analyze_passes_s": hs,
                                                   "batch_analyze_s": statistics.median(us), "batch_analyze_passes_s": us,
                                                   "identical_counts": bool(same)}
            cmd = [sys.executable, os.path.abspath(__file__), "--split", name, op] + (["--quick"] if a.quick else [])
            r["device"] = json.loads(subprocess.run(cmd, capture_output=True, text=True, check=True).stdout.strip().splitlines()[-1])
            sample = build(builders[:: max(1, n // n_loop)][:n_loop])
            r["per_drawing_loop"] = {"drawings": len(sample) - 1, "drawings_per_s": loop_rate(sample, op)}
            r["speedup_steady_vs_loop"] = r["steady_call"]["drawings_per_s"] / r["per_drawing_loop"]["drawings_per_s"]
            d["ops"][op] = r
            print(name, op, json.dumps({k: v for k, v in r.items() if k != "device"}, default=str)[:900], flush=True)
            print("   device split", {k: v for k, v in r["device"].items() if k != "kernels"}, flush=True)
        res["workloads"][name] = d
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(res, f, indent=1)
    print("wrote", a.out)


if __name__ == "__main__":
    main()
