"""fk_systems_solve (fiksi_b200.solve_systems) on one B200: many different drawings in one call, against the per-drawing
System.solve loop.

    python tools/bench_systems_solve.py [--out FILE] [--passes K] [--quick]

Workloads (every drawing built from tests/scenarios.py / tests/cad_drawings.py shapes, seeded):
(a) 65,536 small drawings: hinged chains of 1-16 triangles, trusses of 4-40 points, circle_triangle_line at seeded scales
    with seeded noise, and 3x3 / 4x4 cad_grids with their own seeds -- few structures with many instances (uniform launches)
    next to rare ones (the heterogeneous launch);
(b) 8,192 drawings of 4-12 points built by seeded random Henneberg steps (every new point tied to two random earlier points):
    nearly every structure is distinct, so under LM nearly all go to the heterogeneous launch and under L-BFGS every
    structure is a launch of its own;
(c) 1,024 mid-size drawings: 30x20 lattices (global sparse path), 8x7 cad_grids (one CTA per sketch) and 200-point trusses.
For LM and L-BFGS:
- first call: systems freshly built, so the call builds every drawing's plan; steady call: the plans built beforehand
  (systems_layout, host only), values still unsolved.  Host clock around solve_systems, which returns with the systems
  written; medians of --passes passes, each on a fresh copy of the workload, after one warm-up call;
- the host time of the call's cross-drawing plan: systems_layout on drawings whose plans are cached;
- the per-drawing loop: System.solve on a fresh sample;
- device split: one call under torch.profiler in a process of its own (after a warm-up call there), kernel and copy times
  summed: prepare / heterogeneous launch / other solve launches / scatter / copies.
The card's name and power limit are read in the same run.
"""
import argparse
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
import systems_mix as mix  # noqa: E402


def truss_drawing(n_points, seed):
    w = wl.truss(1, n_points, seed=seed)
    return mix.ppd(w, 0)


def henneberg(n_points, seed):
    def build(S):
        rng = np.random.default_rng(seed)
        s = S()
        p = [s.add_point(*rng.uniform(-5, 5, 2)) for _ in range(n_points)]
        s.point_point_distance(p[0], p[1], float(rng.uniform(1, 3)))
        for i in range(2, n_points):
            a, b = rng.choice(i, 2, replace=False)
            s.point_point_distance(p[i], p[int(a)], float(rng.uniform(1, 3)))
            s.point_point_distance(p[i], p[int(b)], float(rng.uniform(1, 3)))
        return s
    return build


def workload_a(n):
    rng = np.random.default_rng(0xA)
    out = []
    for k in range(n):
        r = rng.integers(16)
        if r < 6:
            out.append(mix.hinged_chain(int(rng.integers(1, 17)), seed=k))
        elif r < 11:
            out.append(truss_drawing(int(rng.integers(4, 41)), seed=k))
        elif r < 15:
            out.append(mix.scaled_ctl(k))
        else:
            out.append(mix.cad(*((3, 3) if rng.integers(2) else (4, 4)), seed=k))
    return out


def workload_b(n):
    rng = np.random.default_rng(0xB)
    return [henneberg(int(rng.integers(4, 13)), seed=k) for k in range(n)]


def workload_c(n):
    rng = np.random.default_rng(0xC)
    out = []
    for k in range(n):
        r = rng.integers(3)
        out.append(mix.ppd(wl.lattice(30, 20, seed=k), 0) if r == 0 else mix.cad(8, 7, seed=k) if r == 1 else truss_drawing(200, seed=k))
    return out


def build(builders):
    return [b(fk.System) for b in builders]


def timed_calls(builders, opt, passes, cached):
    ts = []
    for _ in range(passes):
        systems = build(builders)
        if cached:
            fk.systems_layout(systems, opt)
        t0 = time.perf_counter()
        fk.solve_systems(systems, optimizer=opt)
        ts.append(time.perf_counter() - t0)
    return statistics.median(ts), ts


def device_split(systems, opt):
    import torch
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.init()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fk.solve_systems(systems, optimizer=opt)
        torch.cuda.synchronize()
    split = {"prepare_ms": 0.0, "hetero_ms": 0.0, "solve_ms": 0.0, "scatter_ms": 0.0, "copy_ms": 0.0}
    kernels = {}
    for e in prof.events():
        if e.device_type.name != "CUDA":
            continue
        ms = e.device_time / 1e3
        k = kernels.setdefault(e.name, [0, 0.0])
        k[0] += 1
        k[1] += ms
        key = ("copy_ms" if "Memcpy" in e.name or "Memset" in e.name else "prepare_ms" if "fk_systems_prepare" in e.name
               else "scatter_ms" if "fk_systems_scatter" in e.name else "hetero_ms" if "fk_hetero_lm" in e.name else "solve_ms")
        split[key] += ms
    split["device_ms"] = sum(split.values())
    split["solve_launches"] = sum(v[0] for k, v in kernels.items() if "fk_systems_" not in k and "Memcpy" not in k and "Memset" not in k)
    split["kernels"] = {k: {"launches": v[0], "ms": v[1]} for k, v in sorted(kernels.items(), key=lambda kv: -kv[1][1])[:12]}
    return split


def loop_rate(builders, opt):
    systems = build(builders)
    systems[0].solve(optimizer=opt)  # warm-up
    t = 0.0
    for s in systems[1:]:
        t0 = time.perf_counter()
        s.solve(optimizer=opt)
        t += time.perf_counter() - t0
    return (len(systems) - 1) / t


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r13_systems_solve_1gpu.json"))
    ap.add_argument("--passes", type=int, default=5)
    ap.add_argument("--quick", action="store_true", help="small workloads, for a rehearsal of the script")
    ap.add_argument("--split", nargs=2, metavar=("WORKLOAD", "OPTIMIZER"), help="print the device split of one call (internal)")
    a = ap.parse_args()
    if fk.device_count() < 1:
        raise SystemExit("no CUDA device: nothing to measure")
    sizes = {"a_small_mixed": (workload_a, 65536, 1024), "b_distinct": (workload_b, 8192, 1024), "c_mid_size": (workload_c, 1024, 48)}
    if a.split:
        make, n, _ = sizes[a.split[0]]
        builders = make(min(n, 512) if a.quick else n)
        fk.solve_systems(build(builders), optimizer=a.split[1])  # warm-up
        systems = build(builders)
        fk.systems_layout(systems, a.split[1])
        print(json.dumps(device_split(systems, a.split[1])))
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
        build_s = time.perf_counter() - t0
        d = {"drawings": n, "build_s": build_s, "optimizers": {}}
        for opt in ("lm", "lbfgs"):
            nc, ns, inst, kind = fk.systems_layout(probe, opt)
            r = {"components": nc, "structures": ns, "launch_kinds": {str(k): kind.count(k) for k in (0, 1, 2)},
                 "instances_by_kind": {str(k): int(sum(i for i, q in zip(inst, kind) if q == k)) for k in (0, 1, 2)}}
            fk.solve_systems(build(builders), optimizer=opt)  # warm-up: modules, topologies, device tables, buffers
            med, ts = timed_calls(builders, opt, a.passes, cached=False)
            r["first_call"] = {"s_per_call": med, "drawings_per_s": n / med, "passes_s": ts}
            med, ts = timed_calls(builders, opt, a.passes, cached=True)
            r["steady_call"] = {"s_per_call": med, "drawings_per_s": n / med, "passes_s": ts}
            ps = []
            for _ in range(a.passes):
                t0 = time.perf_counter()
                fk.systems_layout(probe, opt)
                ps.append(time.perf_counter() - t0)
            r["cross_drawing_plan_host_s"] = statistics.median(ps)
            # (a process of its own: events of a later profiler session in one process were found missing)
            cmd = [sys.executable, os.path.abspath(__file__), "--split", name, opt] + (["--quick"] if a.quick else [])
            r["device"] = json.loads(subprocess.run(cmd, capture_output=True, text=True, check=True).stdout.strip().splitlines()[-1])
            sample = builders[:: max(1, n // n_loop)][:n_loop]
            r["per_drawing_loop"] = {"drawings": len(sample) - 1, "drawings_per_s": loop_rate(sample, opt)}
            r["speedup_steady_vs_loop"] = r["steady_call"]["drawings_per_s"] / r["per_drawing_loop"]["drawings_per_s"]
            d["optimizers"][opt] = r
            print(name, opt, json.dumps({k: v for k, v in r.items() if k != "device"}, default=str)[:700], flush=True)
            print("   device split", {k: v for k, v in r["device"].items() if k != "kernels"}, flush=True)
        res["workloads"][name] = d
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(res, f, indent=1)
    print("wrote", a.out)


if __name__ == "__main__":
    main()
