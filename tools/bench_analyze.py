"""System::analyze on one B200: the global-memory kernels (one CTA per sketch, a cooperative group of CTAs per sketch)
against the oracle on one core of the same host.

    python tools/bench_analyze.py [--out FILE] [--passes K]

Per shape: the kernel time (torch.profiler over CUDA activities, summed over the analyze kernels of one call), the
end-to-end call time (host clock around the call, which ends in a stream synchronise), the L2 overwritten with a 256 MB
write before every pass, medians of --passes passes.  Single systems go through Topology.batch_analyze(n=1) and
System.analyze (fk_system_analyze: its topology creation included).  Bytes streamed are computed from the shape and
the flags: the elimination of row i reads rows 0 .. i-1 (8 n_vars bytes each), the Jordan step of an independent row i
reads and writes them.  The oracle runs in child processes pinned to one core each, concurrently with the GPU part; a
shape it does not finish within --oracle-timeout seconds is recorded as not measured.
"""
import argparse
import json
import multiprocessing as mp
import os
import statistics
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from fiksi_b200 import workloads as wl  # noqa: E402

HBM_BYTES_PER_S = 7.7e12
L2_BYTES = 126e6


def triangles(count):
    """50 unconnected triangles: 3 points and 3 distances each."""
    coords, kind, idx, dist = [], [], [], []
    for k in range(count):
        p = len(coords) // 2
        coords += [3.0 * k, 0.0, 3.0 * k + 1.1, 0.05 * k, 3.0 * k + 0.4, 1.0 + 0.01 * k]
        for a, b, d in ((p, p + 1, 1.0), (p + 1, p + 2, 1.2), (p + 2, p, 1.1)):
            kind.append(1)
            idx.append([2 * a, 2 * b, 0, 0])
            dist.append(d)
    return wl.Workload(f"triangles{count}", kind, idx, np.arange(len(coords)), np.arange(len(kind)), np.array([coords]), np.array([dist]))


SINGLES = {
    "hinged64": lambda: wl.hinged_triangles(64),
    "triangles50": lambda: triangles(50),
    "lattice24x20": lambda: wl.lattice(24, 20),
    "lattice32x32": lambda: wl.lattice(32, 32),
    "lattice48x40": lambda: wl.lattice(48, 40),
    "lattice64x50": lambda: wl.lattice(64, 50),
}


def _oracle_job(args):
    name, core = args
    os.sched_setaffinity(0, {core})
    import oracle
    w = (SINGLES[name] if name in SINGLES else (lambda: wl.hinged_triangles(45)))()
    t0 = time.perf_counter()
    oracle.analyze(w.raw_vars[0], w.kind, w.idx, w.raw_param[0])
    return name, time.perf_counter() - t0


def streamed_bytes(n_vars, n_expr, flags):
    ns = min(n_vars, n_expr)
    rows = np.arange(ns, dtype=np.float64)
    elim = 8.0 * n_vars * rows.sum()
    jordan = 16.0 * n_vars * rows[np.asarray(flags[:ns], dtype=bool)].sum()
    return elim + jordan, 8.0 * ns * ((n_vars + 31) // 32 * 32)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None, help="write the JSON result here (it is printed either way)")
    ap.add_argument("--passes", type=int, default=5)
    ap.add_argument("--oracle-timeout", type=float, default=420.0)
    ap.add_argument("--oracle", default="hinged64,triangles50,lattice24x20,lattice32x32,lattice48x40,hinged45")
    args = ap.parse_args()

    import torch
    from torch.profiler import ProfilerActivity, profile

    import fiksi_b200 as fk
    import fiksi_b200.system as fsys
    if not torch.cuda.is_available() or fk.device_count() < 1:
        raise SystemExit("bench_analyze needs a CUDA device")
    ncpu = os.cpu_count() or 1
    jobs = [(name, 2 + k % max(1, ncpu - 2)) for k, name in enumerate(args.oracle.split(",") if args.oracle else [])]
    pool = mp.get_context("spawn").Pool(len(jobs)) if jobs else None
    pending = pool.map_async(_oracle_job, jobs) if pool else None
    t_oracle0 = time.time()

    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()
    out = {"gpu": torch.cuda.get_device_name(0), "nvidia_smi": smi[0] if smi else "unavailable",
           "passes": args.passes, "l2_flush": "256 MB write before every pass", "singles": {}, "batches": {}, "boundaries": {}}
    flush = torch.empty(32 * 1024 * 1024, dtype=torch.float64, device="cuda")

    def topology(w):
        return fk.Topology.from_arrays(w.n_vars, w.kind, w.idx, np.arange(w.n_vars), np.arange(len(w.kind)))

    def kernel_ms(fn):
        flush.zero_()
        torch.cuda.synchronize()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            fn()
            torch.cuda.synchronize()
        us = sum(e.time_range.elapsed_us() for e in prof.events() if "analyze" in e.name and e.device_type.name == "CUDA")
        return us / 1e3

    def wall_ms(fn):
        flush.zero_()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        fn()
        return (time.perf_counter() - t0) * 1e3

    def med(fn, passes):
        fn()  # warm-up: module load, workspace growth
        return statistics.median(fn() for _ in range(passes))

    def forced(kernel):
        if kernel is None:
            os.environ.pop("FK_ANALYZE_KERNEL", None)
        else:
            os.environ["FK_ANALYZE_KERNEL"] = kernel

    def measure(w, n, kernel=None, passes=None):
        passes = passes or args.passes
        forced(kernel)
        topo = topology(w)
        v, p = np.ascontiguousarray(w.raw_vars[:n]), np.ascontiguousarray(w.raw_param[:n])
        call = lambda: topo.batch_analyze(v, p)  # noqa: E731
        flags = call()
        rec = {"kernel": topo.analyze_kernel(n), "n": n, "n_vars": int(w.n_vars), "n_expr": int(len(w.kind)),
               "kernel_ms": med(lambda: kernel_ms(call), passes), "call_ms": med(lambda: wall_ms(call), passes)}
        forced(None)
        if not rec["kernel_ms"]:  # the profiler recorded no analyze kernel: rates below come from the call time
            rec["kernel_ms"] = None
        t = rec["kernel_ms"] or rec["call_ms"]
        rec["rates_from"] = "kernel_ms" if rec["kernel_ms"] else "call_ms"
        total, matrix = streamed_bytes(w.n_vars, len(w.kind), flags[0])
        rec["matrix_bytes"] = matrix
        rec["matrix_in"] = "L2" if matrix * n <= L2_BYTES else "HBM"  # all matrices of the call
        rec["streamed_bytes_per_sketch"] = total
        rec["achieved_bytes_per_s"] = total * n / (t * 1e-3)
        rec["share_of_hbm_7_7_tb_s"] = rec["achieved_bytes_per_s"] / HBM_BYTES_PER_S
        rec["sketches_per_s"] = n / (t * 1e-3)
        return rec, flags

    for name, make in SINGLES.items():
        w = make()
        big = w.n_vars >= 4000
        rec, flags = measure(w, 1, passes=1 if big else None)
        s = fsys.System()
        pts = [s.add_point(float(w.raw_vars[0, 2 * k]), float(w.raw_vars[0, 2 * k + 1])) for k in range(w.n_vars // 2)]
        for e in range(len(w.kind)):
            s.point_point_distance(pts[w.idx[e, 0] // 2], pts[w.idx[e, 1] // 2], float(w.raw_param[0, e]))
        rec["system_analyze_ms"] = med(lambda: wall_ms(s.analyze), 1 if big else args.passes)
        rec["system_analyze_found"] = len(s.analyze())
        assert rec["system_analyze_found"] == int((~flags[0]).sum())
        out["singles"][name] = rec
        print(name, json.dumps(rec), flush=True)

    for name, (make, n) in {"lattice24x20_x1024": (lambda: wl.lattice(24, 20, n_sketches=1024), 1024),
                            "lattice32x32_x256": (lambda: wl.lattice(32, 32, n_sketches=256), 256)}.items():
        rec, _ = measure(make(), n, passes=2)
        out["batches"][name] = rec
        print(name, json.dumps(rec), flush=True)

    # both sides of every selection boundary
    b = out["boundaries"]
    h45 = wl.hinged_triangles(45, n_sketches=1024)
    h45.raw_vars = h45.raw_vars + 0.01 * np.sin(np.arange(h45.raw_vars.size)).reshape(h45.raw_vars.shape)
    for k in ("warp", "cta", "group"):
        b[f"hinged45_x1024_{k}"] = measure(h45, 1024, k)[0]
    l24 = wl.lattice(24, 20, n_sketches=296)
    for n in (1, 74, 148, 296):
        for k in ("cta", "group"):
            b[f"lattice24x20_x{n}_{k}"] = measure(l24, n, k)[0]
    l48 = wl.lattice(48, 40)
    b["lattice48x40_x1_cta"] = measure(l48, 1, "cta", passes=1)[0]
    b["lattice48x40_x1_group"] = out["singles"]["lattice48x40"]
    for key, rec in b.items():
        print(key, json.dumps(rec), flush=True)

    oracle_s = {}
    if pending is not None:
        left = max(1.0, args.oracle_timeout - (time.time() - t_oracle0))
        try:
            oracle_s = dict(pending.get(timeout=left))
        except mp.TimeoutError:
            oracle_s = {}
        pool.terminate()
        pool.join()
    out["oracle_one_core_s"] = {name: oracle_s.get(name, "not measured (did not finish within the timeout)") for name, _ in jobs}
    out["oracle_one_core_s"]["lattice64x50"] = "not measured on this host"
    sp = out["speedup_vs_oracle_one_core"] = {}
    for name, rec in out["singles"].items():
        if isinstance(oracle_s.get(name), float):
            sp[name] = {"kernel": oracle_s[name] / ((rec["kernel_ms"] or rec["call_ms"]) * 1e-3), "call": oracle_s[name] / (rec["call_ms"] * 1e-3),
                        "system_analyze": oracle_s[name] / (rec["system_analyze_ms"] * 1e-3)}
    if isinstance(oracle_s.get("lattice24x20"), float):
        rec = out["batches"]["lattice24x20_x1024"]
        sp["lattice24x20_x1024"] = {"kernel": 1024 * oracle_s["lattice24x20"] / ((rec["kernel_ms"] or rec["call_ms"]) * 1e-3),
                                    "call": 1024 * oracle_s["lattice24x20"] / (rec["call_ms"] * 1e-3)}
    if isinstance(oracle_s.get("lattice32x32"), float):
        rec = out["batches"]["lattice32x32_x256"]
        sp["lattice32x32_x256"] = {"kernel": 256 * oracle_s["lattice32x32"] / ((rec["kernel_ms"] or rec["call_ms"]) * 1e-3),
                                   "call": 256 * oracle_s["lattice32x32"] / (rec["call_ms"] * 1e-3)}
    text = json.dumps(out, indent=1, sort_keys=True)
    if args.out:
        with open(args.out, "w") as f:
            f.write(text)
    else:
        print(text)
    print(json.dumps({"oracle_one_core_s": out["oracle_one_core_s"], "speedup": sp}, indent=1))


if __name__ == "__main__":
    main()
