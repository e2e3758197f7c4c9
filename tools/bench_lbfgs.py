"""Optimizer::LBfgs on one B200: the tile kernel (state in shared memory) and the CTA kernel (one CTA per sketch, state in
global memory) on the same shapes, batches and single systems beyond the tile kernel's wall, against the oracle on one
core of the same host.

    python tools/bench_lbfgs.py [--out FILE] [--passes K]

Device-resident rates: a batch plan uploaded once, then the host clock around plan.run_lbfgs / run_lbfgs_global and a
device synchronise, the L2 overwritten with a 256 MB write before every pass, medians of --passes passes.  Host-buffer
rates: fk_lbfgs_solve_batch over a list of problems (grouping through the topology cache, copies both ways included).
Single systems: fk_lbfgs_solve.  The card's name and power limit are read in the same call.  The oracle runs one sketch
per shape in child processes pinned to one core each, concurrently with the GPU part; a shape it does not finish within
--oracle-timeout seconds, and every shape above 48x40 (its dense m x n Jacobian), is recorded as not measured.
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

# name: (workload maker of n sketches, batch size)
BOTH = {
    "truss20_x65536": (lambda n: wl.truss(n), 65536),
    "cad_mix_x100000": (lambda n: wl.cad_mix(n), 100000),
    "hinged64_x1024": (lambda n: wl.hinged_triangles(64, n_sketches=n), 1024),
}
BEYOND = {
    "lattice10x8_x1024": (lambda n: wl.lattice(10, 8, n_sketches=n), 1024),
    "lattice24x20_x1024": (lambda n: wl.lattice(24, 20, n_sketches=n), 1024),
    "lattice32x32_x1024": (lambda n: wl.lattice(32, 32, n_sketches=n), 1024),
    "lattice48x40_x1024": (lambda n: wl.lattice(48, 40, n_sketches=n), 1024),
    "truss1000_x1024": (lambda n: wl.truss(n, n_points=1000), 1024),
    "lattice64x50_x256": (lambda n: wl.lattice(64, 50, n_sketches=n), 256),
}
SINGLES = {
    "lattice32x32": lambda: wl.lattice(32, 32),
    "lattice48x40": lambda: wl.lattice(48, 40),
    "lattice64x50": lambda: wl.lattice(64, 50),
    "lattice150x120": lambda: wl.lattice(150, 120),
    "lattice400x250": lambda: wl.lattice(400, 250),
}
ORACLE = {  # one sketch each; the oracle's dense Jacobian makes shapes above 48x40 impractical
    "truss20": lambda: wl.truss(1), "cad_mix": lambda: wl.cad_mix(1), "hinged64": lambda: wl.hinged_triangles(64),
    "lattice10x8": lambda: wl.lattice(10, 8), "lattice24x20": lambda: wl.lattice(24, 20), "lattice32x32": lambda: wl.lattice(32, 32),
    "lattice48x40": lambda: wl.lattice(48, 40), "truss1000": lambda: wl.truss(1, n_points=1000),
}
ORACLE_OF = {"truss20_x65536": "truss20", "cad_mix_x100000": "cad_mix", "hinged64_x1024": "hinged64", "lattice10x8_x1024": "lattice10x8",
             "lattice24x20_x1024": "lattice24x20", "lattice32x32_x1024": "lattice32x32", "lattice48x40_x1024": "lattice48x40",
             "truss1000_x1024": "truss1000"}


def _oracle_job(args):
    name, core = args
    os.sched_setaffinity(0, {core})
    import oracle
    w = ORACLE[name]()
    v, p, _ = w.prepare()
    op, keep = oracle.make_problem(v[0], w.kind, w.idx, p[0], w.free_vars, w.rows)
    t0 = time.perf_counter()
    oracle.lbfgs_solve(op, v[0][w.free_vars])
    return name, time.perf_counter() - t0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None, help="write the JSON result here (it is printed either way)")
    ap.add_argument("--passes", type=int, default=5)
    ap.add_argument("--oracle-timeout", type=float, default=900.0)
    args = ap.parse_args()

    import torch

    import fiksi_b200 as fk
    from fiksi_b200._lib import REPORT_DTYPE, lib, make_problem
    if not torch.cuda.is_available() or fk.device_count() < 1:
        raise SystemExit("bench_lbfgs needs a CUDA device")
    ncpu = os.cpu_count() or 1
    jobs = [(name, 2 + k % max(1, ncpu - 2)) for k, name in enumerate(ORACLE)]
    pool = mp.get_context("spawn").Pool(len(jobs))
    pending = pool.map_async(_oracle_job, jobs)
    t_oracle0 = time.time()

    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()
    out = {"gpu": torch.cuda.get_device_name(0), "nvidia_smi": smi[0] if smi else "unavailable", "passes": args.passes,
           "l2_flush": "256 MB write before every pass", "both_kernels": {}, "beyond_the_wall": {}, "singles": {}}
    flush = torch.empty(32 * 1024 * 1024, dtype=torch.float64, device="cuda")

    def timed(fn):
        flush.zero_()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        fn()
        torch.cuda.synchronize()
        return time.perf_counter() - t0

    def med(fn, passes):
        fn()  # warm-up: module load, workspace growth
        return statistics.median(timed(fn) for _ in range(passes))

    def topology(w):
        return fk.Topology.from_arrays(w.n_vars, w.kind, w.idx, w.free_vars, w.rows)

    def resident(w, n, kernels, passes):
        v, p, _ = w.prepare()
        topo = topology(w)
        plan = topo.plan(n)
        plan.upload(v, p)
        lib().fk_batch_plan_sync(plan._h)
        rec = {"n": n, "n_free": int(topo.info["n_free"]), "path": int(topo.info["path"]), "lbfgs_kernel": topo.lbfgs_kernel(n)}
        outs = {}
        for k in kernels:
            run = plan.run_lbfgs if k == "tile" else plan.run_lbfgs_global
            s = med(lambda: (run(), lib().fk_batch_plan_sync(plan._h)), passes)
            rec[f"{k}_s"] = s
            rec[f"{k}_sketches_per_s"] = n / s
            x = np.zeros((n, topo.info["n_free"]))
            rep = np.zeros(n, REPORT_DTYPE)
            plan.download(x, rep)
            lib().fk_batch_plan_sync(plan._h)
            outs[k] = (x, rep)
        if len(kernels) == 2:
            rec["bit_identical"] = bool(outs["tile"][0].tobytes() == outs["cta"][0].tobytes() and outs["tile"][1].tobytes() == outs["cta"][1].tobytes())
            rec["faster"] = "tile" if rec["tile_s"] < rec["cta_s"] else "cta"
        plan.close()
        return rec, v, p

    for name, (make, n) in BOTH.items():
        rec, _, _ = resident(make(n), n, ("tile", "cta"), args.passes)
        out["both_kernels"][name] = rec
        print(name, json.dumps(rec), flush=True)

    for name, (make, n) in BEYOND.items():
        w = make(n)
        rec, v, p = resident(w, n, ("cta",), 3)
        probs = [make_problem(v[k], w.kind, w.idx, p[k], w.free_vars, w.rows) for k in range(n)]
        x0 = [v[k][w.free_vars] for k in range(n)]
        s = med(lambda: fk.lbfgs_solve_batch([q for q, _ in probs], x0), 3)
        rec["host_buffers_s"] = s
        rec["host_buffers_sketches_per_s"] = n / s
        out["beyond_the_wall"][name] = rec
        print(name, json.dumps(rec), flush=True)

    for name, make in SINGLES.items():
        w = make()
        v, p, _ = w.prepare()
        prob, keep = make_problem(v[0], w.kind, w.idx, p[0], w.free_vars, w.rows)
        x0 = v[0][w.free_vars]
        big = w.n_vars > 10000
        _, rep = fk.lbfgs_solve(prob, x0)
        s = med(lambda: fk.lbfgs_solve(prob, x0), 1 if big else 3)
        rec = {"n_free": int(len(w.free_vars)), "s": s, "report": {k: (float(v_) if isinstance(v_, float) else int(v_)) for k, v_ in rep.items()}}
        out["singles"][name] = rec
        print(name, json.dumps(rec), flush=True)

    left = max(1.0, args.oracle_timeout - (time.time() - t_oracle0))
    try:
        oracle_s = dict(pending.get(timeout=left))
    except mp.TimeoutError:
        oracle_s = {}
    pool.terminate()
    pool.join()
    out["oracle_one_core_s"] = {name: oracle_s.get(name, "not measured (did not finish within the timeout)") for name in ORACLE}
    for name in ("lattice64x50", "lattice150x120", "lattice400x250"):
        out["oracle_one_core_s"][name] = "not measured (the oracle's dense m x n Jacobian)"
    sp = out["speedup_vs_oracle_one_core"] = {}
    for group in ("both_kernels", "beyond_the_wall"):
        for name, rec in out[group].items():
            o = oracle_s.get(ORACLE_OF.get(name))
            if isinstance(o, float):
                sp[name] = {k[:-2]: rec["n"] * o / rec[k] for k in ("tile_s", "cta_s", "host_buffers_s") if k in rec}
    for name, rec in out["singles"].items():
        if isinstance(oracle_s.get(name), float):
            sp[name] = {"single": oracle_s[name] / rec["s"]}
    out["targets"] = {
        "lattice24x20_x1024 >= 100x one core": sp.get("lattice24x20_x1024", {}).get("cta", "not measured"),
        "lattice32x32_x1024 >= 100x one core": sp.get("lattice32x32_x1024", {}).get("cta", "not measured"),
        "single lattice48x40 >= 10x one core": sp.get("lattice48x40", {}).get("single", "not measured"),
    }
    text = json.dumps(out, indent=1, sort_keys=True)
    if args.out:
        with open(args.out, "w") as f:
            f.write(text)
    print(json.dumps({"oracle_one_core_s": out["oracle_one_core_s"], "speedup": sp, "targets": out["targets"]}, indent=1))


if __name__ == "__main__":
    main()
