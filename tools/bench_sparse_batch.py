"""Batched LM on the global sparse path (one CTA per sketch over the supernodal tree) against the per-system loop.

For lattices 30x20, 32x32, 48x40, 64x50 and the 1,000-point truss, each sketch with its own noise, it reports:
  device_resident   plan.run between CUDA events on resident inputs, L2 overwritten (256 MB write) before every pass
  end_to_end        fk_batch_solve_device from pinned host buffers, host clock around the (synchronous) call
  per_system_loop   fk_topology_lm_solve over 32 of the same sketches (the only way to solve them before)
  cpu_restatement   the oracle (the reference restated in C++) on one core over a small sample
  fp64              sum of factorisations x chol_flops over kernel time, against the measured DFMA peak
and the GPU name and power limit read in the same run.  Usage: python tools/bench_sparse_batch.py [--out FILE] [--passes K]
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

import torch  # noqa: E402

import fiksi_b200 as fk  # noqa: E402
from fiksi_b200 import workloads as wl  # noqa: E402
from fiksi_b200._lib import REPORT_DTYPE, lib  # noqa: E402

SHAPES = [("lattice30x20", 1024), ("lattice32x32", 1024), ("lattice48x40", 1024), ("lattice64x50", 256), ("truss1000", 1024)]
DECISIONS = ("exit_reason", "trace_hash", "outer_iters", "factorizations", "accepted", "lambda")


def workload(name, n):
    if name.startswith("truss"):
        return wl.truss(n, int(name[5:]))
    nx, ny = (int(a) for a in name[7:].split("x"))
    return wl.lattice(nx, ny, n_sketches=n)


def pinned(a):
    a = np.ascontiguousarray(a)
    buf = lib().fk_host_alloc(C.c_size_t(max(a.nbytes, 1)))
    h = np.ctypeslib.as_array((C.c_uint8 * max(a.nbytes, 1)).from_address(buf))[:a.nbytes].view(a.dtype).reshape(a.shape)
    h[...] = a
    return h, buf


def gpu_identity():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return {"torch_name": torch.cuda.get_device_name(0), "nvidia_smi": q.stdout.strip().splitlines()[0] if q.returncode == 0 else q.stderr.strip()}


def measure(name, n, passes, oracle):
    w = workload(name, n)
    v, p, _ = w.prepare()
    topo = fk.Topology.from_arrays(w.n_vars, w.kind, w.idx, w.free_vars, w.rows)
    info = topo.info
    sn = topo.supernodal()["info"]
    assert info["path"] == 2 and topo.batch_kernel(n) == "sparse_batch"
    nf = w.free_vars.size
    # device resident
    plan = topo.plan(n)
    plan.upload(v, p)
    out = np.zeros((n, nf))
    rep = np.zeros(n, REPORT_DTYPE)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
    plan.run()  # warm-up (module load, first touch of the workspace)
    lib().fk_batch_plan_sync(plan._h)
    times = []
    for _ in range(passes):
        flush.fill_(1)
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        plan.run()
        b.record()
        b.synchronize()
        times.append(a.elapsed_time(b) * 1e-3)
    plan.download(out, rep)
    lib().fk_batch_plan_sync(plan._h)
    plan.close()
    kern = float(np.median(times))
    # end to end from pinned buffers
    hv, bv = pinned(v)
    hp, bp = pinned(p)
    ho, bo = pinned(np.zeros((n, nf)))
    hr, br = pinned(np.zeros(n, REPORT_DTYPE))
    topo.batch_solve_into(0, n, hv.ctypes.data, hp.ctypes.data, ho.ctypes.data, hr.ctypes.data)
    e2e = []
    for _ in range(max(3, passes // 2)):
        t0 = time.perf_counter()
        topo.batch_solve_into(0, n, hv.ctypes.data, hp.ctypes.data, ho.ctypes.data, hr.ctypes.data)
        e2e.append(time.perf_counter() - t0)
    same_as_plan = ho.tobytes() == out.tobytes() and hr.tobytes() == rep.tobytes()
    for b in (bv, bp, bo, br):
        lib().fk_host_free(C.c_void_p(b))
    # per-system loop over 32 of the same sketches (first solve warms the solver up)
    topo.lm_solve(v[0], p[0], v[0][w.free_vars])
    loop_n = min(32, n)
    decisions_equal, max_rel = 0, 0.0
    t0 = time.perf_counter()
    singles = [topo.lm_solve(v[k], p[k], v[k][w.free_vars]) for k in range(loop_n)]
    loop_s = (time.perf_counter() - t0) / loop_n
    for k, (xs, rs) in enumerate(singles):
        decisions_equal += all(rep[k][f] == rs[f] for f in DECISIONS)
        max_rel = max(max_rel, float(np.max(np.abs(out[k] - xs)) / max(np.max(np.abs(xs)), 1e-300)))
    # CPU restatement, one core
    cpu_n = 2
    t0 = time.perf_counter()
    for k in range(cpu_n):
        op, keep = oracle.make_problem(v[k], w.kind, w.idx, p[k], w.free_vars, w.rows)
        oracle.lm_solve(op, v[k][w.free_vars])
    cpu_s = (time.perf_counter() - t0) / cpu_n
    facs = int(np.sum(rep["factorizations"]))
    flops = facs * float(info["chol_flops"])
    return {
        "shape": name, "sketches": n, "n_free": info["n_free"], "n_rows": info["n_rows"], "max_front": sn["max_front"],
        "supernodes": sn["n_supernodes"], "chol_flops": info["chol_flops"], "factorizations_total": facs,
        "exits": {str(e): int(c) for e, c in zip(*np.unique(rep["exit_reason"], return_counts=True))},
        "device_resident": {"kernel_s_median": kern, "kernel_s_all": times, "sketches_per_s": n / kern},
        "end_to_end": {"s_median": float(np.median(e2e)), "sketches_per_s": n / float(np.median(e2e)), "bit_identical_to_plan": same_as_plan},
        "per_system_loop": {"sketches": loop_n, "s_per_sketch": loop_s, "sketches_per_s": 1.0 / loop_s,
                            "decisions_equal": decisions_equal, "max_rel_diff_to_batch": max_rel},
        "cpu_restatement": {"sketches": cpu_n, "s_per_sketch": cpu_s},
        "speedup_resident_over_loop": (n / kern) * loop_s,
        "fp64": {"tflops": flops / kern * 1e-12},
    }


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--passes", type=int, default=10)
    ap.add_argument("--shapes", default=",".join(s for s, _ in SHAPES))
    a = ap.parse_args()
    import oracle
    oracle.build()
    peak = fk.fp64_peak_tflops(0)
    res = {"gpu": gpu_identity(), "fp64_peak_tflops_measured": peak, "results": []}
    want = a.shapes.split(",")
    for name, n in SHAPES:
        if name not in want:
            continue
        r = measure(name, n, a.passes, oracle)
        r["fp64"]["share_of_measured_peak"] = r["fp64"]["tflops"] / peak
        res["results"].append(r)
        print(json.dumps({k: r[k] for k in ("shape", "sketches", "speedup_resident_over_loop")} | {"resident_per_s": r["device_resident"]["sketches_per_s"]}), flush=True)
    text = json.dumps(res, indent=1)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(text + "\n")
    print(text)


if __name__ == "__main__":
    main()
