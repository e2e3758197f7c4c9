#!/usr/bin/env python
"""Benchmark of the Fiksi solve path on B200.

    python bench.py --gpus N --steps K --warmup W            # our arm (CUDA, one rank per GPU)
    python bench.py --impl reference --gpus N --steps K ...  # reference arm: CPU restatement
    python bench.py ... --dump-outputs DIR                   # also write the last timed step's results to DIR/<name>.npy

Workload: BASELINE.json configs[1] — 65,536 randomly perturbed 20-point rigid distance trusses
(40 free variables, 37 point-point-distance rows) per GPU, one sketch per warp, solved to the
reference's own convergence criteria.  A "step" is one Levenberg–Marquardt solve of the whole
batch.  `value` = sketches/s with the inputs already resident in HBM; `e2e` = the same through the
host-buffer C-ABI call (fk_batch_solve_device) with pinned host buffers, H2D + D2H inside the timed
region.  Weak scaling: every rank solves its own 65,536 sketches (different seeds), no collective
on the data path (sketches are independent; SURVEY §8e).
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

N_PER_GPU = 65536
METRIC = "lm_solved_sketches_per_sec"
WORKLOAD = ("configs[1]: batch of 65,536 perturbed 20-point rigid distance trusses per GPU "
            "(40 free vars, 37 PPD rows, 148 J nnz)")
UNIT = "sketches/s"


def _peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        d = json.load(open(path))
        return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md)."""

    FIELDS = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
              "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index = index
        self.rows = []
        self._stop = threading.Event()
        self._t = threading.Thread(target=self._run, daemon=True)

    def _run(self):
        while not self._stop.is_set():
            try:
                out = subprocess.run(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.FIELDS}",
                                      "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=5).stdout
                parts = [x.strip() for x in out.strip().split(",")]
                if len(parts) >= 6:
                    self.rows.append(parts)
            except Exception:
                pass
            self._stop.wait(0.1)

    def __enter__(self):
        self._t.start()
        return self

    def __exit__(self, *a):
        self._stop.set()
        self._t.join(timeout=6)

    def summary(self):
        if not self.rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unsampled"]}
        sm = sorted(float(r[0]) for r in self.rows if r[0].replace(".", "").isdigit())
        mx = max((float(r[1]) for r in self.rows if r[1].replace(".", "").isdigit()), default=None)
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({names[i] for r in self.rows for i in range(4) if r[2 + i].lower().startswith("active")})
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx, "reasons": reasons, "samples": len(self.rows)}


def cpu_reference_run(n_sample, threads, first=0):
    """The reference's CPU algorithm (oracle restatement; the Rust reference cannot be built here:
    no Rust toolchain) on `threads` host threads, one sketch per task."""
    import oracle
    from fiksi_b200 import workloads as wl
    w = wl.truss(n_sample, first=first)
    v, p, scale = w.prepare()
    op, keep = oracle.make_problem(v[0], w.kind, w.idx, p[0], w.free_vars, w.rows)
    x, rep, secs = oracle.lm_solve_batch_uniform(op, v, p, threads=threads)
    return n_sample / secs, secs, x, rep


def solve_outputs(prefix, x, rep):
    """What a caller of a batched solve receives, as float64 arrays: the solved free variables and every report field
    (the counters are exact in float64; the 64-bit trace hash goes as its two 32-bit halves)."""
    import numpy as np
    out = {prefix + "x": np.array(x, dtype=np.float64)}
    for k in ("exit_reason", "outer_iters", "factorizations", "accepted", "ssr", "lambda"):
        out[prefix + k] = rep[k].astype(np.float64)
    out[prefix + "trace_hash_hi"] = (rep["trace_hash"] >> np.uint64(32)).astype(np.float64)
    out[prefix + "trace_hash_lo"] = (rep["trace_hash"] & np.uint64(0xFFFFFFFF)).astype(np.float64)
    return out


def dump_outputs(out_dir, arrays):
    import numpy as np
    total = sum(a.nbytes for a in arrays.values())
    if total > 64 << 20:
        raise SystemExit(f"--dump-outputs: {total} bytes of outputs, more than 64 MB")
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


def run_reference(args, rank, world):
    if rank != 0:
        return
    threads = os.cpu_count() or 1
    n_sample = N_PER_GPU  # the same 65,536 sketches per step as our arm (one step is ~0.3 s on 16 host cores)
    times = []
    for k in range(args.warmup + args.steps):
        rate, secs, x, rep = cpu_reference_run(n_sample, threads, first=k * n_sample)
        if k >= args.warmup:
            times.append(secs)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, solve_outputs("", x, rep))
    total = sum(times)
    value = n_sample * len(times) / total
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * total / len(times), "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": WORKLOAD,
                   "sketches_per_gpu": n_sample, "sketches_per_step": n_sample,
                   "note": "the reference's CPU algorithm (oracle port; no Rust toolchain here) on all host threads, whole 65,536-sketch steps"},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": threads, "kind": "port",
                         "sample": f"{n_sample} sketches per step, {len(times)} steps, one sketch per task on {threads} threads"},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))


def bind_near_gpu(torch, local_rank):
    """Multi-rank runs: keep this rank's threads (and so its pinned host buffers, which are placed on the
    allocating thread's NUMA node) on the CPU cores NVML reports as local to its GPU.  Returns the number of
    cores bound to, or None when NVML gives no answer."""
    try:
        import pynvml
        pynvml.nvmlInit()
        pr = torch.cuda.get_device_properties(local_rank)
        try:
            bus = "%08x:%02x:%02x.0" % (pr.pci_domain_id, pr.pci_bus_id, pr.pci_device_id)
            h = pynvml.nvmlDeviceGetHandleByPciBusId(bus.encode())
        except Exception:  # noqa: BLE001
            h = pynvml.nvmlDeviceGetHandleByIndex(local_rank)
        words = ((os.cpu_count() or 64) + 63) // 64
        mask = pynvml.nvmlDeviceGetCpuAffinity(h, words)
        cpus = {64 * i + b for i, m in enumerate(mask) for b in range(64) if (int(m) >> b) & 1}
        cpus &= os.sched_getaffinity(0)
        if not cpus or cpus == os.sched_getaffinity(0):
            return None
        os.sched_setaffinity(0, cpus)
        return len(cpus)
    except Exception:  # noqa: BLE001
        return None


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-extras", action="store_true", help="skip the assembly / FP64 side measurements")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the last timed step computed as DIR/<name>.npy (float64, rank 0's sketches): x and "
                         "the report fields of the device-resident solve (of the CPU restatement with --impl reference), "
                         "and the same of the streamed end-to-end call as e2e_*")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))

    if args.impl == "reference":
        run_reference(args, rank, world)
        return

    import numpy as np
    import torch
    import torch.distributed as dist

    import fiksi_b200 as fk
    from fiksi_b200 import workloads as wl

    if not torch.cuda.is_available() or fk.device_count() < 1:
        raise SystemExit("bench.py needs a CUDA device: fiksi_b200 has no CPU fallback")
    torch.cuda.set_device(local_rank)
    bound = bind_near_gpu(torch, local_rank) if world > 1 else None
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- workload: this rank's 65,536 sketches ------------------------------------------------------
    n = N_PER_GPU
    w = wl.truss(n, first=rank * n)
    v, p, scale = w.prepare()
    topo = fk.Topology.from_arrays(w.n_vars, w.kind, w.idx, w.free_vars, w.rows)
    info = topo.info
    plan = topo.plan(n, device=local_rank)
    hv = torch.from_numpy(v).pin_memory()
    hp = torch.from_numpy(p).pin_memory()
    hout = torch.empty((n, info["n_free"]), dtype=torch.float64).pin_memory()
    hrep = torch.empty((n, 40), dtype=torch.uint8).pin_memory()
    stream = torch.cuda.current_stream().cuda_stream
    plan.upload_ptr(n, hv.data_ptr(), hp.data_ptr(), stream)
    flush = torch.empty(512 * 1024 * 1024, dtype=torch.uint8, device="cuda")  # > 126 MB L2
    torch.cuda.synchronize()

    for _ in range(args.warmup):
        plan.run(stream)
    barrier()

    # ---- device-resident timing: K steps, L2 flushed between steps, CUDA events on the launch stream
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    launches0 = plan.launches
    with ClockSampler(local_rank) as clocks:
        wall0 = time.perf_counter()
        for a, b in ev:
            flush.zero_()
            a.record()
            plan.run(stream)
            b.record()
        barrier()
        wall = time.perf_counter() - wall0
    step_ms = [a.elapsed_time(b) for a, b in ev]
    total_ms = float(sum(step_ms))
    gpu_launches = plan.launches - launches0
    plan.download_ptr(hout.data_ptr(), hrep.data_ptr(), stream)
    torch.cuda.synchronize()
    rep = hrep.numpy().view(fk.REPORT_DTYPE).reshape(-1).copy()  # the host buffers are reused by the measurements below
    outputs = solve_outputs("", hout.numpy(), rep) if args.dump_outputs else {}
    solved = float(np.mean(rep["ssr"] < 1e-8))
    fact = float(rep["factorizations"].sum())

    # ---- end-to-end through the host-buffer C-ABI calls ------------------------------------------------------
    # (1) the System::solve-level call: RAW variables in, scale + seeded perturbation + LM + write-back on the device,
    #     UNSCALED solved variables out (fk_batch_system_solve; the copies of a truss share one row of distances);
    # (2) the levenberg_marquardt-level call on inputs the host has already scaled and perturbed (fk_batch_solve_device).
    hraw = torch.from_numpy(w.raw_vars).pin_memory()
    shared_row = bool(np.all(w.raw_param == w.raw_param[0]))
    hrawp = torch.from_numpy(np.ascontiguousarray(w.raw_param[0] if shared_row else w.raw_param)).pin_memory()

    def e2e_system():
        topo.batch_system_solve_into(local_rank, n, hraw.data_ptr(), hrawp.data_ptr(), hout.data_ptr(), hrep.data_ptr(), shared_param=shared_row)

    def e2e_prepared():
        topo.batch_solve_into(local_rank, n, hv.data_ptr(), hp.data_ptr(), hout.data_ptr(), hrep.data_ptr())
    e2e_steps = args.steps
    e2e_secs = []
    for fn in (e2e_system, e2e_prepared):
        for _ in range(2):
            fn()
        barrier()
        t0 = time.perf_counter()
        for _ in range(e2e_steps):
            fn()
        barrier()
        e2e_secs.append(time.perf_counter() - t0)
    e2e_s, e2e_prep_s = e2e_secs
    # (1b) the same batches streamed two deep through the two halves of the call (fk_batch_system_solve_begin / _wait): step i + 1 is
    #      enqueued before step i is waited for, so the first upload of one step and the last download of the other run beside
    #      kernels instead of beside an idle device.  Every step still copies its inputs in and its results out inside the timed
    #      region; consecutive steps write to alternating output buffers.
    hout2 = torch.empty_like(hout).pin_memory()
    hrep2 = torch.empty_like(hrep).pin_memory()
    outs = ((hout, hrep), (hout2, hrep2))

    def begin(i):
        return topo.batch_system_solve_begin(local_rank, n, hraw.data_ptr(), hrawp.data_ptr(), outs[i & 1][0].data_ptr(), outs[i & 1][1].data_ptr(),
                                             shared_param=shared_row)
    for i in range(2):
        topo.batch_system_solve_wait(begin(i), local_rank)
    barrier()
    t0 = time.perf_counter()
    prev = begin(0)
    for i in range(1, e2e_steps):
        cur = begin(i)
        topo.batch_system_solve_wait(prev, local_rank)
        prev = cur
    topo.batch_system_solve_wait(prev, local_rank)
    barrier()
    e2e_stream_s = time.perf_counter() - t0
    if args.dump_outputs:
        last_out, last_rep = outs[(e2e_steps - 1) & 1]
        outputs.update(solve_outputs("e2e_", last_out.numpy(), last_rep.numpy().view(fk.REPORT_DTYPE).reshape(-1)))
    streamed_same = bool(np.array_equal(hout2.numpy(), hout.numpy()) and np.array_equal(hrep2.numpy(), hrep.numpy()))
    rep_sys = hrep.numpy().view(fk.REPORT_DTYPE).reshape(-1).copy()
    e2e_system()
    same_as_resident = bool(np.array_equal(hrep.numpy().view(fk.REPORT_DTYPE).reshape(-1)["trace_hash"], rep["trace_hash"]))
    del rep_sys

    # ---- host-copy ceiling: the same bytes as one e2e step, H2D and D2H concurrently on two streams, every rank at
    # once (what the box's host<->device path can carry when nothing is computed) ---------------------------------
    h2d = 8 * n * info["n_vars"] + 8 * info["n_expr"] * (1 if shared_row else n)
    d2h = 8 * n * info["n_free"] + 40 * n
    h2d_prepared = 8 * n * (info["n_vars"] + info["n_expr"])
    dv = torch.empty(v.shape, dtype=torch.float64, device="cuda")
    dp = torch.empty(hrawp.shape, dtype=torch.float64, device="cuda")
    dout = torch.empty((n, info["n_free"]), dtype=torch.float64, device="cuda")
    drep = torch.empty((n, 40), dtype=torch.uint8, device="cuda")
    s_in, s_out = torch.cuda.Stream(), torch.cuda.Stream()

    def copy_step():
        with torch.cuda.stream(s_in):
            dv.copy_(hraw, non_blocking=True)
            dp.copy_(hrawp, non_blocking=True)
        with torch.cuda.stream(s_out):
            hout.copy_(dout, non_blocking=True)
            hrep.copy_(drep, non_blocking=True)
    for _ in range(2):
        copy_step()
    barrier()
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        copy_step()
    barrier()
    copy_s = time.perf_counter() - t0
    del dv, dp, dout, drep

    t = torch.tensor([total_ms, e2e_s, copy_s, e2e_prep_s], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    total_ms, e2e_s, copy_s, e2e_prep_s = float(t[0]), float(t[1]), float(t[2]), float(t[3])

    value = world * n * args.steps / (total_ms * 1e-3)
    e2e_value = world * n * e2e_steps / e2e_s
    e2e_stream_value = world * n * e2e_steps / e2e_stream_s
    copy_ceiling = world * n * e2e_steps / copy_s
    which = topo.batch_kernel(n)
    uses_sketch_kernel = which != "tile"
    kernel_name = {"sketch": "fk_batch_lm_sketch_kernel (one thread per sketch, one warp per 32 sketches)",
                   "sketch_pair": "fk_batch_lm_sketch_pair_kernel (one thread per sketch, leader + helper warp per 32 sketches)",
                   "tile": "fk_batch_lm_kernel<%d,%d> (tile)" % (info["tile"], 1)}[which]

    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": total_ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f64", "data": "synthetic",
        "config": {"workload": WORKLOAD,
                   "sketches_per_gpu": n, "sketches_per_step": n, "kernel": kernel_name,
                   "state_doubles_per_sketch": topo.sketch_kernel_info()["state_doubles"] if uses_sketch_kernel else info["smem_bytes"] // 8,
                   "l2": "flushed between timed steps (512 MB memset)", "parallelism": f"sketch-sharded x{world}, no data-path collective",
                   "fraction_converged": solved, "wall_s_timed_region": wall,
                   "host_affinity": f"rank bound to the {bound} cores NVML reports local to its GPU" if bound else "unbound"},
        "e2e": {"value": e2e_stream_value, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                "steps": e2e_steps,
                "api": "fk_batch_system_solve_begin / fk_batch_system_solve_wait (the two halves of fk_batch_system_solve), batches streamed two deep: "
                       "raw variables in pinned host memory -> scale, seeded perturbation, LM solve and write-back on the device -> unscaled solved "
                       "variables + reports in pinned host memory (chunk pipeline on eight streams); step i + 1 is enqueued before step i is waited "
                       "for, so one step's first upload and the other's last download run beside kernels; every step copies its inputs in and "
                       "its results out inside the timed region, consecutive steps write to alternating output buffers",
                "results_equal_between_the_two_buffer_sets": streamed_same,
                "same_traces_as_device_resident_run": same_as_resident,
                "one_call_at_a_time": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                                       "api": "fk_batch_system_solve, each call returning before the next starts (the device idles while a call's "
                                              "first chunk arrives and while its last chunk leaves)"},
                "note": "streamed steps overlap each other's ends, which also removes the partial last wave of CTAs that every stand-alone launch of "
                        "the device-resident figure (value) pays, and value flushes L2 between steps: e2e can exceed value by a few per cent",
                "prepared_inputs": {"value": world * n * e2e_steps / e2e_prep_s, "unit": UNIT, "h2d_bytes_per_step": h2d_prepared,
                                    "api": "fk_batch_solve_device on inputs scaled and perturbed by the host (levenberg_marquardt-level call)"},
                "copy_ceiling": {"value": copy_ceiling, "unit": UNIT, "gb_per_s_all_ranks": world * (h2d + d2h) * e2e_steps / copy_s / 1e9,
                                 "how": "the step's H2D and D2H bytes copied concurrently on two streams by every rank, nothing computed"},
                "frac_of_copy_ceiling": e2e_stream_value / copy_ceiling},
        "gpu_launches": int(gpu_launches),
        "clocks": clocks.summary(),
    }

    # ---- configs[3] and configs[4] as north_star states them: every rank takes part -------------------------------
    if not args.no_extras:
        try:
            line["config4"] = config4_sharded(fk, wl, torch, dist, rank, world, local_rank, barrier)
        except Exception as e:  # noqa: BLE001
            line["config4"] = {"error": str(e)}
        try:
            line["config5"] = config5_sharded(fk, wl, torch, dist, rank, world, local_rank, barrier)
        except Exception as e:  # noqa: BLE001
            line["config5"] = {"error": str(e)}

    if rank == 0:
        # Roofline of the dominant kernel (the batched LM kernel).  Its state lives in shared memory, so HBM only sees
        # each sketch's inputs and outputs once; the roof that bounds it is the FP64 pipe (north_star: "FP64 pipe
        # utilisation for the factorisations").  achieved = algorithmic flops per launch (factorisations x (sum of
        # squared column counts + 4 nnz(L)), SURVEY 8d) / average launch time; peak = DFMA rate measured on this device
        # by fk_fp64_peak_tflops (MEASURED_PEAKS.json carries no FP64 figure).
        peak, peak_src = _peaks()
        alg_bytes = h2d + d2h
        avg_s = (total_ms / args.steps) * 1e-3 if world == 1 else (float(sum(step_ms)) / args.steps) * 1e-3
        flops = fact * (info["chol_flops"] + 4.0 * info["r_nnz"])
        try:
            fp64_peak = fk.fp64_peak_tflops(local_rank)
        except Exception:  # noqa: BLE001
            fp64_peak = None
        line["roofline"] = {"bound": "fp64", "achieved": flops / avg_s / 1e12, "peak": fp64_peak, "unit": "TFLOP/s",
                            "frac": (flops / avg_s / 1e12 / fp64_peak) if fp64_peak else None, "traffic": None,
                            "kernel": kernel_name,
                            "peak_source": "DFMA microbenchmark on this device (fk_fp64_peak_tflops; the driver's MEASURED_PEAKS.json has no FP64 figure)",
                            "algorithmic_flops_per_launch": flops, "factorizations_per_launch": fact,
                            "flops_per_factorization": info["chol_flops"] + 4.0 * info["r_nnz"],
                            "hbm": {"algorithmic_bytes_per_launch": alg_bytes, "achieved_gbs": alg_bytes / avg_s / 1e9, "peak_gbs": peak,
                                    "frac": alg_bytes / avg_s / 1e9 / peak, "peak_source": peak_src,
                                    "note": "inputs + outputs once per sketch; not the limiter"},
                            "profiles": "ncu --set full summaries of this kernel on this workload: profiles/r02b_lm_sketch_pair_kernel_truss_ncu_full_summary.csv (the kernel is unchanged since), its raw mode (the end-to-end calls): profiles/r02c_lm_sketch_pair_kernel_raw_mode_ncu_full_summary.csv; launch list of this command (--no-extras): profiles/r02c_launches_bench_truss.csv",
                            "note": "latency bound: 32 sketches are solved out of shared memory by one warp (or a leader / helper pair of warps) and "
                                    "only two such groups fit an SM for this topology; see DESIGN.md section 4 for the stall breakdown"}
        if not args.no_extras:
            try:
                line["large_system"] = large_system(fk, wl, peak, fp64_peak)
            except Exception as e:  # noqa: BLE001
                line["large_system"] = {"error": str(e)}
            try:
                line["assembly"] = assembly_bandwidth(fk, wl, torch, local_rank, peak)
            except Exception as e:  # noqa: BLE001
                line["assembly"] = {"error": str(e)}
            try:
                line["single_sketch"] = single_sketch_latency(fk, wl)
            except Exception as e:  # noqa: BLE001
                line["single_sketch"] = {"error": str(e)}
            try:
                line["hinged_triangles"] = hinged_triangles_side(fk, wl)
            except Exception as e:  # noqa: BLE001
                line["hinged_triangles"] = {"error": str(e)}
            try:
                line["single_pass"] = single_pass_side(fk, wl)
            except Exception as e:  # noqa: BLE001
                line["single_pass"] = {"error": str(e)}
            try:
                line["heterogeneous_batch"] = heterogeneous_side(fk, wl)
            except Exception as e:  # noqa: BLE001
                line["heterogeneous_batch"] = {"error": str(e)}
            try:
                line["lbfgs"] = lbfgs_side(fk, wl, local_rank)
            except Exception as e:  # noqa: BLE001
                line["lbfgs"] = {"error": str(e)}
            cores = os.cpu_count() or 1
            n_cpu, passes, secs = 65536, 0, 0.0
            while passes < 8 and secs * cores < 12.0:  # 10-30 s of CPU work: whole steps of the same workload
                _, s1, _, _ = cpu_reference_run(n_cpu, cores, first=passes * n_cpu)
                secs += s1
                passes += 1
            rate = n_cpu * passes / secs
            line["cpu_baseline"] = {"value": rate, "unit": UNIT, "cores": cores, "kind": "port",
                                    "sample": f"{passes} x {n_cpu} sketches of the same workload (whole steps), one sketch per task on {cores} threads, "
                                              f"{secs:.1f} s wall = {secs * cores:.0f} core-seconds"}
        else:
            line["cpu_baseline"] = {"value": None, "unit": UNIT, "cores": 0, "kind": "port", "sample": "skipped (--no-extras)"}
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, outputs)
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


def _allreduce(torch, dist, world, values, op="sum"):
    t = torch.tensor(values, dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX if op == "max" else dist.ReduceOp.SUM)
    return [float(x) for x in t]


def config4_sharded(fk, wl, torch, dist, rank, world, local_rank, barrier):
    """configs[3]: 1,000,000 mixed-primitive CAD sketches (circle_triangle_line topology) sharded by sketch over the
    ranks (strong scaling: the total is fixed), through the host-buffer call fk_batch_solve_device from pinned memory,
    and device resident for comparison.  Max over ranks of the timed region, every rank takes part."""
    import numpy as np
    total = 1_000_000
    lo, hi = total * rank // world, total * (rank + 1) // world
    n = hi - lo
    w = wl.cad_mix(n, first=lo)
    v, p, scale = w.prepare()
    topo = fk.Topology.from_arrays(w.n_vars, w.kind, w.idx, w.free_vars, w.rows)
    info = topo.info
    hv, hp = torch.from_numpy(v).pin_memory(), torch.from_numpy(p).pin_memory()
    hout = torch.empty((n, info["n_free"]), dtype=torch.float64).pin_memory()
    hrep = torch.empty((n, 40), dtype=torch.uint8).pin_memory()
    for _ in range(2):
        topo.batch_solve_into(local_rank, n, hv.data_ptr(), hp.data_ptr(), hout.data_ptr(), hrep.data_ptr())
    barrier()
    steps = 5
    t0 = time.perf_counter()
    for _ in range(steps):
        topo.batch_solve_into(local_rank, n, hv.data_ptr(), hp.data_ptr(), hout.data_ptr(), hrep.data_ptr())
    barrier()
    e2e_s = time.perf_counter() - t0
    rep = hrep.numpy().view(fk.REPORT_DTYPE).reshape(-1)
    # the same steps streamed two deep (fk_batch_solve_device_begin / _wait, alternating output buffers; every step's copies inside)
    hout2, hrep2 = torch.empty_like(hout).pin_memory(), torch.empty_like(hrep).pin_memory()
    outs = ((hout, hrep), (hout2, hrep2))
    begin = lambda i: topo.batch_solve_begin(local_rank, n, hv.data_ptr(), hp.data_ptr(), outs[i & 1][0].data_ptr(), outs[i & 1][1].data_ptr())
    for i in range(2):
        topo.batch_solve_wait(begin(i), local_rank)
    barrier()
    t0 = time.perf_counter()
    prev = begin(0)
    for i in range(1, steps):
        cur = begin(i)
        topo.batch_solve_wait(prev, local_rank)
        prev = cur
    topo.batch_solve_wait(prev, local_rank)
    barrier()
    stream_s = time.perf_counter() - t0
    streamed_same = float(np.array_equal(hout2.numpy(), hout.numpy()) and np.array_equal(hrep2.numpy(), hrep.numpy()))
    plan = topo.plan(n, device=local_rank)
    stream = torch.cuda.current_stream().cuda_stream
    plan.upload_ptr(n, hv.data_ptr(), hp.data_ptr(), stream)
    for _ in range(2):
        plan.run(stream)
    barrier()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(steps):
        plan.run(stream)
    b.record()
    barrier()
    dev_ms = a.elapsed_time(b)
    plan.close()
    e2e_s, dev_ms, stream_s = _allreduce(torch, dist, world, [e2e_s, dev_ms, stream_s], "max")
    streamed_same = _allreduce(torch, dist, world, [streamed_same])[0] == world
    conv, fact = _allreduce(torch, dist, world, [float(np.sum(rep["ssr"] < 1e-8)), float(rep["factorizations"].sum())])
    return {"workload": "configs[3]: 1,000,000 mixed-primitive CAD sketches (11 variables, 8 rows of 6 kinds), sharded by sketch",
            "n_gpus": world, "scaling": "strong", "sketches_total": total,
            "e2e_sketches_per_s": total * steps / stream_s, "e2e_one_call_at_a_time_sketches_per_s": total * steps / e2e_s,
            "streamed_results_equal_between_the_two_buffer_sets": bool(streamed_same),
            "device_resident_sketches_per_s": total * steps / (dev_ms * 1e-3),
            "h2d_bytes_per_sketch": 8 * (info["n_vars"] + info["n_expr"]), "d2h_bytes_per_sketch": 8 * info["n_free"] + 40,
            "fraction_converged": conv / total, "mean_factorizations": fact / total,
            "api": "fk_batch_solve_device_begin / _wait from pinned host buffers, steps streamed two deep (H2D + D2H of every step inside the timed "
                   "region); e2e_one_call_at_a_time: fk_batch_solve_device, each call returning before the next starts"}


def config5_sharded(fk, wl, torch, dist, rank, world, local_rank, barrier):
    """configs[4]: the stress families (under-/over-constrained, rank deficient, badly scaled, NaN; SURVEY App. D),
    8,192 sketches each, every family sharded by sketch over the ranks.  Reports throughput through the host-buffer
    call, the exit-reason histogram per family and the rate at which the accept/reject trace and the exit equal the
    oracle's on a sample of every rank's shard."""
    import numpy as np
    import oracle
    n_each, sample = 8192, 96
    fams = wl.stress_families(n_each)
    out, total_s, total_n = {}, 0.0, 0
    for name, w in fams:
        lo, hi = n_each * rank // world, n_each * (rank + 1) // world
        # (the NaN family must keep its points coincident: the solve's seeded perturbation would separate them)
        v, p, scale = w.prepare(perturb=(name != "nan_coincident_points"))
        v, p = np.ascontiguousarray(v[lo:hi]), np.ascontiguousarray(p[lo:hi])
        topo = fk.Topology.from_arrays(w.n_vars, w.kind, w.idx, w.free_vars, w.rows)
        topo.batch_solve(v, p)  # warm-up at the measured size (the entry point's pooled plans and streams are created once)
        barrier()
        t0 = time.perf_counter()
        for _ in range(3):
            x, rep = topo.batch_solve(v, p)
        barrier()
        secs = (time.perf_counter() - t0) / 3
        hist = np.bincount(rep["exit_reason"], minlength=5)[:5].astype(np.float64)
        m = min(sample, hi - lo)
        op, keep = oracle.make_problem(v[0], w.kind, w.idx, p[0], w.free_vars, w.rows)
        xo, ro, _ = oracle.lm_solve_batch_uniform(op, v[:m], p[:m], threads=min(8, os.cpu_count() or 1))
        same = float(np.sum((rep["trace_hash"][:m] == ro["trace_hash"]) & (rep["exit_reason"][:m] == ro["exit_reason"])))
        red = _allreduce(torch, dist, world, list(hist) + [same, float(m)])
        secs = _allreduce(torch, dist, world, [secs], "max")[0]
        out[name] = {"exit_histogram": {k: int(c) for k, c in zip(("converged", "small_step", "stalled", "max_outer", "lambda_overflow"), red[:5])},
                     "trace_and_exit_equal_to_oracle": red[5] / red[6], "oracle_sample": int(red[6]), "sketches_per_s": n_each / secs}
        total_s += secs
        total_n += n_each
    return {"workload": "configs[4]: %d stress families x %d sketches, sharded by sketch" % (len(fams), n_each), "n_gpus": world,
            "sketches_per_s_all_families": total_n / total_s, "families": out,
            "api": "fk_batch_solve (pageable host buffers, H2D + D2H inside)"}


def single_sketch_latency(fk, wl):
    """configs[0]: ONE circle_triangle_line-shaped sketch (11 variables, 8 rows) solved once.  A single tiny
    system is latency bound on a GPU (launch + two PCIe round trips); reported honestly beside the CPU."""
    import oracle
    w = wl.cad_mix(1)
    v, p, scale = w.prepare()
    topo = fk.Topology.from_arrays(w.n_vars, w.kind, w.idx, w.free_vars, w.rows)
    x0 = v[0][w.free_vars]
    for _ in range(5):
        topo.lm_solve(v[0], p[0], x0)
    reps = 200
    t0 = time.perf_counter()
    for _ in range(reps):
        xg, rg = topo.lm_solve(v[0], p[0], x0)
    gpu_us = (time.perf_counter() - t0) / reps * 1e6
    op, keep = oracle.make_problem(v[0], w.kind, w.idx, p[0], w.free_vars, w.rows)
    t0 = time.perf_counter()
    for _ in range(reps):
        xo, ro, _ = oracle.lm_solve(op, x0)
    cpu_us = (time.perf_counter() - t0) / reps * 1e6
    return {"workload": "configs[0]: one mixed-primitive sketch (circle_triangle_line topology), cached topology",
            "gpu_us_per_solve": gpu_us, "cpu_port_us_per_solve_incl_symbolic": cpu_us,
            "same_trace": bool(rg["trace_hash"] == ro["trace_hash"]),
            "note": "one sketch cannot amortise a kernel launch and two host<->device copies; batches can (see value / config4_lm)"}


def hinged_triangles_side(fk, wl):
    """The reference's own criterion shapes (fiksi/benches/fiksi_bench.rs:15-40: chains of 1 / 4 / 16 / 64 hinged
    triangles, Decomposer::None): one system at a time on the CPU restatement (one core, symbolic analysis inside every
    call as in the reference) and on the GPU (cached topology), and a batch of 16,384 perturbed copies on the GPU."""
    import numpy as np
    import oracle
    out = []
    for nt in (1, 4, 16, 64):
        w1 = wl.hinged_triangles(nt)
        v, p, scale = w1.prepare()
        topo = fk.Topology.from_arrays(w1.n_vars, w1.kind, w1.idx, w1.free_vars, w1.rows)
        x0 = v[0][w1.free_vars]
        for _ in range(3):
            topo.lm_solve(v[0], p[0], x0)
        reps = 50
        t0 = time.perf_counter()
        for _ in range(reps):
            xg, rg = topo.lm_solve(v[0], p[0], x0)
        gpu_us = (time.perf_counter() - t0) / reps * 1e6
        op, keep = oracle.make_problem(v[0], w1.kind, w1.idx, p[0], w1.free_vars, w1.rows)
        creps = max(3, min(200, 2000 // nt))
        t0 = time.perf_counter()
        for _ in range(creps):
            xo, ro, _ = oracle.lm_solve(op, x0)
        cpu_us = (time.perf_counter() - t0) / creps * 1e6
        nb = 16384
        wb = wl.hinged_triangles(nt, nb)
        vb, pb, _ = wb.prepare()
        topo.batch_solve(vb[:256], pb[:256])
        best = float("inf")
        for _ in range(3):
            t0 = time.perf_counter()
            xb, rb = topo.batch_solve(vb, pb)
            best = min(best, time.perf_counter() - t0)
        out.append({"triangles": nt, "variables": int(len(w1.free_vars)), "rows": int(len(w1.rows)), "path": int(topo.info["path"]),
                    "cpu_port_us_per_solve_1core": cpu_us, "gpu_us_per_solve_single_system": gpu_us,
                    "gpu_batch_sketches_per_s": nb / best, "gpu_batch_us_per_sketch": best / nb * 1e6,
                    "same_trace": bool(rg["trace_hash"] == ro["trace_hash"]),
                    "batch_fraction_converged": float(np.mean(rb["ssr"] < 1e-8))})
    return out


def single_pass_side(fk, wl):
    """SURVEY 8f-1: Decomposer::SinglePass on a batch of hinged-triangle chains (fiksi_bench.rs shape, 16
    triangles = 66 variables): one batched LM launch per strongly connected set, beside Decomposer::None on
    the same batch and the CPU restatement of the SinglePass loop."""
    import numpy as np
    import oracle
    n = 131072
    w = wl.hinged_triangles(16, n)
    v, p, scale = w.prepare()
    topo = fk.Topology.from_arrays(w.n_vars, w.kind, w.idx, w.free_vars, w.rows)
    topo.batch_solve_single_pass(v[:256], p[:256])
    sp_s = none_s = float("inf")
    for _ in range(3):  # host buffers are pageable here: best of three
        t0 = time.perf_counter()
        vg, rg = topo.batch_solve_single_pass(v, p)
        sp_s = min(sp_s, time.perf_counter() - t0)
    topo.batch_solve(v[:256], p[:256])
    for _ in range(3):
        t0 = time.perf_counter()
        x, rep = topo.batch_solve(v, p)
        none_s = min(none_s, time.perf_counter() - t0)
    ns = 512
    op, keep = oracle.make_problem(v[0], w.kind, w.idx, p[0], w.free_vars, w.rows)
    t0 = time.perf_counter()
    same = True
    for k in range(ns):
        opk, keepk = oracle.make_problem(v[k], w.kind, w.idx, p[k], w.free_vars, w.rows)
        vo, ro = oracle.single_pass_problem(opk, v[k])
        same = same and np.array_equal(ro["trace_hash"], rg[k]["trace_hash"])
    cpu_s = time.perf_counter() - t0
    return {"workload": "131,072 hinged chains of 16 triangles (66 variables, 48 rows), host buffers, device-resident between sets", "steps": int(rg.shape[1]),
            "gpu_single_pass_sketches_per_s": n / sp_s, "gpu_decomposer_none_sketches_per_s": n / none_s,
            "cpu_port_single_pass_sketches_per_s_1core": ns / cpu_s, "traces_equal_on_sample": bool(same),
            "fraction_converged_single_pass": float(np.mean(rg["ssr"] < 1e-8))}


def heterogeneous_side(fk, wl):
    """Many DIFFERENT small systems in one fk_lm_solve_batch call (the reference solves a drawing component by component,
    fiksi/src/assemble/mod.rs:81): trusses of 4..23 points with different fixed coordinates, `members` copies each.
    Topologies come from the library's cache on the timed calls; all small groups go through one launch of
    fk_hetero_lm_kernel (one warp per system).  Beside it the CPU restatement on one core, symbolic analysis per call as
    in the reference."""
    import numpy as np
    import oracle
    from fiksi_b200 import api
    out = []
    for n_topo, members in ((200, 5), (1000, 1)):
        rng = np.random.default_rng(0)
        probs, x0s, keep, oprobs = [], [], [], []
        for t in range(n_topo):
            n_points = 4 + t % 20
            w = wl.truss(members, n_points=n_points, seed=0xF1C50002 + 1000 * t)
            fixed = set(rng.choice(2 * n_points, size=t // 20 % 3, replace=False).tolist()) if t >= 20 else set()
            free = np.array([q for q in range(2 * n_points) if q not in fixed], np.uint32)
            v, p, s = w.prepare()
            for j in range(members):
                fp, k = fk.make_problem(v[j], w.kind, w.idx, p[j], free, w.rows)
                probs.append(fp); keep.append(k); x0s.append(v[j][free])
                oprobs.append((v[j], w.kind, w.idx, p[j], free, w.rows))
        api.topology_cache_clear()
        t0 = time.perf_counter()
        xs, reps = fk.lm_solve_batch(probs, x0s)
        cold = time.perf_counter() - t0
        warm = float("inf")
        for _ in range(3):
            t0 = time.perf_counter()
            xs, reps = fk.lm_solve_batch(probs, x0s)
            warm = min(warm, time.perf_counter() - t0)
        ns = min(len(probs), 300)
        same = 0
        t0 = time.perf_counter()
        for k in range(ns):
            op, okeep = oracle.make_problem(*oprobs[k])
            xo, ro, _ = oracle.lm_solve(op, x0s[k])
            same += int(ro["trace_hash"] == reps["trace_hash"][k] and ro["exit_reason"] == reps["exit_reason"][k])
        cpu_s = time.perf_counter() - t0
        out.append({"topologies": n_topo, "systems": len(probs), "gpu_systems_per_s_warm_cache": len(probs) / warm,
                    "gpu_first_call_s_incl_symbolic_analysis": cold, "cpu_port_systems_per_s_1core": ns / cpu_s,
                    "trace_and_exit_equal_to_oracle": same / ns, "oracle_sample": ns})
    return out


def lbfgs_side(fk, wl, device):
    """SURVEY 8f-3: the reference's second optimizer (fiksi/src/solve/lbfgs.rs) on the same truss batch,
    through the host-buffer C-ABI call (H2D + D2H inside), beside the CPU restatement."""
    import numpy as np
    import oracle
    n = 65536
    w = wl.truss(n)
    v, p, scale = w.prepare()
    topo = fk.Topology.from_arrays(w.n_vars, w.kind, w.idx, w.free_vars, w.rows)
    import torch
    # caller-owned pinned host buffers, as in the LM end-to-end figure (pageable numpy arrays, with freshly allocated outputs,
    # measured the host's page faults and staging copies: 4.4 M sketches/s)
    hv, hp = torch.from_numpy(v).pin_memory(), torch.from_numpy(p).pin_memory()
    hout = torch.empty((n, topo.info["n_free"]), dtype=torch.float64).pin_memory()
    hrep = torch.empty((n, 40), dtype=torch.uint8).pin_memory()
    call = lambda: topo.batch_solve_lbfgs_into(device, n, hv.data_ptr(), hp.data_ptr(), hout.data_ptr(), hrep.data_ptr())
    call()  # warm-up at the measured size: the pooled plans of the entry point grow once
    gpu_s = float("inf")
    for _ in range(3):
        t0 = time.perf_counter()
        call()
        gpu_s = min(gpu_s, time.perf_counter() - t0)
    x, rep = hout.numpy(), hrep.numpy().view(fk.REPORT_DTYPE).reshape(n)
    plan = topo.plan(n, device=device)
    stream = torch.cuda.current_stream().cuda_stream
    plan.upload(v, p, stream)
    plan.run_lbfgs(stream)
    torch.cuda.synchronize()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record()
    for _ in range(3):
        plan.run_lbfgs(stream)
    ev1.record()
    torch.cuda.synchronize()
    kernel_ms = ev0.elapsed_time(ev1) / 3
    plan.close()
    cores = os.cpu_count() or 1
    ns = 4096
    op, keep = oracle.make_problem(v[0], w.kind, w.idx, p[0], w.free_vars, w.rows)
    xo, ro, cpu_s = oracle.lbfgs_solve_batch_uniform(op, v[:ns], p[:ns], threads=cores)
    same = (rep["trace_hash"][:ns] == ro["trace_hash"]) & (rep["exit_reason"][:ns] == ro["exit_reason"])
    return {"workload": "configs[1] truss batch, Optimizer::LBfgs", "gpu_e2e_sketches_per_s": n / gpu_s,
            "e2e_api": "fk_batch_solve_lbfgs from pinned host buffers (H2D + D2H inside)",
            "gpu_device_resident_sketches_per_s": n / (kernel_ms * 1e-3), "kernel_ms": kernel_ms,
            "mean_line_searches": float(rep["outer_iters"].mean()), "mean_evaluations": float(rep["factorizations"].mean()),
            "fraction_residual_exit": float(np.mean(rep["exit_reason"] == 2)),
            "cpu_port_sketches_per_s": ns / cpu_s, "cpu_cores": cores, "cpu_sample": ns,
            "trace_equal_frac": float(same.mean()), "max_abs_coord_diff": float(np.max(np.abs(x[:ns] - xo)))}


def assembly_bandwidth(fk, wl, torch, device, peak):
    """K1 (residual + Jacobian scatter into the precomputed CSC pattern) on 1,000,000 mixed-primitive
    sketches (config 4 topology): 1,128 algorithmic bytes per sketch -> 1.13 GB per launch, > L2."""
    n = 1_000_000
    w = wl.cad_mix(n)
    v, p, scale = w.prepare()
    topo = fk.Topology.from_arrays(w.n_vars, w.kind, w.idx, w.free_vars, w.rows)
    plan = topo.plan(n, device=device)
    stream = torch.cuda.current_stream().cuda_stream
    plan.upload(v, p, stream)
    torch.cuda.synchronize()
    for _ in range(3):
        plan.eval(0, stream)
    times = []
    for _ in range(10):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        plan.eval(0, stream)
        b.record()
        torch.cuda.synchronize()
        times.append(a.elapsed_time(b))
    ms = sum(times) / len(times)
    alg = topo.info["eval_bytes"] * n
    i = topo.info
    dram = 8 * n * (i["n_vars"] + i["n_expr"] + i["n_rows"] + i["jac_nnz"])  # every input and output byte once
    out = {"kernel": "fk_batch_eval_tiled_kernel<S,true,256,prefetch> (S = 64 for this topology: the inputs of a CTA's next tile arrive by cp.async "
                     "while the current one is evaluated)", "workload": "config 4 topology, 1,000,000 sketches",
           "bound": "hbm", "algorithmic_bytes": alg, "ms": ms, "achieved_algorithmic_gbs": alg / (ms * 1e-3) / 1e9, "peak": peak, "unit": "GB/s"}
    out["frac_algorithmic"] = out["achieved_algorithmic_gbs"] / peak
    # SURVEY 8d's algorithmic bytes count every per-row gather (17 + 4k + 20a B/row); the tile-staged kernel
    # reads each variable once per sketch, so the traffic HBM actually sees is smaller (ncu: 152 MB read +
    # 366 MB written per launch, profiles/r01_k1_tiled_S64_ncu_full_summary.csv)
    out["min_dram_bytes"] = dram
    out["achieved"] = dram / (ms * 1e-3) / 1e9   # REAL bytes (every input and output byte once): the HBM fraction to quote
    out["frac"] = out["achieved"] / peak
    out["traffic"] = None  # ncu --set full captures of this kernel: profiles/r02b_k1_prefetch_ncu_full_summary.csv, profiles/r01_k1_tiled_S64_ncu_full_summary.csv (152 MB read + 366 MB written)
    plan.close()
    # LM solve of the same 1,000,000 mixed-primitive sketches (config 4), device-resident
    try:
        plan = topo.plan(n, device=device)
        plan.upload(v, p, stream)
        plan.run(stream)
        torch.cuda.synchronize()
        ts = []
        for _ in range(3):
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            plan.run(stream)
            b.record()
            torch.cuda.synchronize()
            ts.append(a.elapsed_time(b))
        import numpy as np
        rep = np.zeros(n, dtype=fk.REPORT_DTYPE)
        plan.download(None, rep, stream)
        torch.cuda.synchronize()
        lm_ms = sum(ts) / len(ts)
        out["config4_lm"] = {"workload": "configs[3]: 1,000,000 mixed-primitive CAD sketches (11 variables, 8 rows of 6 kinds), 1 GPU",
                             "ms": lm_ms, "sketches_per_s": n / (lm_ms * 1e-3), "tile_lanes": i["tile"],
                             "fraction_converged": float(np.mean(rep["ssr"] < 1e-8)),
                             "mean_factorizations": float(rep["factorizations"].mean())}
        plan.close()
    except Exception as e:  # noqa: BLE001
        out["config4_lm"] = {"error": str(e)}
    return out


def large_system(fk, wl, hbm_peak, fp64_peak):
    import numpy as np
    """Config 3: one 400x250 lattice (200,000 variables, 298,701 distance rows) through the global
    sparse path: time per LM solve, phase split, FP64 rate of the supernodal multifrontal LDL^T
    (K5), and the K1 assembly rate on its 31.4 MB (L2-resident) table."""
    w = wl.lattice(400, 250)
    v, p, scale = w.prepare()
    t0 = time.perf_counter()
    topo = fk.Topology.from_arrays(w.n_vars, w.kind, w.idx, w.free_vars, w.rows)
    symbolic_s = time.perf_counter() - t0
    x0 = v[0][w.free_vars]
    t0 = time.perf_counter()
    topo.lm_solve(v[0], p[0], x0)  # first solve: supernodal analysis, uploads, allocations, graph capture
    first_s = time.perf_counter() - t0
    t0 = time.perf_counter()
    x, rep = topo.lm_solve(v[0], p[0], x0)
    solve_s = time.perf_counter() - t0
    tm = topo.last_timing()
    r, j, eval_ms = topo.eval_large(v[0], p[0], x0, repeats=50, want_j=False)
    info = topo.info
    flops = float(info["chol_flops"]) * tm["factors"]
    out = {"workload": "configs[2]: 400x250 lattice, 200,000 variables, 298,701 PPD rows, nnz(L) = %d" % info["r_nnz"],
           "symbolic_s_host_once_per_topology": symbolic_s, "first_lm_solve_s_incl_device_setup": first_s,
           "host_threads_symbolic": min(os.cpu_count() or 1, 32), "lm_solve_s": solve_s, "exit_reason": rep["exit_reason"],
           "factorizations": rep["factorizations"], "final_ssr": rep["ssr"],
           "phase_ms": {k: tm[k] for k in ("eval_ms", "assemble_ms", "factor_ms", "tri_ms")},
           "factor_tflops": flops / (tm["factor_ms"] * 1e-3) / 1e12,
           "factor_frac_of_fp64_peak": (flops / (tm["factor_ms"] * 1e-3) / 1e12 / fp64_peak) if fp64_peak else None,
           "eval_ms": eval_ms, "eval_algorithmic_bytes": info["eval_bytes"],
           "eval_gbs": info["eval_bytes"] / (eval_ms * 1e-3) / 1e9, "eval_frac_of_hbm_peak": info["eval_bytes"] / (eval_ms * 1e-3) / 1e9 / hbm_peak,
           "note": "31.4 MB per evaluation is L2-resident; the CPU reference needs O(m n) scratch stores per factorisation "
                   "(qr.rs:286-287) and is timed on the smaller lattices of `sweep` only (10,000 points take 67 s on one core)"}
    # size sweep with the CPU reference algorithm (oracle port, 1 core: the reference is single-threaded) beside the GPU
    import oracle
    sweep = []
    for nx, ny in ((32, 32), (64, 50)):
        ws = wl.lattice(nx, ny)
        vs, ps, _ = ws.prepare()
        ts = fk.Topology.from_arrays(ws.n_vars, ws.kind, ws.idx, ws.free_vars, ws.rows)
        xs0 = vs[0][ws.free_vars]
        ts.lm_solve(vs[0], ps[0], xs0)
        t0 = time.perf_counter()
        xg, rg = ts.lm_solve(vs[0], ps[0], xs0)
        gpu_s = time.perf_counter() - t0
        op, keep = oracle.make_problem(vs[0], ws.kind, ws.idx, ps[0], ws.free_vars, ws.rows)
        t0 = time.perf_counter()
        xo, ro, _ = oracle.lm_solve(op, xs0)
        cpu_s = time.perf_counter() - t0
        sweep.append({"lattice": f"{nx}x{ny}", "variables": int(len(ws.free_vars)), "gpu_lm_solve_s": gpu_s, "cpu_port_lm_solve_s_1core": cpu_s,
                      "same_trace": bool(rg["trace_hash"] == ro["trace_hash"]),
                      "max_rel_coord_diff": float(np.max(np.abs(xg - xo)) / np.max(np.abs(xo)))})
    out["sweep"] = sweep
    return out


if __name__ == "__main__":
    main()
