"""Thin Python face of the C ABI (include/fiksi_b200.h): topology, symbolic probes, LM solves.

All numerics happen inside libfiksi_b200.so (host symbolic pipeline in C++, kernels in CUDA for
sm_100a).  Nothing here computes residuals, Jacobians, orderings or factorizations.
"""
from __future__ import annotations

import ctypes as C

import numpy as np

from ._lib import (FkPrepareOpts, FkProblem, FkReport, FkTopologyInfo, REPORT_DTYPE, check, lib, make_problem, ptr)


class Topology:
    """fk_topology: symbolic analysis computed once per topology."""

    def __init__(self, problem: FkProblem, keepalive=None):
        self._h = C.c_void_p()
        check(lib().fk_topology_create(C.byref(problem), C.byref(self._h)))
        self._keep = keepalive
        info = FkTopologyInfo()
        check(lib().fk_topology_info_get(self._h, C.byref(info)))
        self.info = {n: getattr(info, n) for n, _ in FkTopologyInfo._fields_}

    @classmethod
    def from_arrays(cls, n_vars, kind, idx, free_vars, rows):
        p, keep = make_problem(np.zeros(n_vars), kind, idx, np.zeros(len(kind)), free_vars, rows)
        return cls(p, keep)

    def symbolic(self):
        i = self.info
        n = i["n_free"]
        out = {
            "aug_colptr": np.zeros(n + 1, np.uint32), "aug_rowidx": np.zeros(max(i["aug_nnz"], 1), np.uint32),
            "perm": np.zeros(max(n, 1), np.int32), "etree_parent": np.zeros(max(n, 1), np.int32),
            "r_colptr": np.zeros(n + 1, np.uint32), "r_rowidx": np.zeros(max(i["r_nnz"], 1), np.uint32),
        }
        check(lib().fk_topology_symbolic(self._h, ptr(out["aug_colptr"], C.c_uint32), ptr(out["aug_rowidx"], C.c_uint32),
                                         ptr(out["perm"], C.c_int32), ptr(out["etree_parent"], C.c_int32),
                                         ptr(out["r_colptr"], C.c_uint32), ptr(out["r_rowidx"], C.c_uint32)))
        out["aug_rowidx"] = out["aug_rowidx"][:i["aug_nnz"]]
        out["perm"] = out["perm"][:n]
        out["etree_parent"] = out["etree_parent"][:n]
        out["r_rowidx"] = out["r_rowidx"][:i["r_nnz"]]
        return out

    def supernodal(self):
        """fk_topology_supernodal: host-side analysis of the large-system path (no device needed)."""
        class Info(C.Structure):
            _fields_ = [(n, C.c_uint32) for n in ("n_supernodes", "n_small_subtrees", "n_big", "n_levels", "max_front",
                                                  "n_tasks", "n_launches", "pad0")] + \
                       [(n, C.c_uint64) for n in ("rows_total", "rel_total", "panel_doubles", "update_doubles")]
        info = Info()
        f = lib().fk_topology_supernodal
        null = [None] * 9
        check(f(self._h, C.byref(info), *null))
        S = info.n_supernodes
        out = {"sn_first": np.zeros(S + 1, np.uint32), "front": np.zeros(max(S, 1), np.uint32), "sn_parent": np.zeros(max(S, 1), np.int32),
               "rows": np.zeros(max(info.rows_total, 1), np.uint32), "rel": np.zeros(max(info.rel_total, 1), np.uint32),
               "big": np.zeros(max(S, 1), np.uint8), "level": np.zeros(max(S, 1), np.uint32),
               "tasks": np.zeros(max(4 * info.n_tasks, 1), np.uint32), "launches": np.zeros(max(3 * info.n_launches, 1), np.uint32)}
        check(f(self._h, C.byref(info), ptr(out["sn_first"], C.c_uint32), ptr(out["front"], C.c_uint32), ptr(out["sn_parent"], C.c_int32),
                ptr(out["rows"], C.c_uint32), ptr(out["rel"], C.c_uint32), ptr(out["big"], C.c_uint8), ptr(out["level"], C.c_uint32),
                ptr(out["tasks"], C.c_uint32), ptr(out["launches"], C.c_uint32)))
        out["front"] = out["front"][:S]; out["sn_parent"] = out["sn_parent"][:S]; out["big"] = out["big"][:S]; out["level"] = out["level"][:S]
        out["rows"] = out["rows"][:info.rows_total]; out["rel"] = out["rel"][:info.rel_total]
        out["tasks"] = out["tasks"][:4 * info.n_tasks].reshape(-1, 4); out["launches"] = out["launches"][:3 * info.n_launches].reshape(-1, 3)
        out["info"] = {n: getattr(info, n) for n, _ in Info._fields_}
        return out

    def batch_solve_single_pass(self, vars_, param, n_gpus=1):
        """fk_batch_solve_single_pass: Decomposer::SinglePass on a uniform batch; returns (vars after the
        pass [n][n_vars], reports [n][steps])."""
        v = np.array(vars_, dtype=np.float64, order="C")
        param = np.ascontiguousarray(param, dtype=np.float64)
        n = v.shape[0]
        steps = C.c_uint32(0)
        check(lib().fk_batch_solve_single_pass(self._h, 0, None, None, None, C.byref(steps), n_gpus))
        reports = np.zeros((n, max(steps.value, 1)), dtype=REPORT_DTYPE)
        check(lib().fk_batch_solve_single_pass(self._h, n, ptr(v, C.c_double), ptr(param, C.c_double),
                                               reports.ctypes.data_as(C.POINTER(FkReport)), C.byref(steps), n_gpus))
        return v, reports[:, :steps.value]

    def batch_solve_lbfgs(self, vars_, param, device=0):
        """fk_batch_solve_lbfgs: Optimizer::LBfgs (fiksi/src/solve/lbfgs.rs) on a uniform batch."""
        vars_ = np.ascontiguousarray(vars_, dtype=np.float64)
        param = np.ascontiguousarray(param, dtype=np.float64)
        n = vars_.shape[0]
        out = np.zeros((n, self.info["n_free"]), dtype=np.float64)
        reports = np.zeros(n, dtype=REPORT_DTYPE)
        check(lib().fk_batch_solve_lbfgs(self._h, device, n, ptr(vars_, C.c_double), ptr(param, C.c_double), ptr(out, C.c_double),
                                         reports.ctypes.data_as(C.POINTER(FkReport))))
        return out, reports

    def batch_analyze(self, vars_, param, device=0):
        """fk_batch_analyze: System::analyze's per-expression "independent" flags for n sketches
        (UNSCALED variables / parameters; all variables free, all expressions)."""
        vars_ = np.ascontiguousarray(vars_, dtype=np.float64)
        param = np.ascontiguousarray(param, dtype=np.float64)
        n = vars_.shape[0]
        out = np.zeros((n, max(self.info["n_expr"], 1)), dtype=np.uint8)
        check(lib().fk_batch_analyze(self._h, device, n, ptr(vars_, C.c_double), ptr(param, C.c_double), ptr(out, C.c_uint8)))
        return out[:, :self.info["n_expr"]].astype(bool)

    def batch_solve(self, vars_, param, n_gpus=1):
        """fk_batch_solve on host buffers: vars[n][n_vars], param[n][n_expr] -> (free[n][n_free], reports)."""
        vars_ = np.ascontiguousarray(vars_, dtype=np.float64)
        param = np.ascontiguousarray(param, dtype=np.float64)
        n = vars_.shape[0]
        out = np.zeros((n, self.info["n_free"]), dtype=np.float64)
        reports = np.zeros(n, dtype=REPORT_DTYPE)
        check(lib().fk_batch_solve(self._h, n, ptr(vars_, C.c_double), ptr(param, C.c_double), ptr(out, C.c_double),
                                   reports.ctypes.data_as(C.POINTER(FkReport)), n_gpus))
        return out, reports

    def batch_system_solve(self, raw_vars, raw_param, perturb=True, perturb_vars=None, shared_param=False, device=0, seed=42):
        """fk_batch_system_solve: System::solve for n single-component sketches, scale / perturbation / write-back on
        the device.  raw_param is [n][n_expr], or one row with shared_param.  Returns (unscaled free values, scales, reports)."""
        raw_vars = np.ascontiguousarray(raw_vars, dtype=np.float64)
        raw_param = np.ascontiguousarray(raw_param, dtype=np.float64)
        n = raw_vars.shape[0]
        out = np.zeros((n, self.info["n_free"]), dtype=np.float64)
        scales = np.zeros(n, dtype=np.float64)
        reports = np.zeros(n, dtype=REPORT_DTYPE)
        o = FkPrepareOpts()
        o.flags = (1 if shared_param else 0) | (2 if perturb else 0)
        o.seed = seed
        keep = None
        if perturb_vars is not None:
            keep = np.ascontiguousarray(perturb_vars, dtype=np.uint32)
            o.n_perturb, o.perturb_vars = len(keep), ptr(keep, C.c_uint32)
        check(lib().fk_batch_system_solve(self._h, device, n, ptr(raw_vars, C.c_double), ptr(raw_param, C.c_double), C.byref(o),
                                          ptr(out, C.c_double), ptr(scales, C.c_double), reports.ctypes.data_as(C.POINTER(FkReport))))
        return out, scales, reports

    def batch_system_solve_into(self, device, n, raw_vars_ptr, raw_param_ptr, out_ptr, rep_ptr, shared_param=False, perturb=True):
        """fk_batch_system_solve on caller-owned (ideally pinned) host buffers given as addresses."""
        o = FkPrepareOpts()
        o.flags = (1 if shared_param else 0) | (2 if perturb else 0)
        o.seed = 42
        check(lib().fk_batch_system_solve(self._h, device, n, C.c_void_p(raw_vars_ptr), C.c_void_p(raw_param_ptr), C.byref(o),
                                          C.c_void_p(out_ptr), None, C.c_void_p(rep_ptr)))

    def batch_system_solve_begin(self, device, n, raw_vars_ptr, raw_param_ptr, out_ptr, rep_ptr, shared_param=False, perturb=True):
        """fk_batch_system_solve_begin on caller-owned pinned host buffers: returns a token once the batch is enqueued;
        batch_system_solve_wait(token) returns when its results are in the buffers.  Up to two batches in flight."""
        o = FkPrepareOpts()
        o.flags = (1 if shared_param else 0) | (2 if perturb else 0)
        o.seed = 42
        token = C.c_uint64(0)
        check(lib().fk_batch_system_solve_begin(self._h, device, n, C.c_void_p(raw_vars_ptr), C.c_void_p(raw_param_ptr), C.byref(o),
                                                C.c_void_p(out_ptr), None, C.c_void_p(rep_ptr), C.byref(token)))
        return token.value

    def batch_system_solve_wait(self, token, device=0):
        check(lib().fk_batch_system_solve_wait(self._h, device, C.c_uint64(token)))

    def batch_solve_into(self, device, n, vars_ptr, param_ptr, out_ptr, rep_ptr):
        """fk_batch_solve_device on caller-owned (ideally pinned) host buffers given as addresses."""
        check(lib().fk_batch_solve_device(self._h, device, n, C.c_void_p(vars_ptr), C.c_void_p(param_ptr),
                                          C.c_void_p(out_ptr), C.c_void_p(rep_ptr)))

    def batch_solve_begin(self, device, n, vars_ptr, param_ptr, out_ptr, rep_ptr):
        """fk_batch_solve_device_begin on caller-owned pinned host buffers: token; batch_solve_wait(token) completes it."""
        token = C.c_uint64(0)
        check(lib().fk_batch_solve_device_begin(self._h, device, n, C.c_void_p(vars_ptr), C.c_void_p(param_ptr),
                                                C.c_void_p(out_ptr), C.c_void_p(rep_ptr), C.byref(token)))
        return token.value

    def batch_solve_wait(self, token, device=0):
        check(lib().fk_batch_solve_device_wait(self._h, device, C.c_uint64(token)))

    def batch_solve_lbfgs_into(self, device, n, vars_ptr, param_ptr, out_ptr, rep_ptr):
        """fk_batch_solve_lbfgs on caller-owned (ideally pinned) host buffers given as addresses."""
        check(lib().fk_batch_solve_lbfgs(self._h, device, n, C.cast(C.c_void_p(vars_ptr), C.POINTER(C.c_double)),
                                         C.cast(C.c_void_p(param_ptr), C.POINTER(C.c_double)), C.cast(C.c_void_p(out_ptr), C.POINTER(C.c_double)),
                                         C.cast(C.c_void_p(rep_ptr), C.POINTER(FkReport))))

    def lm_solve(self, vars_, param, free_values):
        """fk_topology_lm_solve: one system, symbolic analysis reused."""
        vars_ = np.ascontiguousarray(vars_, dtype=np.float64)
        param = np.ascontiguousarray(param, dtype=np.float64)
        x = np.array(free_values, dtype=np.float64)
        rep = FkReport()
        check(lib().fk_topology_lm_solve(self._h, ptr(vars_, C.c_double), ptr(param, C.c_double), ptr(x, C.c_double), C.byref(rep)))
        return x, report_dict(rep)

    def eval_large(self, vars_, param, free_values, repeats=0, want_j=True):
        vars_ = np.ascontiguousarray(vars_, dtype=np.float64)
        param = np.ascontiguousarray(param, dtype=np.float64)
        x = np.ascontiguousarray(free_values, dtype=np.float64)
        r = np.zeros(max(self.info["n_rows"], 1))
        j = np.zeros(max(self.info["jac_nnz"], 1)) if want_j else None
        ms = C.c_float(0.0)
        check(lib().fk_topology_eval(self._h, ptr(vars_, C.c_double), ptr(param, C.c_double), ptr(x, C.c_double),
                                     ptr(r, C.c_double), ptr(j, C.c_double) if want_j else None, repeats, C.byref(ms)))
        return r[:self.info["n_rows"]], (j[:self.info["jac_nnz"]] if want_j else None), ms.value

    def last_timing(self):
        out = (C.c_float * 8)()
        check(lib().fk_topology_last_timing(self._h, out))
        return {"eval_ms": out[0], "assemble_ms": out[1], "factor_ms": out[2], "tri_ms": out[3],
                "evals": int(out[4]), "factors": int(out[5]), "fwd_ms": out[6], "bwd_ms": out[7]}

    def sketch_kernel_info(self):
        """fk_topology_sketch_kernel_info: does the topology have a sketch-per-thread LM kernel, its shared-memory
        doubles per sketch and the 16-bit words of its parameter block."""
        ok, ent, words = C.c_int(0), C.c_uint32(0), C.c_uint32(0)
        check(lib().fk_topology_sketch_kernel_info(self._h, C.byref(ok), C.byref(ent), C.byref(words)))
        return {"available": bool(ok.value), "state_doubles": ent.value, "table_words": words.value}

    def batch_kernel(self, n_sketches):
        """fk_topology_batch_kernel: the kernel a batched LM solve of this size launches: 'tile', 'sketch', 'sketch_pair', or
        'sparse_batch' (global sparse path: one CTA per sketch over the supernodal tree)."""
        k = lib().fk_topology_batch_kernel(self._h, int(n_sketches))
        if k < 0:
            check(k)
        return {0: "tile", 1: "sketch", 2: "sketch_pair", 3: "sparse_batch"}[k]

    def analyze_kernel(self, n_sketches):
        """fk_topology_analyze_kernel: the kernel batch_analyze of this size launches on the current device: 'warp' (matrix
        in shared memory), 'cta' (one CTA per sketch, matrix in global memory) or 'group' (a group of CTAs per sketch)."""
        k = lib().fk_topology_analyze_kernel(self._h, int(n_sketches))
        if k < 0:
            check(k)
        return {0: "warp", 1: "cta", 2: "group"}[k]

    def lbfgs_kernel(self, n_sketches):
        """fk_topology_lbfgs_kernel: the L-BFGS kernel the batch calls launch: 0 the tile kernel (state in shared memory),
        1 the CTA kernel (one CTA per sketch, state in global memory; any size)."""
        k = lib().fk_topology_lbfgs_kernel(self._h, int(n_sketches))
        if k < 0:
            check(k)
        return k

    def plan(self, capacity, device=0):
        return BatchPlan(self, capacity, device)

    def close(self):
        if self._h:
            lib().fk_topology_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class BatchPlan:
    """fk_batch_plan: device-resident buffers for n sketches of one topology on one device."""

    def __init__(self, topo: Topology, capacity: int, device: int = 0):
        self.topo = topo
        self._h = C.c_void_p()
        check(lib().fk_batch_plan_create(topo._h, capacity, device, C.byref(self._h)))
        self.capacity = capacity
        self.n = 0

    def upload(self, vars_, param, stream=0):
        n = vars_.shape[0]
        check(lib().fk_batch_plan_upload(self._h, n, C.c_void_p(vars_.ctypes.data), C.c_void_p(param.ctypes.data), C.c_void_p(stream)))
        self.n = n

    def upload_ptr(self, n, vars_ptr, param_ptr, stream=0):
        check(lib().fk_batch_plan_upload(self._h, n, C.c_void_p(vars_ptr), C.c_void_p(param_ptr), C.c_void_p(stream)))
        self.n = n

    def run(self, stream=0):
        check(lib().fk_batch_plan_run(self._h, C.c_void_p(stream)))

    def run_lbfgs(self, stream=0):
        check(lib().fk_batch_plan_run_lbfgs(self._h, C.c_void_p(stream)))

    def run_lbfgs_global(self, stream=0):
        """fk_batch_plan_run_lbfgs_global: L-BFGS with the CTA kernel on any plan."""
        check(lib().fk_batch_plan_run_lbfgs_global(self._h, C.c_void_p(stream)))

    def download(self, free_out, reports, stream=0):
        check(lib().fk_batch_plan_download(self._h, C.c_void_p(free_out.ctypes.data if free_out is not None else 0),
                                           C.c_void_p(reports.ctypes.data if reports is not None else 0), C.c_void_p(stream)))

    def download_ptr(self, free_ptr, rep_ptr, stream=0):
        check(lib().fk_batch_plan_download(self._h, C.c_void_p(free_ptr), C.c_void_p(rep_ptr), C.c_void_p(stream)))

    def eval(self, mode=0, stream=0):
        check(lib().fk_batch_plan_eval(self._h, mode, C.c_void_p(stream)))

    def eval_download(self, out_r, out_j, stream=0):
        check(lib().fk_batch_plan_eval_download(self._h, C.c_void_p(out_r.ctypes.data if out_r is not None else 0),
                                                C.c_void_p(out_j.ctypes.data if out_j is not None else 0), C.c_void_p(stream)))

    @property
    def launches(self):
        return int(lib().fk_batch_plan_launches(self._h))

    def close(self):
        if self._h:
            lib().fk_batch_plan_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def fp64_peak_tflops(device=0) -> float:
    out = C.c_double(0.0)
    check(lib().fk_fp64_peak_tflops(device, C.byref(out)))
    return out.value


class lm_kernel:
    """Context manager around fk_set_lm_kernel: 'auto' | 'tile' | 'sketch' | 'sketch_solo' | 'sketch_pair' (tests, A/B)."""
    _CODES = {"auto": -1, "tile": 0, "sketch": 1, "sketch_solo": 2, "sketch_pair": 3}

    def __init__(self, choice):
        self.code = self._CODES[choice]

    def __enter__(self):
        self.prev = lib().fk_get_lm_kernel()
        lib().fk_set_lm_kernel(self.code)
        return self

    def __exit__(self, *exc):
        lib().fk_set_lm_kernel(self.prev)
        return False


def topology_cache_stats():
    """fk_topology_cache_stats: (hits, misses, entries) of the process-wide topology cache of fk_lm_solve*."""
    h, m, e = C.c_uint64(0), C.c_uint64(0), C.c_uint32(0)
    lib().fk_topology_cache_stats(C.byref(h), C.byref(m), C.byref(e))
    return h.value, m.value, e.value


def topology_cache_clear():
    lib().fk_topology_cache_clear()


def topology_cache_configure(capacity):
    lib().fk_topology_cache_configure(int(capacity))


def device_count() -> int:
    return int(lib().fk_device_count())


def lm_solve(problem: FkProblem, free_values):
    """== levenberg_marquardt(problem, variables) (fiksi/src/solve/lm.rs:21) through fk_lm_solve."""
    x = np.array(free_values, dtype=np.float64)
    rep = FkReport()
    check(lib().fk_lm_solve(C.byref(problem), ptr(x, C.c_double), C.byref(rep)))
    return x, report_dict(rep)


def _solve_batch(fn, problems, free_values_list, n_gpus):
    n = len(problems)
    arr = (C.POINTER(FkProblem) * max(n, 1))(*[C.pointer(p) for p in problems])
    xs = [np.array(v, dtype=np.float64) for v in free_values_list]
    fv = (C.POINTER(C.c_double) * max(n, 1))(*[ptr(x, C.c_double) for x in xs])
    reports = np.zeros(n, dtype=REPORT_DTYPE)
    check(fn(n, arr, fv, reports.ctypes.data_as(C.POINTER(FkReport)), n_gpus))
    return xs, reports


def lm_solve_batch(problems, free_values_list, n_gpus=1):
    return _solve_batch(lib().fk_lm_solve_batch, problems, free_values_list, n_gpus)


def lbfgs_solve(problem: FkProblem, free_values):
    """== lbfgs(problem, variables) (fiksi/src/solve/lbfgs.rs:20) through fk_lbfgs_solve (any size)."""
    x = np.array(free_values, dtype=np.float64)
    rep = FkReport()
    check(lib().fk_lbfgs_solve(C.byref(problem), ptr(x, C.c_double), C.byref(rep)))
    return x, report_dict(rep)


def lbfgs_solve_batch(problems, free_values_list, n_gpus=1):
    """fk_lbfgs_solve_batch: problems of any structure and size, grouped by topology."""
    return _solve_batch(lib().fk_lbfgs_solve_batch, problems, free_values_list, n_gpus)


def report_dict(rep):
    return {"exit_reason": rep.exit_reason, "outer_iters": rep.outer_iters, "factorizations": rep.factorizations,
            "accepted": rep.accepted, "ssr": rep.ssr, "lambda": rep.lambda_, "trace_hash": rep.trace_hash}
