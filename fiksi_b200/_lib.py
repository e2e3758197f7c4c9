"""ctypes loader for libfiksi_b200.so, the C-ABI product library (include/fiksi_b200.h).

The library is built in-tree by ``__graft_entry__.build()`` (``make -C fiksi_b200/csrc``).  There
is no fallback: if the shared object is missing, loading fails loudly.
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libfiksi_b200.so")


class FkProblem(C.Structure):
    _fields_ = [
        ("n_vars", C.c_uint32), ("vars", C.POINTER(C.c_double)),
        ("n_expr", C.c_uint32), ("kind", C.POINTER(C.c_uint8)),
        ("idx", C.POINTER(C.c_uint32)), ("param", C.POINTER(C.c_double)),
        ("n_free", C.c_uint32), ("free_vars", C.POINTER(C.c_uint32)),
        ("n_rows", C.c_uint32), ("rows", C.POINTER(C.c_uint32)),
    ]


class FkReport(C.Structure):
    _fields_ = [
        ("exit_reason", C.c_uint32), ("outer_iters", C.c_uint32),
        ("factorizations", C.c_uint32), ("accepted", C.c_uint32),
        ("ssr", C.c_double), ("lambda_", C.c_double), ("trace_hash", C.c_uint64),
    ]


class FkPrepareOpts(C.Structure):
    _fields_ = [("flags", C.c_uint32), ("n_perturb", C.c_uint32), ("perturb_vars", C.POINTER(C.c_uint32)),
                ("seed", C.c_uint32), ("pad", C.c_uint32)]


class FkSolvingOptions(C.Structure):
    _fields_ = [("optimizer", C.c_uint32), ("decomposer", C.c_uint32), ("perturb", C.c_uint32), ("pad", C.c_uint32)]


class FkTopologyInfo(C.Structure):
    _fields_ = [(n, C.c_uint32) for n in (
        "n_vars", "n_expr", "n_free", "n_rows", "jac_nnz", "aug_nnz", "r_nnz", "etree_height",
        "path", "tile", "smem_bytes", "eval_bytes")] + [("chol_flops", C.c_uint64)]


REPORT_DTYPE = np.dtype([
    ("exit_reason", "<u4"), ("outer_iters", "<u4"), ("factorizations", "<u4"), ("accepted", "<u4"),
    ("ssr", "<f8"), ("lambda", "<f8"), ("trace_hash", "<u8"),
])
assert REPORT_DTYPE.itemsize == C.sizeof(FkReport) == 40

EXPORTS = [
    "fk_version", "fk_last_error", "fk_device_count", "fk_topology_create", "fk_topology_destroy",
    "fk_topology_info_get", "fk_topology_symbolic", "fk_symbolic", "fk_lm_solve", "fk_lm_solve_batch",
    "fk_batch_solve", "fk_batch_plan_create", "fk_batch_plan_destroy", "fk_batch_plan_upload",
    "fk_batch_plan_run", "fk_batch_plan_download", "fk_batch_plan_device_ptrs",
    "fk_batch_plan_launches", "fk_host_alloc", "fk_host_free", "fk_batch_plan_eval",
    "fk_batch_plan_eval_download", "fk_batch_solve_device", "fk_fp64_peak_tflops",
    "fk_topology_lm_solve", "fk_topology_eval", "fk_topology_last_timing", "fk_batch_plan_sync",
    "fk_system_create", "fk_system_destroy", "fk_system_add_length", "fk_system_add_point", "fk_system_add_line",
    "fk_system_add_circle", "fk_system_fix", "fk_system_add_constraint", "fk_system_num_variables",
    "fk_system_num_constraints", "fk_system_element_variable", "fk_system_get_variables", "fk_system_set_variable",
    "fk_system_set_parameter", "fk_system_solve", "fk_system_residuals", "fk_system_num_components",
    "fk_system_component", "fk_topology_supernodal", "fk_batch_analyze", "fk_topology_analyze_kernel", "fk_system_analyze", "fk_batch_solve_lbfgs", "fk_batch_plan_run_lbfgs", "fk_system_solve_opts", "fk_system_single_pass_plan", "fk_system_recursive_assembly_plan", "fk_batch_solve_single_pass",
    "fk_set_lm_kernel", "fk_get_lm_kernel", "fk_topology_sketch_kernel_info",
    "fk_topology_batch_kernel", "fk_topology_lbfgs_kernel", "fk_lbfgs_solve", "fk_lbfgs_solve_batch", "fk_batch_plan_run_lbfgs_global",
    "fk_system_solve_options", "fk_batch_system_solve", "fk_batch_system_solve_begin", "fk_batch_system_solve_wait", "fk_batch_solve_device_begin", "fk_batch_solve_device_wait", "fk_topology_cache_configure", "fk_topology_cache_clear", "fk_topology_cache_stats",
    "fk_system_batch_solve", "fk_system_batch_layout", "fk_system_batch_solve_single_pass", "fk_system_single_pass_batch_layout",
    "fk_system_batch_solve_recursive_assembly", "fk_system_recursive_assembly_batch_layout", "fk_system_batch_analyze",
    "fk_system_batch_residuals", "fk_systems_solve", "fk_systems_layout", "fk_systems_analyze", "fk_systems_residuals",
    "fk_systems_analyze_layout",
]

_lib = None


class FiksiError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__(f"fiksi_b200 error {code}: {msg}")
        self.code = code


def lib() -> C.CDLL:
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise ImportError(
                f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                "(fiksi_b200 has no CPU / pure-Python fallback)")
        L = C.CDLL(LIB_PATH)
        L.fk_last_error.restype = C.c_char_p
        L.fk_host_alloc.restype = C.c_void_p
        L.fk_host_alloc.argtypes = [C.c_size_t]
        L.fk_host_free.argtypes = [C.c_void_p]
        L.fk_batch_plan_launches.restype = C.c_uint64
        L.fk_batch_plan_launches.argtypes = [C.c_void_p]
        for name in ("fk_system_add_length", "fk_system_add_point", "fk_system_add_line", "fk_system_add_circle",
                     "fk_system_add_constraint", "fk_system_num_variables", "fk_system_num_constraints",
                     "fk_system_element_variable", "fk_system_num_components"):
            getattr(L, name).restype = C.c_uint32
        u32p, f64p = C.POINTER(C.c_uint32), C.POINTER(C.c_double)
        for name in ("fk_system_batch_solve_single_pass", "fk_system_batch_solve_recursive_assembly"):
            getattr(L, name).argtypes = [C.c_void_p, C.c_int, C.c_uint32, f64p, f64p, f64p, C.POINTER(FkReport), C.c_uint32, u32p,
                                         C.c_int]
        for name in ("fk_system_single_pass_batch_layout", "fk_system_recursive_assembly_batch_layout"):
            getattr(L, name).argtypes = [C.c_void_p, u32p, u32p, u32p, u32p, u32p]
        L.fk_system_batch_analyze.argtypes = [C.c_void_p, C.c_uint32, f64p, f64p, C.POINTER(C.c_uint8), C.c_int]
        L.fk_system_batch_residuals.argtypes = [C.c_void_p, C.c_uint32, f64p, f64p, f64p, C.c_int]
        sysp, optp = C.POINTER(C.c_void_p), C.POINTER(FkSolvingOptions)
        L.fk_systems_solve.argtypes = [C.c_uint32, sysp, optp, C.POINTER(FkReport), C.c_uint32, u32p, C.c_int]
        L.fk_systems_layout.argtypes = [C.c_uint32, sysp, optp, u32p, u32p, u32p, u32p]
        L.fk_systems_analyze.argtypes = [C.c_uint32, sysp, C.POINTER(C.c_uint8), C.c_uint64, C.c_int]
        L.fk_systems_residuals.argtypes = [C.c_uint32, sysp, f64p, C.c_uint64, C.c_int]
        L.fk_systems_analyze_layout.argtypes = [C.c_uint32, sysp, u32p, u32p, u32p]
        _lib = L
    return _lib


def check(rc):
    if rc != 0:
        raise FiksiError(rc, lib().fk_last_error().decode())


def ptr(a, t):
    return a.ctypes.data_as(C.POINTER(t))


def make_problem(vars_, kind, idx, param, free_vars, rows):
    """FkProblem over numpy arrays; returns (problem, keepalive tuple)."""
    vars_ = np.ascontiguousarray(vars_, dtype=np.float64)
    kind = np.ascontiguousarray(kind, dtype=np.uint8)
    idx = np.ascontiguousarray(idx, dtype=np.uint32).reshape(-1, 4)
    param = np.ascontiguousarray(param, dtype=np.float64)
    free_vars = np.ascontiguousarray(free_vars, dtype=np.uint32)
    rows = np.ascontiguousarray(rows, dtype=np.uint32)
    p = FkProblem(len(vars_), ptr(vars_, C.c_double), len(kind), ptr(kind, C.c_uint8),
                  ptr(idx, C.c_uint32), ptr(param, C.c_double), len(free_vars),
                  ptr(free_vars, C.c_uint32), len(rows), ptr(rows, C.c_uint32))
    return p, (vars_, kind, idx, param, free_vars, rows)
