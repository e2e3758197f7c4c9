"""fiksi_b200 — B200-native (sm_100a) implementation of Fiksi's numeric solve path.

The product is ``libfiksi_b200.so`` (C ABI in ``include/fiksi_b200.h``); this package is the thin
ctypes face used by the tests and the benchmark.
"""
from ._lib import FiksiError, FkProblem, FkReport, REPORT_DTYPE, LIB_PATH, lib, make_problem  # noqa: F401
from .api import (BatchPlan, Topology, device_count, fp64_peak_tflops, lbfgs_solve, lbfgs_solve_batch, lm_solve,  # noqa: F401
                  lm_solve_batch)
from .system import (System, analyze_systems, solve_systems, systems_analyze_layout, systems_layout,  # noqa: F401
                     systems_residuals)
