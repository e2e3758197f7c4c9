"""Python mirror of fiksi::System over the C ABI's fk_system_* functions (same operations, names
and argument order as the reference's constructors; see include/fiksi_b200.h).  Same duck-typed
interface as ``oracle.System`` so that tests/scenarios.py builds both."""
from __future__ import annotations

import ctypes as C

import numpy as np

from ._lib import FkReport, FkSolvingOptions, REPORT_DTYPE, check, lib, ptr

_BAD = 0xFFFFFFFF
_OPTIMIZERS = {"lm": 0, "lbfgs": 1}


class System:
    def __init__(self):
        self._h = C.c_void_p()
        check(lib().fk_system_create(C.byref(self._h)))
        self._reports = np.zeros(0, dtype=REPORT_DTYPE)

    def _id(self, v):
        if v == _BAD:
            raise ValueError("invalid element / constraint arguments")
        return v

    # elements (fiksi/src/elements/mod.rs:280-454)
    def add_point(self, x, y): return self._id(lib().fk_system_add_point(self._h, C.c_double(x), C.c_double(y)))
    def add_length(self, l): return self._id(lib().fk_system_add_length(self._h, C.c_double(l)))
    def add_line(self, p1, p2): return self._id(lib().fk_system_add_line(self._h, p1, p2))
    def add_circle(self, c, r): return self._id(lib().fk_system_add_circle(self._h, c, r))
    def fix(self, e): check(lib().fk_system_fix(self._h, e, 1))
    def unfix(self, e): check(lib().fk_system_fix(self._h, e, 0))

    def _c(self, tag, elements, param=0.0):
        arr = (C.c_uint32 * len(elements))(*elements)
        return self._id(lib().fk_system_add_constraint(self._h, tag, arr, len(elements), C.c_double(param)))

    # constraints (fiksi/src/constraints/mod.rs:317-891)
    def point_point_coincidence(self, a, b): return self._c(0, [a, b])
    def point_point_distance(self, a, b, d): return self._c(1, [a, b], d)
    def point_point_point_angle(self, a, b, c, ang): return self._c(2, [a, b, c], ang)
    def point_line_incidence(self, p, l): return self._c(3, [p, l])
    def point_line_distance(self, p, l, d): return self._c(4, [p, l], d)
    def point_circle_incidence(self, p, c): return self._c(5, [p, c])
    def segment_segment_length_equality(self, a, b, c, d): return self._c(6, [a, b, c, d])
    def line_line_angle(self, a, b, ang): return self._c(7, [a, b], ang)
    def line_line_parallelism(self, a, b): return self._c(8, [a, b])
    def line_line_perpendicularity(self, a, b): return self._c(9, [a, b])
    def line_circle_tangency(self, l, c): return self._c(10, [l, c])

    @property
    def variables(self):
        n = lib().fk_system_num_variables(self._h)
        out = np.zeros(max(n, 1))
        check(lib().fk_system_get_variables(self._h, ptr(out, C.c_double)))
        return out[:n]

    def set_variable(self, i, v): check(lib().fk_system_set_variable(self._h, i, C.c_double(v)))
    def set_parameter(self, c, v): check(lib().fk_system_set_parameter(self._h, c, C.c_double(v)))
    def element_variable(self, e): return lib().fk_system_element_variable(self._h, e)
    def num_constraints(self): return lib().fk_system_num_constraints(self._h)

    def point(self, e):
        i = self.element_variable(e)
        v = self.variables
        return float(v[i]), float(v[i + 1])

    def _solve(self, decomposer, perturb, optimizer, cap):
        if optimizer not in _OPTIMIZERS:
            raise ValueError(f"optimizer must be 'lm' or 'lbfgs', not {optimizer!r}")
        opts = FkSolvingOptions(_OPTIMIZERS[optimizer], decomposer, int(bool(perturb)), 0)
        reps = np.zeros(max(1, cap), dtype=REPORT_DTYPE)
        n = C.c_uint32(0)
        check(lib().fk_system_solve_options(self._h, C.byref(opts), reps.ctypes.data_as(C.POINTER(FkReport)), len(reps), C.byref(n)))
        self._reports = reps[:n.value]

    def solve(self, perturb=True, optimizer="lm"):
        """System::solve(SolvingOptions { optimizer, decomposer: None, perturb }) on the GPU; optimizer 'lm'
        (LevenbergMarquardt, the default) or 'lbfgs' (LBfgs)."""
        self._solve(0, perturb, optimizer, lib().fk_system_num_components(self._h))

    def _variant_rows(self, vars, params, n):
        """(n_variables, vars [count][n_variables] or None, params [count][n_constraints] or None, count) of a batch call."""
        nv, ncon = lib().fk_system_num_variables(self._h), self.num_constraints()
        def rows(a, width):
            a = np.ascontiguousarray(a, dtype=np.float64)
            return a.reshape(len(a) if a.ndim == 2 else -1, width)
        if vars is not None:
            vars = rows(vars, nv)
        if params is not None:
            params = rows(params, ncon)
        sizes = {len(a) for a in (vars, params) if a is not None}
        if n is not None:
            sizes.add(int(n))
        if len(sizes) != 1:
            raise ValueError("give vars, params or n, with one number of variants")
        return nv, vars, params, sizes.pop()

    def batch_layout(self):
        """(solved components, distinct component structures, [components per structure]) of batch_solve's plan (host
        only)."""
        nc, ns = C.c_uint32(0), C.c_uint32(0)
        check(lib().fk_system_batch_layout(self._h, C.byref(nc), C.byref(ns), None))
        mult = np.zeros(max(ns.value, 1), np.uint32)
        check(lib().fk_system_batch_layout(self._h, C.byref(nc), C.byref(ns), ptr(mult, C.c_uint32)))
        return int(nc.value), int(ns.value), mult[:ns.value].tolist()

    def batch_solve(self, vars=None, params=None, optimizer="lm", perturb=True, n_gpus=1, n=None):
        """System.solve(perturb, optimizer) of n variants of this drawing in one call (fk_system_batch_solve): variant v
        starts from variables vars[v] ([n][n_variables]) and constraint parameters params[v] ([n][n_constraints]); None
        takes this system's own values (then `n` says how many variants).  The system itself is not modified.  Returns
        (variables after each variant's solve [n][n_variables], reports [n][solved components] as REPORT_DTYPE)."""
        if optimizer not in _OPTIMIZERS:
            raise ValueError(f"optimizer must be 'lm' or 'lbfgs', not {optimizer!r}")
        nv, vars, params, count = self._variant_rows(vars, params, n)
        n_solved = self.batch_layout()[0]
        out = np.zeros((count, nv))
        reps = np.zeros((count, n_solved), dtype=REPORT_DTYPE)
        opts = FkSolvingOptions(_OPTIMIZERS[optimizer], 0, int(bool(perturb)), 0)
        got = C.c_uint32(0)
        check(lib().fk_system_batch_solve(
            self._h, C.byref(opts), count, None if vars is None else ptr(vars, C.c_double),
            None if params is None else ptr(params, C.c_double), ptr(out, C.c_double),
            reps.ctypes.data_as(C.POINTER(FkReport)), n_solved, C.byref(got), int(n_gpus)))
        return out, reps

    def solve_single_pass(self, perturb=True, optimizer="lm"):
        """System::solve with Decomposer::SinglePass (assemble/mod.rs:169-210) on the GPU.  The reference runs LM here
        whatever the optimizer (assemble/mod.rs:191)."""
        self._solve(1, perturb, optimizer, len(self.single_pass_plan()))

    def _wave_layout(self, fn):
        n, nw, ns = C.c_uint32(0), C.c_uint32(0), C.c_uint32(0)
        check(fn(self._h, C.byref(n), C.byref(nw), C.byref(ns), None, None))
        wave = np.zeros(max(n.value, 1), np.uint32)
        struct = np.zeros(max(n.value, 1), np.uint32)
        check(fn(self._h, C.byref(n), C.byref(nw), C.byref(ns), ptr(wave, C.c_uint32), ptr(struct, C.c_uint32)))
        return int(n.value), int(nw.value), int(ns.value), wave[:n.value].tolist(), struct[:n.value].tolist()

    def _wave_solve(self, fn, n_steps, vars, params, perturb, n_gpus, n):
        nv, vars, params, count = self._variant_rows(vars, params, n)
        out = np.zeros((count, nv))
        reps = np.zeros((count, n_steps), dtype=REPORT_DTYPE)
        got = C.c_uint32(0)
        check(fn(self._h, int(bool(perturb)), count, None if vars is None else ptr(vars, C.c_double),
                 None if params is None else ptr(params, C.c_double), ptr(out, C.c_double),
                 reps.ctypes.data_as(C.POINTER(FkReport)), n_steps, C.byref(got), int(n_gpus)))
        return out, reps

    def single_pass_batch_layout(self):
        """(sets, waves, distinct set structures, [wave of each set], [structure of each set]) of batch_solve_single_pass's
        plan (host only)."""
        return self._wave_layout(lib().fk_system_single_pass_batch_layout)

    def batch_solve_single_pass(self, vars=None, params=None, perturb=True, n_gpus=1, n=None):
        """System.solve_single_pass(perturb) of n variants of this drawing in one call (fk_system_batch_solve_single_pass);
        arguments as batch_solve.  The system itself is not modified.  Returns (variables after each variant's solve
        [n][n_variables], reports [n][solved sets] as REPORT_DTYPE, in the order solve_single_pass reports them)."""
        return self._wave_solve(lib().fk_system_batch_solve_single_pass, self.single_pass_batch_layout()[0], vars, params, perturb,
                                n_gpus, n)

    def solve_recursive_assembly(self, perturb=True, optimizer="lm"):
        """System::solve with Decomposer::RecursiveAssembly (assemble/mod.rs:212-277) on the GPU.  The reference runs LM
        here whatever the optimizer (assemble/mod.rs:224)."""
        self._solve(2, perturb, optimizer, self.recursive_assembly_plan()[0])

    def recursive_assembly_plan(self):
        """(number of steps, serialised plan words) of fk_system_recursive_assembly_plan (host only)."""
        nw, ns = C.c_uint32(0), C.c_uint32(0)
        check(lib().fk_system_recursive_assembly_plan(self._h, None, 0, C.byref(nw), C.byref(ns)))
        out = np.zeros(max(nw.value, 1), dtype=np.uint32)
        check(lib().fk_system_recursive_assembly_plan(self._h, ptr(out, C.c_uint32), nw.value, C.byref(nw), C.byref(ns)))
        return int(ns.value), out[:nw.value].tolist()

    def recursive_assembly_batch_layout(self):
        """(steps, waves, distinct step structures, [wave of each step], [structure of each step]) of
        batch_solve_recursive_assembly's plan (host only)."""
        return self._wave_layout(lib().fk_system_recursive_assembly_batch_layout)

    def batch_solve_recursive_assembly(self, vars=None, params=None, perturb=True, n_gpus=1, n=None):
        """System.solve_recursive_assembly(perturb) of n variants of this drawing in one call
        (fk_system_batch_solve_recursive_assembly); arguments as batch_solve.  The system itself is not modified.  Returns
        (variables after each variant's solve [n][n_variables], reports [n][steps] as REPORT_DTYPE, in the order
        solve_recursive_assembly reports them).  Where a step moves points, coordinates may differ from the per-variant solve
        in the last places (include/fiksi_b200.h states the contract)."""
        return self._wave_solve(lib().fk_system_batch_solve_recursive_assembly, self.recursive_assembly_batch_layout()[0], vars,
                                params, perturb, n_gpus, n)

    def batch_analyze(self, vars=None, params=None, n_gpus=1, n=None):
        """System.analyze() of n variants of this drawing in one call (fk_system_batch_analyze); arguments as batch_solve.
        Returns uint8 [n][n_constraints]: how many of each constraint's expressions were found dependent, so that variant
        v's analyze() is np.repeat(np.arange(n_constraints), dependent[v]).  The system itself is not modified."""
        _, vars, params, count = self._variant_rows(vars, params, n)
        out = np.zeros((count, self.num_constraints()), np.uint8)
        check(lib().fk_system_batch_analyze(self._h, count, None if vars is None else ptr(vars, C.c_double),
                                            None if params is None else ptr(params, C.c_double), ptr(out, C.c_uint8), int(n_gpus)))
        return out

    def batch_residuals(self, vars=None, params=None, n_gpus=1, n=None):
        """System.residuals() of n variants of this drawing in one call (fk_system_batch_residuals); arguments as batch_solve.
        Returns float64 [n][n_constraints].  The system itself is not modified."""
        _, vars, params, count = self._variant_rows(vars, params, n)
        out = np.zeros((count, self.num_constraints()))
        check(lib().fk_system_batch_residuals(self._h, count, None if vars is None else ptr(vars, C.c_double),
                                              None if params is None else ptr(params, C.c_double), ptr(out, C.c_double), int(n_gpus)))
        return out

    def single_pass_plan(self):
        """[(free variables, expressions), ...] of fk_system_single_pass_plan (host only)."""
        sizes = np.zeros(3, dtype=np.uint32)
        check(lib().fk_system_single_pass_plan(self._h, ptr(sizes, C.c_uint32), None, None, None, None))
        n, nf, ne = (int(x) for x in sizes)
        fp = np.zeros(n + 1, np.uint32); fv = np.zeros(max(nf, 1), np.uint32)
        ep = np.zeros(n + 1, np.uint32); ex = np.zeros(max(ne, 1), np.uint32)
        check(lib().fk_system_single_pass_plan(self._h, ptr(sizes, C.c_uint32), ptr(fp, C.c_uint32), ptr(fv, C.c_uint32),
                                               ptr(ep, C.c_uint32), ptr(ex, C.c_uint32)))
        return [(fv[fp[k]:fp[k + 1]].tolist(), ex[ep[k]:ep[k + 1]].tolist()) for k in range(n)]

    def reports(self):
        return [{k: r[k].item() for k in REPORT_DTYPE.names} for r in self._reports]

    def residuals(self):
        n = self.num_constraints()
        out = np.zeros(max(n, 1))
        check(lib().fk_system_residuals(self._h, ptr(out, C.c_double)))
        return out[:n]

    def analyze(self):
        """System::analyze (lib.rs:454-458): ids of the constraints flagged as over-constraining."""
        cap = max(1, 2 * self.num_constraints())
        out = np.zeros(cap, dtype=np.uint32)
        n = C.c_uint32(0)
        check(lib().fk_system_analyze(self._h, ptr(out, C.c_uint32), cap, C.byref(n)))
        return out[:n.value].tolist()

    def calculate_residual(self, c):
        return float(self.residuals()[c])

    def components(self):
        out = []
        for ci in range(lib().fk_system_num_components(self._h)):
            ne, nc = C.c_uint32(0), C.c_uint32(0)
            check(lib().fk_system_component(self._h, ci, C.byref(ne), None, C.byref(nc), None))
            el = np.zeros(max(ne.value, 1), np.uint32)
            co = np.zeros(max(nc.value, 1), np.uint32)
            check(lib().fk_system_component(self._h, ci, None, ptr(el, C.c_uint32), None, ptr(co, C.c_uint32)))
            out.append((el[:ne.value].tolist(), co[:nc.value].tolist()))
        return out

    def close(self):
        if self._h:
            lib().fk_system_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def _systems_call(systems, optimizer, perturb):
    if optimizer not in _OPTIMIZERS:
        raise ValueError(f"optimizer must be 'lm' or 'lbfgs', not {optimizer!r}")
    handles = (C.c_void_p * max(len(systems), 1))(*[s._h for s in systems])
    return handles, FkSolvingOptions(_OPTIMIZERS[optimizer], 0, int(bool(perturb)), 0)


def systems_layout(systems, optimizer="lm"):
    """(solved components, distinct structures across the drawings, [instances per structure], [launch kind per structure:
    0 heterogeneous, 1 uniform batch, 2 sparse batch]) of solve_systems' plan (host only, fk_systems_layout)."""
    handles, opts = _systems_call(systems, optimizer, True)
    nc, ns = C.c_uint32(0), C.c_uint32(0)
    check(lib().fk_systems_layout(len(systems), handles, C.byref(opts), C.byref(nc), C.byref(ns), None, None))
    inst = np.zeros(max(ns.value, 1), np.uint32)
    kind = np.zeros(max(ns.value, 1), np.uint32)
    check(lib().fk_systems_layout(len(systems), handles, C.byref(opts), C.byref(nc), C.byref(ns), ptr(inst, C.c_uint32),
                                  ptr(kind, C.c_uint32)))
    return int(nc.value), int(ns.value), inst[:ns.value].tolist(), kind[:ns.value].tolist()


def solve_systems(systems, optimizer="lm", perturb=True, n_gpus=1):
    """System.solve(perturb, optimizer) of every system in `systems` (different drawings) in one call (fk_systems_solve).
    The systems are modified in place, exactly as each one's own solve() would modify it; nothing is modified when the call
    fails.  Returns one REPORT_DTYPE array per system: the reports of its solved components, in component order."""
    handles, opts = _systems_call(systems, optimizer, perturb)
    n = len(systems)
    cap = sum(lib().fk_system_num_constraints(s._h) for s in systems)  # every solved component holds a constraint
    reps = np.zeros(max(cap, 1), dtype=REPORT_DTYPE)
    solved = np.zeros(max(n, 1), np.uint32)
    check(lib().fk_systems_solve(n, handles, C.byref(opts), reps.ctypes.data_as(C.POINTER(FkReport)), len(reps), ptr(solved, C.c_uint32),
                                 int(n_gpus)))
    ends = np.cumsum(solved[:n])
    return [reps[e - k:e].copy() for e, k in zip(ends.tolist(), solved[:n].tolist())]


def _handles(systems):
    return (C.c_void_p * max(len(systems), 1))(*[s._h for s in systems])


def systems_analyze_layout(systems):
    """(distinct analyze structures across the drawings, [instances per structure], [launch kind per structure: 0 heterogeneous
    warp launch, 1 one launch of the kernel choose_analyze picks]) of analyze_systems' plan (host only,
    fk_systems_analyze_layout)."""
    handles = _handles(systems)
    ns = C.c_uint32(0)
    check(lib().fk_systems_analyze_layout(len(systems), handles, C.byref(ns), None, None))
    inst = np.zeros(max(ns.value, 1), np.uint32)
    kind = np.zeros(max(ns.value, 1), np.uint32)
    check(lib().fk_systems_analyze_layout(len(systems), handles, C.byref(ns), ptr(inst, C.c_uint32), ptr(kind, C.c_uint32)))
    return int(ns.value), inst[:ns.value].tolist(), kind[:ns.value].tolist()


def _ragged(systems, out):
    ends = np.cumsum([s.num_constraints() for s in systems], dtype=np.int64)
    return [out[e - s.num_constraints():e].copy() for e, s in zip(ends.tolist(), systems)]


def analyze_systems(systems, n_gpus=1):
    """System.analyze() of every system in `systems` (different drawings) in one call (fk_systems_analyze).  Returns one uint8
    array per system: how many of each constraint's expressions were found dependent, so that system i's analyze() is
    np.repeat(np.arange(num_constraints), counts[i]).  No system is modified; the same system may appear more than once."""
    total = sum(s.num_constraints() for s in systems)
    out = np.zeros(max(total, 1), np.uint8)
    check(lib().fk_systems_analyze(len(systems), _handles(systems), ptr(out, C.c_uint8), total, int(n_gpus)))
    return _ragged(systems, out)


def systems_residuals(systems, n_gpus=1):
    """System.residuals() of every system in `systems` (different drawings) in one call (fk_systems_residuals).  Returns one
    float64 array per system.  No system is modified; the same system may appear more than once."""
    total = sum(s.num_constraints() for s in systems)
    out = np.zeros(max(total, 1))
    check(lib().fk_systems_residuals(len(systems), _handles(systems), ptr(out, C.c_double), total, int(n_gpus)))
    return _ragged(systems, out)
