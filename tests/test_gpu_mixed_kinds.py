"""Mixed-kind CAD drawings (tests/cad_drawings.py: every constraint-level kind, fixed points, rows that name a shared
corner twice) on every LM path, against the CPU oracle under the parity rules of test_gpu_parity.py, and every kind
against an extended-precision evaluation of the mathematical constraint functions.

The extended-precision part (mpmath at 50 digits, no GPU) writes each function from its geometric definition, not from
the reference's formulas, and differentiates it numerically with respect to each free variable, so a row that names a
variable in two slots gets the sum the LM Jacobian must hold.  The oracle is pinned to the mathematics there; the
evaluation kernels are pinned to the oracle bit for bit (test_gpu_parity.py::test_eval_kernels_bit_exact_where_possible
and the eval_large test here); and every sketch that reports the residual exit is checked against the mathematics at
the coordinates it returned."""
import os

import mpmath
import numpy as np
import pytest

import cad_drawings as cd
import fiksi_b200 as fk
from fiksi_b200 import api

REL = 1e-9
SEED = 20261021
PATH1_SIZES = {"low": cd.PATH1_LOW, "mid": cd.PATH1_MID, "high": cd.PATH1_HIGH}
# (nx, ny, shared_vertices) -> (path, tile, smem_bytes): the footprints these sizes reach (symbolic.cpp, path selection)
FOOTPRINTS = {
    cd.PATH0 + (True,): (0, 16, 6024),
    cd.PATH0 + (False,): (0, 16, 6216),
    cd.PATH1_LOW + (True,): (1, 256, 27048),
    cd.PATH1_MID + (True,): (1, 256, 76464),
    cd.PATH1_HIGH + (True,): (1, 256, 184896),
    cd.PATH2_NATURAL + (True,): (2, 0, 558464),
}
PATH2_MAX_FRONT = 94


@pytest.fixture(scope="module")
def drawings():
    """Prepared drawings by (nx, ny, shared_vertices), built once per module."""
    cache = {}

    def get(nx, ny, shared=True):
        key = (nx, ny, shared)
        if key not in cache:
            cache[key] = cd.prepared(nx, ny, seed=SEED, shared_vertices=shared)
        return cache[key]
    return get


@pytest.fixture
def force_sparse():
    os.environ["FK_FORCE_PATH"] = "2"
    yield
    os.environ.pop("FK_FORCE_PATH", None)


def _topo(keep):
    vars_, kind, idx, param, free_vars, rows = keep
    return fk.Topology.from_arrays(len(vars_), kind, idx, free_vars, rows)


# ---- the mathematics, at 50 digits ---------------------------------------------------------------------------------
def _mp_residual(kind, v, p):
    """Constraint function of one expression from its geometric definition; v: slot values (mpf), p: parameter."""
    M = mpmath

    def cross(ax, ay, bx, by):
        return ax * by - ay * bx

    def angle(ux, uy, wx, wy):  # signed angle from u to w, in (-pi, pi]
        return M.atan2(cross(ux, uy, wx, wy), ux * wx + uy * wy)

    if kind == 0:  # the second variable equals the first
        return v[1] - v[0]
    if kind == 1:  # distance between two points
        return M.hypot(v[0] - v[2], v[1] - v[3]) - p
    if kind == 2:  # angle at the middle point, from the first arm to the second
        return angle(v[0] - v[2], v[1] - v[3], v[4] - v[2], v[5] - v[3]) - p
    if kind == 3:  # the point is on the line: (l2 - l1) x (p - l1)
        return cross(v[4] - v[2], v[5] - v[3], v[0] - v[2], v[1] - v[3])
    if kind == 4:  # signed distance of the point to the line
        return cross(v[4] - v[2], v[5] - v[3], v[0] - v[2], v[1] - v[3]) / M.hypot(v[4] - v[2], v[5] - v[3]) - p
    if kind == 5:  # the point is on the circle
        return M.hypot(v[0] - v[2], v[1] - v[3]) - v[4]
    if kind == 6:  # second segment's length minus the first's
        return M.hypot(v[4] - v[6], v[5] - v[7]) - M.hypot(v[0] - v[2], v[1] - v[3])
    if kind == 7:  # angle from the first line's direction to the second's
        return angle(v[2] - v[0], v[3] - v[1], v[6] - v[4], v[7] - v[5]) - p
    if kind == 8:  # parallel: second direction x first direction
        return cross(v[6] - v[4], v[7] - v[5], v[2] - v[0], v[3] - v[1])
    if kind == 9:  # perpendicular: first direction . second direction
        return (v[2] - v[0]) * (v[6] - v[4]) + (v[3] - v[1]) * (v[7] - v[5])
    if kind == 10:  # tangent: |distance of the centre to the line| - radius
        return abs(cross(v[2] - v[0], v[3] - v[1], v[4] - v[0], v[5] - v[1])) / M.hypot(v[2] - v[0], v[3] - v[1]) - v[6]
    raise ValueError(kind)


def _row_slots(keep):
    vars_, kind, idx, param, free_vars, rows = keep
    return [cd.slot_vars(int(kind[r]), idx[r]) for r in rows]


def mp_residuals(keep, vars_row, param_row, slots=None):
    """The mathematical residual of every row at the float values of vars_row (mpf list)."""
    vars_, kind, idx, param, free_vars, rows = keep
    slots = _row_slots(keep) if slots is None else slots
    with mpmath.workdps(50):
        return [_mp_residual(int(kind[r]), [mpmath.mpf(float(vars_row[q])) for q in sv], mpmath.mpf(float(param_row[r])))
                for r, sv in zip(rows, slots)]


def mp_jacobian(keep, vars_row, param_row):
    """Dense d(row)/d(free variable) at vars_row; a variable in two slots of a row moves both."""
    vars_, kind, idx, param, free_vars, rows = keep
    col = {int(q): c for c, q in enumerate(free_vars)}
    J = np.zeros((len(rows), len(free_vars)))
    with mpmath.workdps(50):
        for i, (r, sv) in enumerate(zip(rows, _row_slots(keep))):
            v0 = [mpmath.mpf(float(vars_row[q])) for q in sv]
            p = mpmath.mpf(float(param_row[r]))
            for q in sorted(set(sv) & set(col)):
                def f(t, q=q):
                    return _mp_residual(int(kind[r]), [x + t if s == q else x for s, x in zip(sv, v0)], p)
                J[i, col[q]] = float(mpmath.diff(f, 0))
    return J


def oracle_dense_jacobian(oracle, keep, vars_row, param_row):
    """oracle.evaluate's residuals and CSC Jacobian (augmented pattern without the damping rows) as a dense matrix."""
    vars_, kind, idx, param, free_vars, rows = keep
    op, okeep = oracle.make_problem(vars_row, kind, idx, param_row, free_vars, rows)
    sym = oracle.symbolic(op)
    n = len(free_vars)
    r, j = oracle.evaluate(op, np.asarray(vars_row)[free_vars], jac_nnz=len(sym["aug_rowidx"]) - n)
    J = np.zeros((len(rows), n))
    cp, ri, w = sym["aug_colptr"], sym["aug_rowidx"], 0
    for c in range(n):
        for k in range(cp[c], cp[c + 1] - 1):  # the last entry of a column is its damping row
            J[ri[k], c] = j[w]
            w += 1
    return r, J


def check_convergence_claim(keep, vars_row, param_row, x, rep):
    """A sketch that reports the residual exit: the mathematical residuals r* at its returned coordinates have
    ssr* < 1e-8 and agree with the reported ssr to 1e-10 relative + 1e-24, widened by what rounding the residuals alone
    allows: a double residual is within d = 8 ulp(1 + max |input|) of r* (+ 4 ulp(pi) for the atan2 kinds), so the
    sum of squares is within 2 |r*| |d| + |d|^2.  Near ssr ~ 1e-12 the residuals are ~ 1e-7 and their last-place
    rounding alone is 1e-9 of each, beyond a flat 1e-10."""
    if int(rep["exit_reason"]) != 0:
        return
    vars_, kind, idx, param, free_vars, rows = keep
    v = np.array(vars_row, dtype=np.float64)
    v[free_vars] = x
    slots = _row_slots(keep)
    with mpmath.workdps(50):
        res = mp_residuals(keep, v, param_row, slots)
        ssr = float(mpmath.fsum(r * r for r in res))
    inputs = np.array([max(np.max(np.abs(v[sv])), abs(param_row[e])) for e, sv in zip(rows, slots)])
    d = np.linalg.norm(8 * np.spacing(1.0 + inputs) + np.where(np.isin(kind[rows], (2, 7)), 4 * np.spacing(np.pi), 0.0))
    assert ssr < 1e-8, ssr
    assert abs(ssr - float(rep["ssr"])) <= 1e-10 * ssr + 1e-24 + 2 * np.sqrt(ssr) * d + d * d, (ssr, float(rep["ssr"]))


# ---- host only: the generator and the sizes ------------------------------------------------------------------------
SIZES = [cd.PATH0 + (True,), cd.PATH0 + (False,), cd.PATH1_LOW + (True,), cd.PATH1_MID + (True,),
         cd.PATH1_HIGH + (True,), cd.PATH2_NATURAL + (True,)]


@pytest.mark.parametrize("nx,ny,shared", SIZES)
def test_generator_invariants(oracle, drawings, nx, ny, shared):
    prep = drawings(nx, ny, shared)
    keep = prep["keep"]
    vars_, kind, idx, param, free_vars, rows = keep
    d = prep["drawing"]
    assert len(d["s"].prepare(perturb=False)) == 1  # one connected component
    fixed = {int(d["s"].element_variable(p)) + k for p in d["fixed"] for k in (0, 1)}
    assert sorted(free_vars.tolist()) == sorted(set(range(len(vars_))) - fixed)
    assert set(kind[rows].tolist()) == set(range(11)) and set(d["kinds"]) == set(range(11))
    slots = _row_slots(keep)
    assert sum(bool(set(sv) & fixed) for sv in slots) >= 4  # rows read the fixed points
    assert all(set(sv) - fixed for sv in slots)  # and every row has a free slot
    dup = cd.duplicated_free_slots(keep)
    assert (dup > 0) if shared else (dup == 0)
    # consistent by construction: the ground truth solves every row
    r, J = oracle_dense_jacobian(oracle, keep, vars_, param)
    assert np.max(np.abs(r)) < 1e-13
    # full column rank at the ground truth
    sv = np.linalg.svd(J, compute_uv=False)
    assert sv[-1] / sv[0] >= 1e-8, sv[-1] / sv[0]
    # every angle row more than 0.1 rad away from +-pi (the wrap decision is not an atan2 last-place question)
    ang = np.isin(kind[rows], (2, 7))
    res = mp_residuals(keep, vars_, param)
    for k in np.nonzero(ang)[0]:
        assert abs(float(res[k]) + param[rows[k]]) < np.pi - cd.ANGLE_MARGIN
    # the Workload form (raw numbers, scaled by Workload.prepare) is the same problem
    w = cd.workload(nx, ny, 2, seed=SEED, shared_vertices=shared, amount=0.0)
    v, p, scale = w.prepare(perturb=False)
    assert np.array_equal(v[0], vars_) and np.array_equal(p[0], param) and scale[0] == prep["scale"]
    assert np.array_equal(w.kind, kind) and np.array_equal(w.idx, idx) and np.array_equal(w.rows, rows)


@pytest.mark.parametrize("nx,ny,shared", SIZES)
def test_sizes_land_on_their_paths(drawings, nx, ny, shared):
    keep = drawings(nx, ny, shared)["keep"]
    topo = _topo(keep)
    i = topo.info
    assert (i["path"], i["tile"], i["smem_bytes"]) == FOOTPRINTS[(nx, ny, shared)]
    assert set(keep[1][keep[5]].tolist()) == set(range(11))
    if i["path"] == 0:
        assert topo.sketch_kernel_info()["available"] == (not shared)
        assert topo.batch_kernel(4096) == ("tile" if shared else "sketch_pair")
    if i["path"] == 1:
        assert 24 * 1024 < i["smem_bytes"] <= 200 * 1024 and topo.batch_kernel(69) == "tile"
    if i["path"] == 2:
        assert 1500 <= i["n_free"] <= 3000
        assert topo.supernodal()["info"]["max_front"] == PATH2_MAX_FRONT
        assert topo.batch_kernel(8) == "sparse_batch"


# ---- host only: the oracle against the mathematics -----------------------------------------------------------------
@pytest.mark.parametrize("nx,ny,shared", [cd.PATH0 + (True,), cd.PATH0 + (False,), cd.PATH1_LOW + (True,)])
def test_oracle_evaluation_matches_extended_precision(oracle, drawings, nx, ny, shared):
    """oracle.evaluate's residuals and Jacobian against the 50-digit evaluation, at the ground truth and at two start
    variants: |r - r*| <= 1e-13 (1 + max |input|) (+ 4 ulp(pi) for the atan2 kinds), |J - J*| <= 1e-12 max(1, |J*|)."""
    prep = drawings(nx, ny, shared)
    keep = prep["keep"]
    vars_, kind, idx, param, free_vars, rows = keep
    v, p = cd.start_variants(prep, 2, seed=SEED + 1)
    slots = _row_slots(keep)
    trig = np.isin(kind[rows], (2, 7))
    for vr, pr in ((vars_, param), (v[0], p[0]), (v[1], p[1])):
        r, J = oracle_dense_jacobian(oracle, keep, vr, pr)
        rs = np.array([float(x) for x in mp_residuals(keep, vr, pr, slots)])
        inputs = np.array([max(np.max(np.abs(vr[sv])), abs(pr[e])) for e, sv in zip(rows, slots)])
        tol = 1e-13 * (1.0 + inputs) + np.where(trig, 4 * np.spacing(np.pi), 0.0)
        bad = np.abs(r - rs) > tol
        assert not bad.any(), [(int(kind[rows[k]]), r[k], rs[k]) for k in np.nonzero(bad)[0][:5]]
        Js = mp_jacobian(keep, vr, pr)
        bad = np.abs(J - Js) > 1e-12 * np.maximum(1.0, np.abs(Js))
        assert not bad.any(), [(int(kind[rows[a]]), a, b, J[a, b], Js[a, b]) for a, b in np.argwhere(bad)[:5]]


# ---- on the device -------------------------------------------------------------------------------------------------
def _rel(a, b):
    return float(np.max(np.abs(a - b)) / max(np.max(np.abs(b)), 1e-300)) if len(b) else 0.0


def _same_report(got, ref, what):
    for key in ("exit_reason", "trace_hash", "outer_iters", "factorizations", "accepted", "lambda"):
        assert got[key] == ref[key], (what, key, got, ref)
    assert abs(got["ssr"] - ref["ssr"]) <= REL * max(ref["ssr"], 1.0), what


def _single_against_oracle(oracle, keep, vr, pr, solve):
    """solve(vars row, param row, x0) -> (x, report) against oracle.lm_solve, then the convergence claim."""
    vars_, kind, idx, param, free_vars, rows = keep
    op, okeep = oracle.make_problem(vr, kind, idx, pr, free_vars, rows)
    xo, ro, trace = oracle.lm_solve(op, vr[free_vars])
    xg, rg = solve(vr, pr, vr[free_vars])
    _same_report(rg, ro, trace)
    assert _rel(xg, xo) <= REL, _rel(xg, xo)
    check_convergence_claim(keep, vr, pr, xg, rg)
    return xg, rg


def _batch_against_oracle(oracle, keep, v, p, xg, rg, claim_every=1):
    """A batch against oracle.lm_solve_batch_uniform: traces equal for >= 99.9 % of the sketches (every drawing has
    atan2 rows), the parity rules on those, the convergence claim on every claim_every-th sketch."""
    vars_, kind, idx, param, free_vars, rows = keep
    op, okeep = oracle.make_problem(v[0], kind, idx, p[0], free_vars, rows)
    xo, ro, _ = oracle.lm_solve_batch_uniform(op, v, p, threads=8)
    same = (rg["trace_hash"] == ro["trace_hash"]) & (rg["exit_reason"] == ro["exit_reason"])
    assert same.mean() >= 0.999, (same.mean(), np.nonzero(~same)[0][:8])
    for key in ("outer_iters", "factorizations", "accepted", "lambda"):
        assert np.array_equal(rg[key][same], ro[key][same]), key
    err = np.max(np.abs(xg[same] - xo[same]), axis=1) / np.max(np.abs(xo[same]), axis=1)
    assert err.max() <= REL, err.max()
    assert np.all(np.abs(rg["ssr"][same] - ro["ssr"][same]) <= REL * np.maximum(ro["ssr"][same], 1.0))
    for k in range(0, len(v), claim_every):
        check_convergence_claim(keep, v[k], p[k], xg[k], rg[k])
    return same


@pytest.mark.gpu
def test_eval_large_matches_oracle(oracle, drawings):
    """Topology.eval_large (K1/K2 on the global path, sparse_eval_kernel) on the natural path-2 drawing and on forced
    path-0 / path-1 drawings: residuals bit for bit except the atan2 kinds (within 4 ulp(pi)), Jacobian bit for bit."""
    cases = [(cd.PATH2_NATURAL + (True,), False), (cd.PATH0 + (True,), True), (cd.PATH1_MID + (True,), True)]
    for (nx, ny, shared), force in cases:
        prep = drawings(nx, ny, shared)
        keep = prep["keep"]
        vars_, kind, idx, param, free_vars, rows = keep
        if force:
            os.environ["FK_FORCE_PATH"] = "2"
        try:
            topo = _topo(keep)
        finally:
            os.environ.pop("FK_FORCE_PATH", None)
        assert topo.info["path"] == 2
        trig = np.isin(kind[rows], (2, 7))
        v, p = cd.start_variants(prep, 2, seed=SEED + 2)
        for vr, pr in ((vars_, param), (v[0], p[0]), (v[1], p[1])):
            r, j, _ = topo.eval_large(vr, pr, vr[free_vars])
            op, okeep = oracle.make_problem(vr, kind, idx, pr, free_vars, rows)
            ro, jo = oracle.evaluate(op, vr[free_vars], jac_nnz=topo.info["jac_nnz"])
            assert np.array_equal(r[~trig], ro[~trig]), (nx, ny)
            assert np.all(np.abs(r[trig] - ro[trig]) <= 4 * np.spacing(np.pi)), (nx, ny)
            assert np.array_equal(j, jo), (nx, ny, np.nonzero(j != jo)[0][:8])


@pytest.mark.gpu
def test_path0_tile_kernel_with_shared_vertices(oracle, drawings):
    """Rows that name a shared corner twice (eval_row sums their slots) through the tile kernel: a batch and lm_solve."""
    prep = drawings(*cd.PATH0, True)
    keep = prep["keep"]
    vars_, kind, idx, param, free_vars, rows = keep
    topo = _topo(keep)
    n = 1000
    assert topo.info["path"] == 0 and topo.batch_kernel(n) == "tile"
    v, p = cd.start_variants(prep, n, seed=SEED + 3)
    xg, rg = topo.batch_solve(v, p)
    _batch_against_oracle(oracle, keep, v, p, xg, rg, claim_every=7)
    for k in (0, 1, 2):
        fp, fkeep = fk.make_problem(v[k], kind, idx, p[k], free_vars, rows)
        _single_against_oracle(oracle, keep, v[k], p[k], lambda vr, pr, x0: fk.lm_solve(fp, x0))


@pytest.mark.gpu
@pytest.mark.parametrize("kernel", ["sketch_solo", "sketch_pair"])
def test_path0_sketch_kernel_without_shared_vertices(oracle, drawings, kernel):
    prep = drawings(*cd.PATH0, False)
    keep = prep["keep"]
    topo = _topo(keep)
    n = 2048 + 17
    assert topo.info["path"] == 0 and topo.batch_kernel(n) == "sketch_pair"
    v, p = cd.start_variants(prep, n, seed=SEED + 4)
    with api.lm_kernel(kernel):
        xg, rg = topo.batch_solve(v, p)
    _batch_against_oracle(oracle, keep, v, p, xg, rg, claim_every=23)


@pytest.mark.gpu
@pytest.mark.parametrize("size", list(PATH1_SIZES))
def test_path1_cta_kernel(oracle, drawings, size):
    """fk_batch_lm_kernel<256, -1> (mixed kinds, fixed slots, duplicated slots) at the three footprints: 69 sketches,
    every one against the oracle; single lm_solve calls run the same kernel and equal the batch bit for bit."""
    prep = drawings(*PATH1_SIZES[size], True)
    keep = prep["keep"]
    vars_, kind, idx, param, free_vars, rows = keep
    topo = _topo(keep)
    n = 69
    assert topo.info["path"] == 1 and topo.info["tile"] == 256 and topo.batch_kernel(n) == "tile"
    v, p = cd.start_variants(prep, n, seed=SEED + 5)
    xg, rg = topo.batch_solve(v, p)
    _batch_against_oracle(oracle, keep, v, p, xg, rg)
    for k in (0, 31, 68):
        xs, rs = topo.lm_solve(v[k], p[k], v[k][free_vars])
        assert np.array_equal(xs, xg[k])
        for key in rg.dtype.names:
            assert rs[key] == rg[k][key], key


@pytest.mark.gpu
def test_path2_natural_size(oracle, drawings):
    """K5 (multifrontal LDLt) through lm_solve on the natural path-2 drawing against the oracle."""
    prep = drawings(*cd.PATH2_NATURAL, True)
    keep = prep["keep"]
    topo = _topo(keep)
    assert topo.info["path"] == 2
    v, p = cd.start_variants(prep, 2, seed=SEED + 6)
    for k in range(2):
        _single_against_oracle(oracle, keep, v[k], p[k], topo.lm_solve)


@pytest.mark.gpu
@pytest.mark.parametrize("nx,ny,shared", [cd.PATH0 + (True,), cd.PATH0 + (False,), cd.PATH1_LOW + (True,)])
def test_forced_path2(oracle, drawings, force_sparse, nx, ny, shared):
    """The path-0 and path-1 drawings on the global sparse path: single (K5) and batched (sparse batch kernel)."""
    prep = drawings(nx, ny, shared)
    keep = prep["keep"]
    topo = _topo(keep)
    n = 6
    assert topo.info["path"] == 2 and topo.batch_kernel(n) == "sparse_batch"
    v, p = cd.start_variants(prep, n, seed=SEED + 7)
    for k in range(2):
        _single_against_oracle(oracle, keep, v[k], p[k], topo.lm_solve)
    xg, rg = topo.batch_solve(v, p)
    _batch_against_oracle(oracle, keep, v, p, xg, rg)
