"""Batched LM solves of topologies on the global sparse path (info.path == 2): one CTA per sketch over the supernodal
tree (fk_sparse_batch_lm_kernel).  Every sketch must take the decisions of the single-system path and of the oracle;
small problems are forced onto the path with FK_FORCE_PATH=2 so that the reference scenarios reach it."""
import ctypes as C
import os

import numpy as np
import pytest

import cad_drawings as cd
import scenarios as sc
import fiksi_b200 as fk
from fiksi_b200 import workloads as wl
from fiksi_b200._lib import REPORT_DTYPE, lib

pytestmark = pytest.mark.gpu
REL_ORACLE = 1e-9
REL_SINGLE = 1e-11
DECISIONS = ("exit_reason", "trace_hash", "outer_iters", "factorizations", "accepted", "lambda")


@pytest.fixture
def force_sparse():
    os.environ["FK_FORCE_PATH"] = "2"
    yield
    os.environ.pop("FK_FORCE_PATH", None)


def _rel(a, b):
    return float(np.max(np.abs(a - b)) / max(np.max(np.abs(b)), 1e-300)) if len(b) else 0.0


def _topo(w):
    t = fk.Topology.from_arrays(w.n_vars, w.kind, w.idx, w.free_vars, w.rows)
    assert t.info["path"] == 2 and t.batch_kernel(8) == "sparse_batch"
    return t


def _perturbed(vars_, n, seed, amount=1e-3):
    """n copies of one variable row, copy 0 as given, the others scaled per variable by 1 + amount * U(-1, 1)."""
    rng = np.random.default_rng(seed)
    v = np.tile(vars_, (n, 1))
    v[1:] *= 1.0 + amount * rng.uniform(-1.0, 1.0, size=v[1:].shape)
    return np.ascontiguousarray(v)


def _check_oracle(oracle, kind, idx, free_vars, rows, v, p, xb, rb, k):
    op, keep = oracle.make_problem(v[k], kind, idx, p[k], free_vars, rows)
    xo, ro, trace = oracle.lm_solve(op, v[k][free_vars])
    for f in DECISIONS:
        assert rb[k][f] == ro[f], (k, f, trace, rb[k], ro)
    assert _rel(xb[k], xo) <= REL_ORACLE, (k, _rel(xb[k], xo))
    assert abs(rb[k]["ssr"] - ro["ssr"]) <= REL_ORACLE * max(ro["ssr"], 1.0)


def _check_single(topo, free_vars, v, p, xb, rb, ks):
    for k in ks:
        xs, rs = topo.lm_solve(v[k], p[k], v[k][free_vars])
        for f in DECISIONS:
            assert rb[k][f] == rs[f], (k, f, rb[k], rs)
        assert _rel(xb[k], xs) <= REL_SINGLE, (k, _rel(xb[k], xs))


# ---- 1. oracle parity on forced small systems ---------------------------------------------------------------
@pytest.mark.parametrize("name", sorted(sc.ALL))
def test_reference_scenarios_batched(oracle, force_sparse, name):
    b = sc.ALL[name](oracle.System)
    for c, (prob, scale, keep) in enumerate(b["s"].prepare(perturb=True)):
        vars_, kind, idx, param, free_vars, rows = keep
        topo = fk.Topology.from_arrays(len(vars_), kind, idx, free_vars, rows)
        assert topo.info["path"] == 2
        v = _perturbed(np.asarray(vars_, np.float64), 5, 100 + c)
        p = np.ascontiguousarray(np.tile(param, (5, 1)))
        xb, rb = topo.batch_solve(v, p)
        for k in range(5):
            _check_oracle(oracle, kind, idx, free_vars, rows, v, p, xb, rb, k)


@pytest.mark.parametrize("nx,ny", [(5, 4), (12, 9)])
def test_small_lattices_forced_batched(oracle, force_sparse, nx, ny):
    w = wl.lattice(nx, ny, n_sketches=6)
    v, p, _ = w.prepare()
    topo = _topo(w)
    xb, rb = topo.batch_solve(v, p)
    for k in range(6):
        _check_oracle(oracle, w.kind, w.idx, w.free_vars, w.rows, v, p, xb, rb, k)


# ---- 2. parity with the single-system path at natural size ---------------------------------------------------
@pytest.mark.parametrize("shape,n", [((30, 20), 64), ((32, 32), 16), ((64, 50), 8), ("truss", 32), ("cad", 6)])
def test_natural_size_matches_single_system_path(oracle, shape, n):
    if shape == "cad":  # every kind, fixed points, rows that name a variable twice, far-apart length equalities
        w = cd.workload(*cd.PATH2_NATURAL, n, seed=1)
    else:
        w = wl.truss(n, 1000) if shape == "truss" else wl.lattice(*shape, n_sketches=n)
    v, p, _ = w.prepare()
    topo = _topo(w)
    xb, rb = topo.batch_solve(v, p)
    _check_single(topo, w.free_vars, v, p, xb, rb, range(n))
    for k in range(4):
        _check_oracle(oracle, w.kind, w.idx, w.free_vars, w.rows, v, p, xb, rb, k)


def _irregular(seed, n_pts, extra, n):
    rng = np.random.default_rng(seed)
    pts = rng.uniform(0.0, 10.0, size=(n_pts, 2))
    edges = [(0, 1)]
    for k in range(2, n_pts):
        d = np.sum((pts[:k] - pts[k]) ** 2, axis=1)
        a, b = np.argsort(d)[:2]
        edges += [(int(a), k), (int(b), k)]
    for _ in range(extra):
        a, b = rng.choice(n_pts, size=2, replace=False)
        edges.append((int(min(a, b)), int(max(a, b))))
    kind = np.ones(len(edges), np.uint8)
    idx = np.array([[2 * a, 2 * b, 0, 0] for a, b in edges], np.uint32)
    dist = np.array([np.hypot(*(pts[a] - pts[b])) for a, b in edges])
    noisy = pts[None] + rng.uniform(-0.02, 0.02, size=(n,) + pts.shape)
    free_vars = np.arange(4, 2 * n_pts, dtype=np.uint32)  # the first two points pinned
    return wl.Workload("irregular", kind, idx, free_vars, np.arange(len(edges)), noisy.reshape(n, -1), np.tile(dist, (n, 1)))


@pytest.mark.parametrize("seed,n_pts,extra", [(2, 400, 150), (3, 700, 0)])
def test_irregular_graphs_batched(oracle, force_sparse, seed, n_pts, extra):
    w = _irregular(seed, n_pts, extra, 12)
    v, p, _ = w.prepare()
    topo = _topo(w)
    xb, rb = topo.batch_solve(v, p)
    _check_single(topo, w.free_vars, v, p, xb, rb, range(12))
    for k in range(4):
        _check_oracle(oracle, w.kind, w.idx, w.free_vars, w.rows, v, p, xb, rb, k)


# ---- 3. independence and determinism ------------------------------------------------------------------------
def _bits(x, r):
    return x.tobytes(), r.tobytes()


def test_independent_of_batch_position_and_deterministic():
    w = wl.lattice(30, 20, n_sketches=64)
    v, p, _ = w.prepare()
    topo = _topo(w)
    xb, rb = topo.batch_solve(v, p)
    xb2, rb2 = topo.batch_solve(v, p)
    assert _bits(xb, rb) == _bits(xb2, rb2)
    for k in (0, 17, 63):
        xa, ra = topo.batch_solve(v[k:k + 1], p[k:k + 1])
        assert _bits(xa[0], ra[0:1]) == _bits(xb[k], rb[k:k + 1])
    order = np.random.default_rng(5).permutation(64)
    xp, rp = topo.batch_solve(v[order], p[order])
    assert _bits(xp, rp) == _bits(xb[order], rb[order])


def test_nan_and_inconsistent_sketches_do_not_disturb_the_others():
    w = wl.lattice(30, 20, n_sketches=16)
    v, p, _ = w.prepare()
    topo = _topo(w)
    xb, rb = topo.batch_solve(v, p)
    bad_v = np.concatenate([v, v[:2]])
    bad_p = np.concatenate([p, p[:2]])
    bad_v[16, 7] = np.nan                 # a NaN coordinate
    bad_p[17, 5] *= 3.0                   # one distance that contradicts the others
    xm, rm = topo.batch_solve(bad_v, bad_p)
    assert _bits(xm[:16], rm[:16]) == _bits(xb, rb)
    for k in (16, 17):
        xs, rs = topo.lm_solve(bad_v[k], bad_p[k], bad_v[k][w.free_vars])
        for f in ("exit_reason", "trace_hash", "outer_iters", "factorizations", "accepted"):
            assert rm[k][f] == rs[f], (k, f, rm[k], rs)


# ---- 4. entry points ------------------------------------------------------------------------------------------
def _pinned(a):
    a = np.ascontiguousarray(a)
    buf = lib().fk_host_alloc(C.c_size_t(a.nbytes))
    h = np.ctypeslib.as_array((C.c_uint8 * a.nbytes).from_address(buf)).view(a.dtype).reshape(a.shape)
    h[...] = a
    return h, buf


def test_entry_points_agree_bit_for_bit():
    w = wl.lattice(30, 20, n_sketches=24)
    v, p, scale = w.prepare()
    topo = _topo(w)
    xb, rb = topo.batch_solve(v, p)
    n, nf = v.shape[0], w.free_vars.size
    hv, bv = _pinned(v)
    hp, bp = _pinned(p)
    outs = [_pinned(np.zeros((n, nf))) for _ in range(2)]
    reps = [_pinned(np.zeros(n, REPORT_DTYPE)) for _ in range(2)]
    try:
        topo.batch_solve_into(0, n, hv.ctypes.data, hp.ctypes.data, outs[0][0].ctypes.data, reps[0][0].ctypes.data)
        assert _bits(outs[0][0], reps[0][0]) == _bits(xb, rb)
        # two batches in flight, alternating output buffers
        for o, r in zip(outs, reps):
            o[0][...] = 0.0
            r[0][...] = np.zeros(n, REPORT_DTYPE)
        t0 = topo.batch_solve_begin(0, n, hv.ctypes.data, hp.ctypes.data, outs[0][0].ctypes.data, reps[0][0].ctypes.data)
        t1 = topo.batch_solve_begin(0, n, hv.ctypes.data, hp.ctypes.data, outs[1][0].ctypes.data, reps[1][0].ctypes.data)
        topo.batch_solve_wait(t0)
        topo.batch_solve_wait(t1)
        for o, r in zip(outs, reps):
            assert _bits(o[0], r[0]) == _bits(xb, rb)
    finally:
        for _, b in [(None, bv), (None, bp)] + outs + reps:
            lib().fk_host_free(C.c_void_p(b))
    # System::solve level: scale, perturbation and write-back on the device against host-prepared inputs
    xs, scales, rs = topo.batch_system_solve(w.raw_vars, w.raw_param)
    assert np.array_equal(scales, scale)
    assert rs.tobytes() == rb.tobytes()
    assert np.array_equal(xs, w.write_back(w.raw_vars, xb, scale)[:, w.free_vars])  # (xs: unscaled on the device)


def test_batch_system_solve_begin_wait_two_in_flight():
    w = wl.lattice(30, 20, n_sketches=10)
    topo = _topo(w)
    xs, scales, rs = topo.batch_system_solve(w.raw_vars, w.raw_param)
    n, nf = w.n, w.free_vars.size
    hv, bv = _pinned(w.raw_vars)
    hp, bp = _pinned(w.raw_param)
    outs = [_pinned(np.zeros((n, nf))) for _ in range(2)]
    reps = [_pinned(np.zeros(n, REPORT_DTYPE)) for _ in range(2)]
    try:
        toks = [topo.batch_system_solve_begin(0, n, hv.ctypes.data, hp.ctypes.data, outs[a][0].ctypes.data, reps[a][0].ctypes.data) for a in range(2)]
        for t in toks:
            topo.batch_system_solve_wait(t)
        for o, r in zip(outs, reps):
            assert o[0].tobytes() == xs.tobytes() and r[0].tobytes() == rs.tobytes()
    finally:
        for _, b in [(None, bv), (None, bp)] + outs + reps:
            lib().fk_host_free(C.c_void_p(b))


def test_batch_sizes(force_sparse):
    """0, 1, 3, one more than the resident CTAs (2 x 148 on a B200 at most), and several pipeline chunks (> 2,048)."""
    w = wl.lattice(5, 4, n_sketches=2600)
    v, p, _ = w.prepare()
    topo = _topo(w)
    x0, r0 = topo.batch_solve(v[:0], p[:0])
    assert x0.shape == (0, w.free_vars.size)
    xb, rb = topo.batch_solve(v, p)
    for n in (1, 3, 297, 2600):
        xs, rs = topo.batch_solve(v[:n], p[:n])
        assert _bits(xs, rs) == _bits(xb[:n], rb[:n]), n
    _check_single(topo, w.free_vars, v, p, xb, rb, [0, 1, 296, 2599])


def test_plan_run_is_idempotent():
    w = wl.lattice(32, 32, n_sketches=8)
    v, p, _ = w.prepare()
    topo = _topo(w)
    xb, rb = topo.batch_solve(v, p)
    plan = topo.plan(8)
    plan.upload(v, p)
    out = np.zeros((8, w.free_vars.size))
    rep = np.zeros(8, REPORT_DTYPE)
    for _ in range(3):
        out[...] = 0.0
        plan.run()
        plan.download(out, rep)
        lib().fk_batch_plan_sync(plan._h)
        assert _bits(out, rep) == _bits(xb, rb)
    plan.close()


@pytest.mark.skipif(fk.device_count() < 2, reason="needs two devices")
def test_two_devices_match_one():
    w = wl.lattice(30, 20, n_sketches=32)
    v, p, _ = w.prepare()
    topo = _topo(w)
    x1, r1 = topo.batch_solve(v, p, n_gpus=1)
    x2, r2 = topo.batch_solve(v, p, n_gpus=2)
    assert _bits(x1, r1) == _bits(x2, r2)


# ---- 5. limits -----------------------------------------------------------------------------------------------
def test_front_limit_and_refusals():
    w = wl.lattice(80, 60, n_sketches=2)  # largest front 260 rows
    v, p, _ = w.prepare()
    topo = fk.Topology.from_arrays(w.n_vars, w.kind, w.idx, w.free_vars, w.rows)
    for call in (lambda: topo.plan(2), lambda: topo.batch_solve(v, p), lambda: topo.batch_kernel(2)):
        with pytest.raises(fk.FiksiError) as e:
            call()
        assert e.value.code == -5 and "260" in str(e.value)
    w = wl.lattice(30, 20, n_sketches=2)
    v, p, _ = w.prepare()
    topo = _topo(w)
    plan = topo.plan(2)
    plan.upload(v, p)
    for call in (plan.eval, plan.run_lbfgs, lambda: topo.batch_solve_lbfgs(v, p)):
        with pytest.raises(fk.FiksiError) as e:
            call()
        assert e.value.code == -5
    plan.close()


# ---- 6. several topologies on one device, memory budget ---------------------------------------------------------
def test_topologies_with_different_fronts_share_the_device():
    """The larger front first (48x40: 174 rows), then a smaller one (30x20: 80 rows), then the first again: setting up
    the second topology must not shrink what the first may launch with."""
    big = wl.lattice(48, 40, n_sketches=4)
    vb, pb, _ = big.prepare()
    tb = _topo(big)
    plan_b = tb.plan(4)
    plan_b.upload(vb, pb)
    ref_b = tb.batch_solve(vb, pb)
    small = wl.lattice(30, 20, n_sketches=4)
    vs, ps, _ = small.prepare()
    ts = _topo(small)
    plan_s = ts.plan(4)
    plan_s.upload(vs, ps)
    ref_s = ts.batch_solve(vs, ps)
    for plan, ref, nf in ((plan_b, ref_b, big.free_vars.size), (plan_s, ref_s, small.free_vars.size), (plan_b, ref_b, big.free_vars.size)):
        out = np.zeros((4, nf))
        rep = np.zeros(4, REPORT_DTYPE)
        plan.run()
        plan.download(out, rep)
        lib().fk_batch_plan_sync(plan._h)
        assert _bits(out, rep) == _bits(*ref)
    x, r = tb.batch_solve(vb, pb)
    assert _bits(x, r) == _bits(*ref_b)
    plan_b.close()
    plan_s.close()


def test_workspace_budget_caps_ctas_for_long_systems():
    """A 12,000-point truss needs 3.9 MiB of workspace per CTA: a plan gets the 266 CTAs that 1 GiB holds rather than one
    per resident CTA (296 on a B200), and a batch larger than that still solves every sketch as the single-system path does."""
    w = wl.truss(300, 12000)
    v, p, _ = w.prepare()
    topo = _topo(w)
    xb, rb = topo.batch_solve(v, p)
    assert np.all(rb["exit_reason"] == 0)
    _check_single(topo, w.free_vars, v, p, xb, rb, [0, 299])
