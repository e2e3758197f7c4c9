"""Optimizer::LBfgs beyond shared memory: fk_lbfgs_cta_kernel (one CTA per sketch, the L-BFGS state in global memory),
fk_lbfgs_solve / fk_lbfgs_solve_batch for systems of every size, and System::solve with an optimizer.

Parity rule (as tests/test_gpu_lbfgs.py): on distance-only topologies every report field and every coordinate is
bit-identical to the oracle; with angle kinds at least 99.5 % of the traces are equal (an atan2 ulp may flip a Wolfe
test), coordinates within 1e-9 and ssr within 1e-9 * max(ssr, 1).  The CTA kernel repeats every floating-point operation
of the tile kernel in its order, so the two are bit-identical everywhere."""
import ctypes as C
import os

import numpy as np
import pytest

import oracle_system
import scenarios as sc
import fiksi_b200 as fk
from fiksi_b200 import workloads as wl
from fiksi_b200._lib import FkReport, FkSolvingOptions, REPORT_DTYPE, lib, make_problem

pytestmark = pytest.mark.gpu
REL = 1e-9
FIELDS = ("exit_reason", "outer_iters", "factorizations", "accepted", "ssr", "lambda", "trace_hash")


@pytest.fixture
def force_sparse():
    os.environ["FK_FORCE_PATH"] = "2"
    yield
    os.environ.pop("FK_FORCE_PATH", None)


def topo_of(w):
    return fk.Topology.from_arrays(w.n_vars, w.kind, w.idx, w.free_vars, w.rows)


def run_plan(topo, v, p, cta):
    n = v.shape[0]
    plan = topo.plan(n)
    plan.upload(v, p)
    plan.run_lbfgs_global() if cta else plan.run_lbfgs()
    x = np.zeros((n, topo.info["n_free"]))
    rep = np.zeros(n, REPORT_DTYPE)
    plan.download(x, rep)
    lib().fk_batch_plan_sync(plan._h)
    plan.close()
    return x, rep


def same_bits(a, b):
    a, b = np.ascontiguousarray(a), np.ascontiguousarray(b)
    return a.shape == b.shape and a.tobytes() == b.tobytes()


def problems_of(w, v, p, ks):
    out = [make_problem(v[k], w.kind, w.idx, p[k], w.free_vars, w.rows) for k in ks]
    return [q for q, _ in out], [keep for _, keep in out]


def solve_list(w, v, p, ks, n_gpus=1):
    probs, keep = problems_of(w, v, p, ks)
    xs, reps = fk.lbfgs_solve_batch(probs, [v[k][w.free_vars] for k in ks], n_gpus=n_gpus)
    return np.array(xs).reshape(len(ks), -1), reps


def check_oracle(oracle, w, v, p, xg, rg, exact, threads=8):
    op, _ = oracle.make_problem(v[0], w.kind, w.idx, p[0], w.free_vars, w.rows)
    xo, ro, _ = oracle.lbfgs_solve_batch_uniform(op, v, p, threads=threads)
    if exact:
        assert same_bits(rg, ro), [(k, rg[k], ro[k]) for k in range(len(rg)) if rg[k].tobytes() != ro[k].tobytes()][:3]
        assert same_bits(xg, xo)
        return
    same = (rg["trace_hash"] == ro["trace_hash"]) & (rg["exit_reason"] == ro["exit_reason"]) & (rg["outer_iters"] == ro["outer_iters"])
    assert same.mean() >= 0.995, f"trace equality {same.mean():.5f}"
    err = np.max(np.abs(xg[same] - xo[same]), axis=1) / np.maximum(np.max(np.abs(xo[same]), axis=1), 1e-300)
    assert err.max() <= REL, err.max()
    assert np.all(np.abs(rg["ssr"][same] - ro["ssr"][same]) <= REL * np.maximum(ro["ssr"][same], 1.0))


def tiled_cad(copies):
    """Disjoint circle_triangle_line copies (kinds 1, 2, 3, 7, 10) in one system, each with its own noise."""
    w = wl.cad_mix(copies)
    nv = w.n_vars
    idx = np.vstack([w.idx.astype(np.int64) + c * nv for c in range(copies)])
    kind = np.tile(w.kind, copies)
    raw = w.raw_vars[:copies].reshape(1, -1)
    par = w.raw_param[:copies].reshape(1, -1)
    free = np.concatenate([w.free_vars + c * nv for c in range(copies)])
    rows = np.concatenate([w.rows + c * len(w.kind) for c in range(copies)])
    return wl.Workload(f"cad_x{copies}", kind, idx, free, rows, raw, par)


# ---- 1. the CTA kernel against the tile kernel --------------------------------------------------------------------
def _tile_shapes():
    out = [("truss", wl.truss(2048)), ("cad_mix", wl.cad_mix(2048)),
           ("hinged16", wl.hinged_triangles(16, n_sketches=256)), ("hinged64", wl.hinged_triangles(64, n_sketches=64))]
    fams = wl.stress_families(n_each=128)
    names = [n for n, _ in fams]
    assert "nan_coincident_points" in names
    out += [(n, f) for n, f in fams if n in ("nan_coincident_points", "two_components_a") or names.index(n) % 3 == 0]
    return out


@pytest.mark.parametrize("name,w", _tile_shapes(), ids=lambda x: x if isinstance(x, str) else "")
def test_cta_kernel_matches_tile_kernel(name, w):
    v, p, _ = w.prepare()
    topo = topo_of(w)
    assert topo.info["path"] == 0 and topo.lbfgs_kernel(len(v)) == 0
    xt, rt = run_plan(topo, v, p, cta=False)
    xc, rc = run_plan(topo, v, p, cta=True)
    assert same_bits(rt, rc), name
    assert same_bits(xt, xc), name


# ---- 2. against the oracle beyond the wall ------------------------------------------------------------------------
@pytest.mark.parametrize("nx,ny,n,path", [(10, 8, 64, 1), (24, 20, 16, 2), (32, 32, 8, 2)])
def test_lattices_match_oracle(oracle, nx, ny, n, path):
    w = wl.lattice(nx, ny, n_sketches=n)
    v, p, _ = w.prepare()
    topo = topo_of(w)
    assert topo.info["path"] == path and topo.lbfgs_kernel(n) == 1
    xg, rg = run_plan(topo, v, p, cta=True)
    check_oracle(oracle, w, v, p, xg, rg, exact=True)
    xb, rb = solve_list(w, v, p, range(n))   # host buffers through fk_lbfgs_solve_batch: the same bits
    assert same_bits(rb, rg) and same_bits(xb, xg)


def test_single_48x40_matches_oracle(oracle):
    w = wl.lattice(48, 40)
    v, p, _ = w.prepare()
    prob, _ = make_problem(v[0], w.kind, w.idx, p[0], w.free_vars, w.rows)
    x, rep = fk.lbfgs_solve(prob, v[0][w.free_vars])
    rg = np.array([tuple(rep[f] for f in FIELDS)], dtype=REPORT_DTYPE)
    check_oracle(oracle, w, v, p, x[None, :], rg, exact=True, threads=1)


def test_long_truss_matches_oracle(oracle):
    w = wl.truss(4, n_points=1000)
    v, p, _ = w.prepare()
    assert topo_of(w).lbfgs_kernel(4) == 1
    xg, rg = solve_list(w, v, p, range(4))
    check_oracle(oracle, w, v, p, xg, rg, exact=True)


def test_tiled_cad_path1_matches_oracle(oracle):
    w = tiled_cad(40)
    v, p, _ = w.prepare()
    topo = topo_of(w)
    assert topo.info["path"] == 1 and topo.lbfgs_kernel(1) == 1
    xg, rg = solve_list(w, v, p, [0])
    check_oracle(oracle, w, v, p, xg, rg, exact=False, threads=1)


@pytest.mark.parametrize("nx,ny", [(4, 3), (7, 5)])
def test_forced_sparse_path_matches_oracle(oracle, force_sparse, nx, ny):
    w = wl.lattice(nx, ny, n_sketches=32)
    v, p, _ = w.prepare()
    topo = topo_of(w)
    assert topo.info["path"] == 2 and topo.lbfgs_kernel(32) == 1
    xg, rg = run_plan(topo, v, p, cta=True)
    check_oracle(oracle, w, v, p, xg, rg, exact=True)


# ---- 3. fk_lbfgs_solve_batch ---------------------------------------------------------------------------------------
def test_batch_of_mixed_paths_matches_single_solves():
    parts = [wl.truss(6), wl.lattice(10, 8, n_sketches=3), wl.lattice(24, 20, n_sketches=3)]  # paths 0, 1, 2
    items = []
    for w in parts:
        v, p, _ = w.prepare()
        for k in range(len(v)):
            items.append((w, v, p, k))
    order = [i for r in range(6) for i in range(len(items)) if (i % 6) == r]   # interleave the groups
    probs = [make_problem(v_[k], w_.kind, w_.idx, p_[k], w_.free_vars, w_.rows) for w_, v_, p_, k in (items[i] for i in order)]
    x0 = [items[i][1][items[i][3]][items[i][0].free_vars] for i in order]
    xs, reps = fk.lbfgs_solve_batch([q for q, _ in probs], x0)
    for j, i in enumerate(order):
        w, v, p, k = items[i]
        prob, _ = make_problem(v[k], w.kind, w.idx, p[k], w.free_vars, w.rows)
        x1, r1 = fk.lbfgs_solve(prob, v[k][w.free_vars])
        assert same_bits(xs[j], x1)
        assert all(reps[j][f] == r1[f] for f in FIELDS), (j, reps[j], r1)
    # the path-0 group is bit-identical to fk_batch_solve_lbfgs
    w = parts[0]
    v, p, _ = w.prepare()
    xt, rt = topo_of(w).batch_solve_lbfgs(v, p)
    xl, rl = solve_list(w, v, p, range(len(v)))
    assert same_bits(xt, xl) and same_bits(rt, rl)
    # the order of the list does not matter
    rev = order[::-1]
    xs2, reps2 = fk.lbfgs_solve_batch([probs[order.index(i)][0] for i in rev], [x0[order.index(i)] for i in rev])
    for j, i in enumerate(rev):
        jj = order.index(i)
        assert same_bits(xs2[j], xs[jj]) and reps2[j].tobytes() == reps[jj].tobytes()
    xs0, reps0 = fk.lbfgs_solve_batch([], [])
    assert xs0 == [] and len(reps0) == 0


@pytest.mark.skipif(fk.device_count() < 2, reason="needs two devices")
def test_two_devices_bit_identical():
    w = wl.lattice(24, 20, n_sketches=8)
    v, p, _ = w.prepare()
    x1, r1 = solve_list(w, v, p, range(8), n_gpus=1)
    x2, r2 = solve_list(w, v, p, range(8), n_gpus=2)
    assert same_bits(x1, x2) and same_bits(r1, r2)


# ---- 4. batch semantics ------------------------------------------------------------------------------------------
def test_independent_of_batch_and_repeatable():
    w = wl.lattice(10, 8, n_sketches=1000)
    v, p, _ = w.prepare()
    topo = topo_of(w)
    x, r = run_plan(topo, v, p, cta=True)   # 1,000 sketches: more than the resident CTAs
    x2, r2 = run_plan(topo, v, p, cta=True)
    assert same_bits(x, x2) and same_bits(r, r2)
    for k in (0, 517, 999):
        xa, ra = run_plan(topo, v[k:k + 1], p[k:k + 1], cta=True)
        assert same_bits(xa[0], x[k]) and same_bits(ra[0], r[k])


def test_workspace_budget_caps_ctas():
    """150x120 lattices (36,000 variables, about 5.6 MB of state per CTA): the 1 GiB workspace holds about 190 CTAs, fewer
    than the device keeps resident, and 200 sketches take more than one CTA each in turn.  Every copy of the same sketch
    gives the same bits as the sketch solved alone."""
    w = wl.lattice(150, 120, n_sketches=2)
    v, p, _ = w.prepare()
    ks = [k % 2 for k in range(200)]
    probs = [make_problem(v[k], w.kind, w.idx, p[k], w.free_vars, w.rows) for k in ks]
    xs, reps = fk.lbfgs_solve_batch([q for q, _ in probs], [v[k][w.free_vars] for k in ks])
    for k in (0, 1):
        prob, _ = make_problem(v[k], w.kind, w.idx, p[k], w.free_vars, w.rows)
        x1, r1 = fk.lbfgs_solve(prob, v[k][w.free_vars])
        for j in range(k, 200, 2):
            assert same_bits(xs[j], x1) and all(reps[j][f] == r1[f] for f in FIELDS), j


def test_nan_sketch_leaves_neighbours(oracle):
    fams = dict(wl.stress_families(n_each=64))
    w = fams["nan_coincident_points"]
    v, p, _ = w.prepare()
    good = wl.lattice(10, 8, n_sketches=4)
    vg, pg, _ = good.prepare()
    topo = topo_of(good)
    x0, r0 = run_plan(topo, vg, pg, cta=True)
    bad = vg.copy()
    bad[1, good.free_vars[0]] = np.nan
    x1, r1 = run_plan(topo, bad, pg, cta=True)
    for k in (0, 2, 3):
        assert same_bits(x0[k], x1[k]) and same_bits(r0[k], r1[k])
    # Against the oracle a NaN sketch compares exit reason and counters only: the oracle's dense gradient multiplies every
    # residual by the zeros of its row, so one non-finite residual makes every gradient entry NaN there, while the column
    # sums over the sparse pattern keep the other entries finite.
    op, _ = oracle.make_problem(bad[1], good.kind, good.idx, pg[1], good.free_vars, good.rows)
    r = oracle.evaluate(op, bad[1][good.free_vars])
    assert np.isnan(r).any() and np.isfinite(r).any()   # one NaN point: some rows NaN, the others finite
    xo, ro = oracle.lbfgs_solve(op, bad[1][good.free_vars])
    for f in ("exit_reason", "outer_iters", "factorizations", "accepted"):
        assert r1[1][f] == ro[f], (f, r1[1], ro)
    # the NaN family of the stress workload through both kernels
    topo_n = topo_of(w)
    xt, rt = run_plan(topo_n, v, p, cta=False)
    xc, rc = run_plan(topo_n, v, p, cta=True)
    assert same_bits(xt, xc) and same_bits(rt, rc)


def test_guard_exit_reproduced(oracle):
    """Exit 4 (the bisection guard of update(), lbfgs.rs:338-351) on the sketches of the stress families that reach it."""
    hits = 0
    for name, w in wl.stress_families(n_each=256):
        v, p, _ = w.prepare()
        topo = topo_of(w)
        xt, rt = run_plan(topo, v, p, cta=False)
        if not (rt["exit_reason"] == 4).any():
            continue
        xc, rc = run_plan(topo, v, p, cta=True)
        assert same_bits(rt, rc) and same_bits(xt, xc)
        ks = np.nonzero(rc["exit_reason"] == 4)[0][:4]
        for k in ks:
            op, _ = oracle.make_problem(v[k], w.kind, w.idx, p[k], w.free_vars, w.rows)
            _, ro = oracle.lbfgs_solve(op, v[k][w.free_vars])
            assert ro["exit_reason"] == 4 and ro["factorizations"] == rc[k]["factorizations"]
        hits += len(ks)
    if hits == 0:
        pytest.skip("no stress sketch reaches the guard")


# ---- 5. selection and limits -------------------------------------------------------------------------------------
def test_kernel_selection():
    for w in (wl.truss(4), wl.cad_mix(4), wl.hinged_triangles(64, n_sketches=4)):
        assert topo_of(w).lbfgs_kernel(4) == 0
    assert topo_of(wl.lattice(10, 8)).info["path"] == 1 and topo_of(wl.lattice(10, 8)).lbfgs_kernel(4) == 1
    assert topo_of(wl.lattice(24, 20)).info["path"] == 2 and topo_of(wl.lattice(24, 20)).lbfgs_kernel(4) == 1


def test_front_260_solves_while_the_plan_is_refused():
    w = wl.lattice(80, 60)
    v, p, _ = w.prepare()
    topo = topo_of(w)
    with pytest.raises(fk.FiksiError) as e:
        topo.plan(1)
    assert e.value.code == -5 and "260" in str(e.value)
    prob, _ = make_problem(v[0], w.kind, w.idx, p[0], w.free_vars, w.rows)
    x, rep = fk.lbfgs_solve(prob, v[0][w.free_vars])
    assert np.isfinite(x).all() and rep["exit_reason"] in (1, 2, 3)
    with pytest.raises(fk.FiksiError):
        topo.plan(1)    # still refused after the L-BFGS solve set up the topology's device tables


def test_150x120_repeatable_and_ssr_is_the_sequential_sum():
    w = wl.lattice(150, 120)
    v, p, _ = w.prepare()
    prob, _ = make_problem(v[0], w.kind, w.idx, p[0], w.free_vars, w.rows)
    x1, r1 = fk.lbfgs_solve(prob, v[0][w.free_vars])
    x2, r2 = fk.lbfgs_solve(prob, v[0][w.free_vars])
    assert same_bits(x1, x2) and r1 == r2
    topo = topo_of(w)
    r, _, _ = topo.eval_large(v[0], p[0], x1, want_j=False)
    s = 0.0
    for q in r:
        s += q * q
    assert s == r1["ssr"], (s, r1["ssr"])


# ---- 6. facade ---------------------------------------------------------------------------------------------------
def _facade_pair(name, oracle):
    return sc.ALL[name](oracle.System), sc.ALL[name](fk.System)


@pytest.mark.parametrize("name", sorted(sc.ALL))
def test_facade_scenarios_match_oracle(oracle, name):
    bo, bg = _facade_pair(name, oracle)
    vo, ro = oracle_system.solve(oracle, bo["s"], optimizer="lbfgs")
    bg["s"].solve(optimizer="lbfgs")
    rg = bg["s"].reports()
    assert len(rg) == len(ro)
    for a, b in zip(rg, ro):
        for f in ("exit_reason", "outer_iters", "factorizations", "accepted", "trace_hash", "lambda"):
            assert a[f] == b[f] or (a[f] != a[f] and b[f] != b[f]), (name, f, a, b)
        assert abs(a["ssr"] - b["ssr"]) <= REL * max(b["ssr"], 1.0) or (a["ssr"] != a["ssr"] and b["ssr"] != b["ssr"])
    vg = bg["s"].variables
    fin = np.isfinite(vo)
    assert np.array_equal(np.isfinite(vg), fin)
    assert np.all(np.abs(vg[fin] - vo[fin]) <= REL * np.maximum(np.abs(vo[fin]), 1.0)), name
    # residuals of the GPU system at its solved coordinates against the oracle system set to the oracle's coordinates
    for i, x in enumerate(vo):
        bo["s"].set_variable(i, float(x))
    res_o = np.array([bo["s"].calculate_residual(c) for c in range(bo["s"].num_constraints())])
    res_g = bg["s"].residuals()
    fin = np.isfinite(res_o)
    tol = 1e-6 * max(1.0, float(np.max(np.abs(vo[np.isfinite(vo)]), initial=1.0)))
    assert np.all(np.abs(res_g[fin] - res_o[fin]) <= tol), name


def test_facade_multi_component_with_a_large_one(oracle):
    """A small triangle next to a 24x20 lattice (path 2) in one system: both components through one batch call."""
    def build(S):
        s = S()
        w = wl.lattice(24, 20)
        raw = w.raw_vars[0]
        pts = [s.add_point(float(raw[2 * i]), float(raw[2 * i + 1])) for i in range(w.n_vars // 2)]
        for e in range(len(w.kind)):
            s.point_point_distance(pts[w.idx[e][0] // 2], pts[w.idx[e][1] // 2], float(w.raw_param[0][e]))
        a, b, c = s.add_point(500.0, 0.0), s.add_point(510.0, 1.0), s.add_point(505.0, 9.0)
        s.point_point_distance(a, b, 10.0); s.point_point_distance(b, c, 10.0); s.point_point_distance(c, a, 10.0)
        s.fix(pts[0])
        return s
    so, sg = build(oracle.System), build(fk.System)
    vo, ro = oracle_system.solve(oracle, so, optimizer="lbfgs")
    sg.solve(optimizer="lbfgs")
    rg = sg.reports()
    assert len(rg) == len(ro) == 2
    for a, b in zip(rg, ro):
        assert all(a[f] == b[f] for f in FIELDS), (a, b)
    assert np.array_equal(sg.variables, vo)


@pytest.mark.parametrize("method", ["solve_single_pass", "solve_recursive_assembly"])
@pytest.mark.parametrize("name", ["circle_triangle_line", "connected_triangles", "two_connected_components"])
def test_decomposers_run_lm_whatever_the_optimizer(method, name):
    """Same variables and reports, or the same refusal (RecursiveAssembly refuses the systems the reference panics on)."""
    def run(optimizer):
        b = sc.ALL[name](fk.System)
        try:
            getattr(b["s"], method)(optimizer=optimizer)
        except fk.FiksiError as e:
            return e.code
        return b["s"].variables, b["s"].reports()
    a, b = run("lm"), run("lbfgs")
    if isinstance(a, int):
        assert a == b
    else:
        assert np.array_equal(a[0], b[0]) and a[1] == b[1]


def test_invalid_options():
    b = sc.ALL["single_triangle"](fk.System)
    h = b["s"]._h
    n = C.c_uint32(0)
    reps = (FkReport * 4)()
    for opts in ((2, 0, 1, 0), (0, 3, 1, 0), (1, 0, 2, 0), (1, 0, 1, 7)):
        o = FkSolvingOptions(*opts)
        assert lib().fk_system_solve_options(h, C.byref(o), reps, 4, C.byref(n)) == -1, opts
    assert lib().fk_system_solve_options(h, None, reps, 4, C.byref(n)) == -1
    with pytest.raises(ValueError):
        b["s"].solve(optimizer="newton")
