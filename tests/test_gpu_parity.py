"""GPU parity tests proper (run on the B200 box with -m gpu): the CUDA path through the C ABI vs
the CPU oracle on the same seeded inputs.

Parity rules (SURVEY App. D): accept/reject trace, exit reason and iteration counts equal to the
oracle's; converged coordinates within 1e-9 relative (inf-norm, the tolerance north_star states);
final sum of squared residuals within 1e-9 of max(ssr_ref, ssr_initial-scale) — a pure relative
test on a converged ~1e-12 norm is ill-posed.  Residuals and Jacobian entries of the evaluation
kernels are bit-exact for every kind that has no atan2 and within 4 ulp of pi otherwise."""
import numpy as np
import pytest

import cad_drawings as cd
import scenarios as sc
import fiksi_b200 as fk
from fiksi_b200 import workloads as wl

pytestmark = pytest.mark.gpu
REL = 1e-9


def _rel(a, b):
    return float(np.max(np.abs(a - b)) / max(np.max(np.abs(b)), 1e-300)) if len(b) else 0.0


def _same_reports(got, ref):
    for key in ("exit_reason", "outer_iters", "factorizations", "accepted", "trace_hash"):
        assert np.array_equal(got[key], ref[key]), key
    assert np.array_equal(got["lambda"], ref["lambda"])


@pytest.mark.parametrize("name", sorted(sc.ALL))
def test_reference_scenarios_lm(oracle, name):
    """Every fiksi/src/tests scenario: the flattened problems assemble::solve would hand to
    levenberg_marquardt go through fk_lm_solve and through the oracle."""
    b = sc.ALL[name](oracle.System)
    for prob, scale, keep in b["s"].prepare(perturb=True):
        x0 = keep[0][keep[4]]
        xo, ro, trace = oracle.lm_solve(prob, x0)
        fp, fkeep = fk.make_problem(*keep)
        xg, rg = fk.lm_solve(fp, x0)
        assert rg["exit_reason"] == ro["exit_reason"], (name, trace, rg, ro)
        assert rg["trace_hash"] == ro["trace_hash"], (name, trace, rg, ro)
        assert (rg["outer_iters"], rg["factorizations"], rg["accepted"]) == (ro["outer_iters"], ro["factorizations"], ro["accepted"])
        assert rg["lambda"] == ro["lambda"]
        assert _rel(xg * scale, xo * scale) <= REL, (name, _rel(xg, xo))
        assert abs(rg["ssr"] - ro["ssr"]) <= REL * max(ro["ssr"], 1.0)


def test_fixed_variables_never_written(oracle):
    # tests/fixed.rs:36-40: only free values come back; fixed ones are not part of the output at all
    b = sc.single_triangle(oracle.System, fixed=1)
    (prob, scale, keep), = b["s"].prepare()
    assert keep[4].tolist() == [0, 1, 4, 5]
    fp, fkeep = fk.make_problem(*keep)
    xg, rg = fk.lm_solve(fp, keep[0][keep[4]])
    xo, ro, _ = oracle.lm_solve(prob, keep[0][keep[4]])
    assert len(xg) == 4 and rg["trace_hash"] == ro["trace_hash"] and _rel(xg, xo) <= REL


@pytest.mark.parametrize("maker,n", [(wl.truss, 2048), (wl.cad_mix, 2048)])
def test_uniform_batch_matches_oracle(oracle, maker, n):
    w = maker(n)
    v, p, scale = w.prepare()
    topo = fk.Topology.from_arrays(w.n_vars, w.kind, w.idx, w.free_vars, w.rows)
    xg, rg = topo.batch_solve(v, p)
    op, keep = oracle.make_problem(v[0], w.kind, w.idx, p[0], w.free_vars, w.rows)
    xo, ro, _ = oracle.lm_solve_batch_uniform(op, v, p, threads=8)
    same = (rg["trace_hash"] == ro["trace_hash"]) & (rg["exit_reason"] == ro["exit_reason"])
    # H2 of the survey: a near-threshold decision may flip; it must be (very) rare
    assert same.mean() >= 0.999, f"trace equality {same.mean():.5f}"
    err = np.max(np.abs(xg[same] - xo[same]), axis=1) / np.max(np.abs(xo[same]), axis=1)
    assert err.max() <= REL, err.max()
    assert np.all(rg["ssr"][same] <= ro["ssr"][same] + REL)
    unscaled = w.write_back(w.raw_vars, xg, scale)
    assert np.all(np.isfinite(unscaled))


def test_eval_kernels_bit_exact_where_possible(oracle):
    """K1 / K2 of paths 0 and 1 against oracle.evaluate.  The CAD drawings bring every kind, fixed variables and, with
    shared vertices, rows that name a free variable twice (K1's scatter sums those slots); the last one is on path 1."""
    cad = [lambda n: cd.workload(*cd.PATH0, n, seed=1, shared_vertices=True),
           lambda n: cd.workload(*cd.PATH0, n, seed=1, shared_vertices=False),
           lambda n: cd.workload(*cd.PATH1_MID, n, seed=1, shared_vertices=True)]
    for maker in [wl.truss, wl.cad_mix] + cad:
        w = maker(500)  # ragged last tile of the tile-staged kernel (S = 32 / 128)
        v, p, scale = w.prepare()
        topo = fk.Topology.from_arrays(w.n_vars, w.kind, w.idx, w.free_vars, w.rows)
        plan = topo.plan(w.n)
        plan.upload(v, p)
        m, jn = topo.info["n_rows"], topo.info["jac_nnz"]
        r = np.zeros((w.n, m)); j = np.zeros((w.n, jn)); r2 = np.zeros((w.n, m))
        plan.eval(0); plan.eval_download(r, j)
        plan.eval(1); plan.eval_download(r2, None)
        import torch
        torch.cuda.synchronize()
        assert np.array_equal(r, r2)
        trig = np.isin(w.kind[w.rows], (2, 7))
        for s in range(0, w.n, 37):
            op, keep = oracle.make_problem(v[s], w.kind, w.idx, p[s], w.free_vars, w.rows)
            ro, jo = oracle.evaluate(op, v[s][w.free_vars], jac_nnz=jn)
            assert np.array_equal(r[s][~trig], ro[~trig])
            assert np.all(np.abs(r[s][trig] - ro[trig]) <= 4 * np.spacing(np.pi))
            assert np.array_equal(j[s], jo)  # gradients contain no transcendental


def test_full_size_truss_batch_properties():
    """BASELINE config 2 at full size: 65,536 sketches.  Size-independent properties: every sketch
    leaves through the residual exit, the reported ssr is the K2 kernel's residual at the returned
    coordinates, re-solving the solution is a fixed point (idempotence), shards concatenate."""
    n = 65536
    w = wl.truss(n)
    v, p, scale = w.prepare()
    topo = fk.Topology.from_arrays(w.n_vars, w.kind, w.idx, w.free_vars, w.rows)
    x, rep = topo.batch_solve(v, p)
    assert np.all(rep["exit_reason"] == 0) and np.all(rep["ssr"] < 1e-8)
    assert rep["factorizations"].min() >= 1 and rep["factorizations"].max() < 40
    # residual check through the standalone evaluation kernel
    plan = topo.plan(n)
    v2 = v.copy(); v2[:, w.free_vars] = x
    plan.upload(v2, p)
    r = np.zeros((n, 37))
    plan.eval(1); plan.eval_download(r, None)
    import torch
    torch.cuda.synchronize()
    ssr = np.zeros(n)
    for k in range(37):
        ssr = ssr + r[:, k] * r[:, k]
    assert np.array_equal(ssr, rep["ssr"])
    # idempotence: solved sketches exit immediately with zero factorizations
    x2, rep2 = topo.batch_solve(v2, p)
    assert np.array_equal(x2, x) and np.all(rep2["factorizations"] == 0) and np.all(rep2["exit_reason"] == 0)
    # sharding: two halves solved separately == the whole
    xa, ra = topo.batch_solve(v[: n // 2], p[: n // 2])
    xb, rb = topo.batch_solve(v[n // 2:], p[n // 2:])
    assert np.array_equal(np.vstack([xa, xb]), x)
    assert np.array_equal(np.concatenate([ra["trace_hash"], rb["trace_hash"]]), rep["trace_hash"])


def test_tile_variants_agree():
    import os
    w = wl.cad_mix(1024)
    v, p, scale = w.prepare()
    outs = []
    for tile in ("1", "2", "4", "8", "16", "32"):
        os.environ["FK_TILE"] = tile
        topo = fk.Topology.from_arrays(w.n_vars, w.kind, w.idx, w.free_vars, w.rows)
        assert topo.info["tile"] == int(tile)
        outs.append(topo.batch_solve(v, p))
    os.environ.pop("FK_TILE")
    for x, rep in outs[1:]:
        assert np.array_equal(x, outs[0][0]) and np.array_equal(rep, outs[0][1])


def test_cta_path_hinged64(oracle):
    # 514 free variables, ~50 KB of shared state: one CTA per sketch (path 1)
    w = wl.hinged_triangles(128, n_sketches=3)
    v, p, scale = w.prepare()
    topo = fk.Topology.from_arrays(w.n_vars, w.kind, w.idx, w.free_vars, w.rows)
    assert topo.info["path"] == 1 and topo.info["tile"] == 256
    xg, rg = topo.batch_solve(v, p)
    op, keep = oracle.make_problem(v[0], w.kind, w.idx, p[0], w.free_vars, w.rows)
    xo, ro, _ = oracle.lm_solve_batch_uniform(op, v, p)
    _same_reports(rg, ro)
    assert _rel(xg, xo) <= REL


def test_nan_sketch_hits_the_guard(oracle):
    # coincident points under a distance constraint: 1/0 -> NaN; the reference would spin forever
    kind, idx = [1], [[0, 2, 0, 0]]
    vars_ = np.array([1., 1., 1., 1.])
    fp, keep = fk.make_problem(vars_, kind, idx, [1.0], [0, 1, 2, 3], [0])
    x, rep = fk.lm_solve(fp, vars_)
    op, okeep = oracle.make_problem(vars_, kind, idx, [1.0], [0, 1, 2, 3], [0])
    xo, ro, _ = oracle.lm_solve(op, vars_)
    assert rep["exit_reason"] == 4 == ro["exit_reason"]
    assert rep["factorizations"] == ro["factorizations"] and rep["trace_hash"] == ro["trace_hash"]
    assert np.array_equal(x, vars_)


def test_mixed_topology_batch(oracle):
    """fk_lm_solve_batch groups by topology: all reference scenarios in one call."""
    probs, x0s, refs, keeps = [], [], [], []
    for name in sorted(sc.ALL):
        b = sc.ALL[name](oracle.System)
        for prob, scale, keep in b["s"].prepare():
            fp, fkeep = fk.make_problem(*keep)
            probs.append(fp); keeps.append(fkeep); x0s.append(keep[0][keep[4]])
            refs.append(oracle.lm_solve(prob, keep[0][keep[4]]))
    xs, reps = fk.lm_solve_batch(probs, x0s)
    for x, rep, (xo, ro, trace) in zip(xs, reps, refs):
        assert rep["trace_hash"] == ro["trace_hash"] and rep["exit_reason"] == ro["exit_reason"]
        assert _rel(x, xo) <= REL
