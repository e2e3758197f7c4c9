"""The oracle's fast QR mode (oracle.qr_fast: Qr::factorize without the reference's per-column O(m) scratch fill,
solvi/src/decomposition/sparse/qr.rs:287) must not change a single bit.  It exists only so that the oracle can
reach BASELINE config 3 for the golden fixtures (tests/golden/make_large_system_goldens.py); the slow mode stays
the default because its cost IS the reference's cost.  Checked on every kind of input the slow mode reaches."""
import json
import os

import numpy as np
import pytest

import scenarios as sc
from fiksi_b200 import workloads as wl
from large_cases import X_FULL_MAX

HERE = os.path.dirname(os.path.abspath(__file__))


def _both(oracle, fn):
    with oracle.qr_fast(False):
        slow = fn()
    with oracle.qr_fast(True):
        fast = fn()
    return slow, fast


def test_qr_kats_identical_in_both_modes(oracle):
    """R values and solutions of random augmented systems, natural and COLAMD ordering, repeated factorisations of
    one symbolic object (the scratch vector carries over between them)."""
    rng = np.random.default_rng(3)
    for trial in range(25):
        m, n = int(rng.integers(4, 60)), int(rng.integers(2, 30))
        dense = rng.normal(size=(m, n)) * (rng.random(size=(m, n)) < 0.25)
        a = np.vstack([dense, np.diag(rng.uniform(0.1, 1.0, size=n))])
        rows, cols = np.nonzero(a)
        _shape, colptr, rowidx, vals = oracle.from_triplets(m + n, n, rows, cols, a[rows, cols])
        for ordering in ("natural", "colamd"):
            def run():
                s = oracle.Symbolic(m + n, n, colptr, rowidx, ordering)
                out = []
                for rep in range(3):
                    s.factorize(vals * (1.0 + rep))
                    b = rng2.normal(size=m + n)
                    out.append((s.r_values().copy(), s.solve(b)))
                return out
            rng2 = np.random.default_rng(trial)
            slow = None
            with oracle.qr_fast(False):
                slow = run()
            rng2 = np.random.default_rng(trial)
            with oracle.qr_fast(True):
                fast = run()
            for (rs, (oks, xs)), (rf, (okf, xf)) in zip(slow, fast):
                assert oks == okf and np.array_equal(rs, rf, equal_nan=True) and np.array_equal(xs, xf, equal_nan=True)


@pytest.mark.parametrize("name", sorted(sc.ALL))
def test_reference_scenarios_identical_in_both_modes(oracle, name):
    b = sc.ALL[name](oracle.System)
    for prob, scale, keep in b["s"].prepare(perturb=True):
        x0 = keep[0][keep[4]]
        (xs, rs, ts), (xf, rf, tf) = _both(oracle, lambda: oracle.lm_solve(prob, x0))
        assert ts == tf and np.array_equal(xs, xf, equal_nan=True)
        assert {k: v for k, v in rs.items() if k != "ssr"} == {k: v for k, v in rf.items() if k != "ssr"}
        assert rs["ssr"] == rf["ssr"] or (rs["ssr"] != rs["ssr"] and rf["ssr"] != rf["ssr"])


@pytest.mark.parametrize("maker", [lambda: wl.lattice(30, 20), lambda: wl.lattice(48, 40), lambda: wl.truss(1), lambda: wl.cad_mix(1),
                                   lambda: wl.hinged_triangles(64)])
def test_workloads_identical_in_both_modes(oracle, maker):
    w = maker()
    v, p, scale = w.prepare()
    op, keep = oracle.make_problem(v[0], w.kind, w.idx, p[0], w.free_vars, w.rows)
    x0 = v[0][w.free_vars]
    (xs, rs, ts), (xf, rf, tf) = _both(oracle, lambda: oracle.lm_solve(op, x0))
    assert ts == tf and rs == rf and np.array_equal(xs, xf)


def test_golden_fixtures_are_consistent():
    """Every committed large-system golden has its coordinate file, the sizes agree and the generator is committed."""
    g = os.path.join(HERE, "golden")
    assert os.path.exists(os.path.join(g, "make_large_system_goldens.py"))
    metas = [f for f in os.listdir(g) if f.startswith("large_") and f.endswith(".json")]
    assert metas
    for f in metas:
        meta = json.load(open(os.path.join(g, f)))
        x = np.load(os.path.join(g, f[:-5] + "_x.npy"))
        if "x_sample" in meta:
            assert meta["n_free"] > X_FULL_MAX and x.shape == (meta["x_sample"]["size"],)
            assert np.max(np.abs(x)) <= float.fromhex(meta["x_sample"]["max_abs"])
        else:
            assert x.shape == (meta["n_free"],)
        assert x.dtype == np.float64 and np.all(np.isfinite(x))
        assert os.path.getsize(os.path.join(g, f[:-5] + "_x.npy")) < 1 << 20
        assert len(meta["trace"]) == meta["report"]["factorizations"]
