"""Column pairs in the sketch kernels' tables (symbolic.cpp, build_sketch_tables): when L(:,k) = {k+1} u L(:,k+1), one
record eliminates columns k and k+1 in one LDLt step and one back-substitution step.  Every entry still receives the
same operations in the same order, so a topology built with pairs (the default) and the same topology built with
single-column records only (FK_SK_COLPAIR=0, read when the topology's tables are built) give bit-identical results,
in the solo kernel and in the warp-pair kernel alike, including rejected steps, non-positive and NaN pivots."""
import numpy as np
import pytest

import cad_drawings as cd
import fiksi_b200 as fk
from fiksi_b200 import api, workloads as wl

TOPOLOGIES = {
    "truss20": lambda n: wl.truss(n),
    "truss14": lambda n: wl.truss(n, n_points=14),
    "truss10": lambda n: wl.truss(n, n_points=10),
    "cad_mix": lambda n: wl.cad_mix(n),
    "hinged4": lambda n: wl.hinged_triangles(4, n),
    "cad4x4": lambda n: cd.workload(*cd.PATH0, n, seed=1, shared_vertices=False),  # every kind, fixed points
}
FIELDS = ("exit_reason", "outer_iters", "factorizations", "accepted", "trace_hash", "lambda", "ssr")


@pytest.fixture
def paired_and_single(monkeypatch):
    """Builds a workload's topology twice: with column pairs and with single-column records only."""
    def build(w):
        def topo():
            return fk.Topology.from_arrays(w.n_vars, w.kind, w.idx, w.free_vars, w.rows)
        monkeypatch.delenv("FK_SK_COLPAIR", raising=False)
        paired = topo()
        monkeypatch.setenv("FK_SK_COLPAIR", "0")
        single = topo()
        monkeypatch.delenv("FK_SK_COLPAIR")
        return paired, single
    return build


def _words(topo):
    return topo.sketch_kernel_info()["table_words"]


def _assert_same(a, b, what):
    (xa, ra), (xb, rb) = a, b
    for key in FIELDS:
        assert np.array_equal(ra[key], rb[key], equal_nan=True), (what, key)
    assert np.array_equal(xa, xb, equal_nan=True), what


@pytest.mark.parametrize("name", list(TOPOLOGIES))
def test_pairs_shrink_the_tables(name, paired_and_single):
    paired, single = paired_and_single(TOPOLOGIES[name](4))
    assert paired.sketch_kernel_info()["available"] and single.sketch_kernel_info()["available"]
    assert paired.sketch_kernel_info()["state_doubles"] == single.sketch_kernel_info()["state_doubles"]
    assert _words(paired) < _words(single)


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(TOPOLOGIES))
def test_pairs_are_bit_identical(name, paired_and_single):
    w = TOPOLOGIES[name](2048 + 17)
    v, p, _ = w.prepare()
    paired, single = paired_and_single(w)
    assert _words(paired) < _words(single)
    for kernel in ("sketch_solo", "sketch_pair"):
        with api.lm_kernel(kernel):
            _assert_same(paired.batch_solve(v, p), single.batch_solve(v, p), (name, kernel))


@pytest.mark.gpu
def test_pairs_are_bit_identical_on_stress_families(paired_and_single):
    paired_families = 0
    for name, w in wl.stress_families(n_each=512):
        v, p, _ = w.prepare(perturb=(name != "nan_coincident_points"))
        paired, single = paired_and_single(w)
        if not single.sketch_kernel_info()["available"]:
            continue
        paired_families += _words(paired) < _words(single)
        for kernel in ("sketch_solo", "sketch_pair"):
            with api.lm_kernel(kernel):
                _assert_same(paired.batch_solve(v, p), single.batch_solve(v, p), (name, kernel))
    assert paired_families >= 8
