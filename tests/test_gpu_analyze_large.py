"""System::analyze beyond shared memory: fk_batch_analyze with the matrix in global memory, one CTA per sketch or a
cooperative group of CTAs per sketch.  Every comparison is np.array_equal of the "independent" flags against the oracle
(the CPU restatement of analyze/numerical/mod.rs), its goldens, or another kernel: nothing is toleranced."""
import contextlib
import json
import math
import os

import numpy as np
import pytest

import fiksi_b200 as fk
from fiksi_b200 import workloads as wl

pytestmark = pytest.mark.gpu
GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


@contextlib.contextmanager
def forced(kernel):
    """FK_ANALYZE_KERNEL=kernel for the calls inside (the library reads it on every call)."""
    prev = os.environ.get("FK_ANALYZE_KERNEL")
    os.environ["FK_ANALYZE_KERNEL"] = kernel
    try:
        yield
    finally:
        if prev is None:
            del os.environ["FK_ANALYZE_KERNEL"]
        else:
            os.environ["FK_ANALYZE_KERNEL"] = prev


def topology(w):
    return fk.Topology.from_arrays(w.n_vars, w.kind, w.idx, np.arange(w.n_vars), np.arange(len(w.kind)))


def oracle_flags(oracle, w, sketches=None):
    sketches = range(w.n) if sketches is None else sketches
    return np.array([oracle.analyze(w.raw_vars[s], w.kind, w.idx, w.raw_param[s]) for s in sketches])


def tile(parts, name):
    """One system of several workloads' first sketches side by side: variable indices offset, expressions in order."""
    kind, idx, raw, par = [], [], [], []
    off = 0
    for w in parts:
        kind.append(w.kind)
        idx.append(w.idx.astype(np.int64) + off)
        raw.append(w.raw_vars[:1])
        par.append(w.raw_param[:1])
        off += w.n_vars
    kind = np.concatenate(kind)
    return wl.Workload(name, kind, np.vstack(idx), np.arange(off), np.arange(len(kind)), np.hstack(raw), np.hstack(par))


def cad_drawing(copies):
    """Disjoint circle_triangle_line copies (kinds 1, 2, 3, 7, 10), each with its own noise."""
    w = wl.cad_mix(copies)
    parts = [wl.Workload("c", w.kind, w.idx, np.arange(11), np.arange(8), w.raw_vars[c:c + 1], w.raw_param[c:c + 1]) for c in range(copies)]
    return tile(parts, f"cad_mix_x{copies}")


def stress_drawing(copies):
    """BASELINE config 5's families (all but the NaN one, which has its own test) tiled into one system."""
    fams = [w for name, w in wl.stress_families(copies) if name != "nan_coincident_points"]
    parts = [wl.Workload("s", w.kind, w.idx, np.arange(w.n_vars), np.arange(len(w.kind)), w.raw_vars[c:c + 1], w.raw_param[c:c + 1])
             for c in range(copies) for w in fams]
    return tile(parts, f"stress_x{copies}")


def with_free_point(w):
    """The workload plus one point no expression mentions: an all-zero column."""
    raw = np.hstack([w.raw_vars, np.full((w.n, 2), 0.5)])
    return wl.Workload(w.name + "+free", w.kind, w.idx, np.arange(raw.shape[1]), w.rows, raw, w.raw_param)


def chain_in_cloud(n_sketches, n_points=6000, links=200, seed=7):
    """A chain of `links` distance constraints among the first points of a cloud of n_points: m = 200 rows, n = 12,000
    columns, a 19.2 MB matrix per sketch."""
    rng = np.random.default_rng(seed)
    base = rng.uniform(-10, 10, size=(1, 2 * n_points))
    raw = base + 0.01 * rng.uniform(-1, 1, size=(n_sketches, 2 * n_points))
    kind = np.full(links, 1, np.uint8)
    idx = np.zeros((links, 4), np.uint32)
    idx[:, 0] = 2 * np.arange(links)
    idx[:, 1] = 2 * np.arange(1, links + 1)
    par = np.tile(np.linspace(1.0, 3.0, links), (n_sketches, 1))
    return wl.Workload("chain_cloud", kind, idx, np.arange(2 * n_points), np.arange(links), raw, par)


def lattice_batch(nx, ny, n):
    return wl.lattice(nx, ny, n_sketches=n)


# ---- 1. oracle parity on the global-memory kernels ---------------------------------------------------------------------
PARITY = {
    "lattice12x10": lambda: lattice_batch(12, 10, 3),        # m > n
    "lattice16x12": lambda: lattice_batch(16, 12, 3),
    "lattice20x15": lambda: lattice_batch(20, 15, 3),
    "lattice24x20": lambda: lattice_batch(24, 20, 2),
    "hinged64": lambda: wl.hinged_triangles(64),             # m < n
    "truss300": lambda: wl.truss(2, n_points=300),           # m = n - 3
    "cad_drawing40": lambda: cad_drawing(40),
    "stress_drawing": lambda: stress_drawing(12),
    "lattice12x10_free_point": lambda: with_free_point(lattice_batch(12, 10, 2)),
    "two_trusses": lambda: tile([wl.truss(1, n_points=101)] * 2, "two_trusses"),  # m = n - 6
}


@pytest.mark.parametrize("case", sorted(PARITY))
def test_global_kernels_match_oracle(oracle, case):
    w = PARITY[case]()
    topo = topology(w)
    kernel = topo.analyze_kernel(w.n)
    assert kernel != "warp", case
    ref = oracle_flags(oracle, w)
    assert np.array_equal(topo.batch_analyze(w.raw_vars, w.raw_param), ref), (case, kernel)
    other = "cta" if kernel == "group" else "group"
    with forced(other):
        assert topo.analyze_kernel(w.n) == other
        assert np.array_equal(topo.batch_analyze(w.raw_vars, w.raw_param), ref), (case, other)


def test_square_system_matches_oracle(oracle):
    """m == n: the 300-point truss (597 rows, 600 columns) with its first three edges repeated at other lengths."""
    w = wl.truss(2, n_points=300)
    kind = np.concatenate([w.kind, w.kind[:3]])
    idx = np.vstack([w.idx, w.idx[:3]])
    par = np.hstack([w.raw_param, w.raw_param[:, :3] * 1.01])
    sq = wl.Workload("truss300_square", kind, idx, np.arange(w.n_vars), np.arange(len(kind)), w.raw_vars, par)
    assert len(sq.kind) == sq.n_vars
    topo = topology(sq)
    assert topo.analyze_kernel(sq.n) != "warp"
    got = topo.batch_analyze(sq.raw_vars, sq.raw_param)
    assert np.array_equal(got, oracle_flags(oracle, sq))
    assert not got[:, -3:].any()  # repeated edges are dependent


# ---- 2. fk_system_analyze on large systems ---------------------------------------------------------------------------
def _triangles(System, count):
    s = System()
    for k in range(count):
        a = s.add_point(3.0 * k, 0.0)
        b = s.add_point(3.0 * k + 1.1, 0.05 * k)
        c = s.add_point(3.0 * k + 0.4, 1.0 + 0.01 * k)
        s.point_point_distance(a, b, 1.0)
        s.point_point_distance(b, c, 1.2)
        s.point_point_distance(c, a, 1.1)
        if k % 7 == 3:
            s.point_point_distance(a, b, 1.5)  # contradictory duplicate
    return s


def _every_tag(System, copies):
    s = System()
    for k in range(copies):
        x = 10.0 * k
        p = [s.add_point(x + 0.0, 0.0), s.add_point(x + 2.0, 0.1), s.add_point(x + 0.2, 2.1), s.add_point(x + 2.2, 2.0),
             s.add_point(x + 1.0, 1.0), s.add_point(x + 3.0, 0.5)]
        r = s.add_length(0.7 + 0.01 * k)
        l1, l2, l3 = s.add_line(p[0], p[1]), s.add_line(p[2], p[3]), s.add_line(p[0], p[2])
        circ = s.add_circle(p[4], r)
        s.point_point_coincidence(p[5], p[1])
        s.point_point_distance(p[0], p[1], 2.0)
        s.point_point_point_angle(p[0], p[1], p[2], 1.2)
        s.point_line_incidence(p[5], l1)
        s.point_line_distance(p[4], l1, 1.0)
        s.point_circle_incidence(p[3], circ)
        s.segment_segment_length_equality(p[0], p[1], p[2], p[3])
        s.line_line_angle(l1, l3, math.pi / 2)
        s.line_line_parallelism(l1, l2)
        s.line_line_perpendicularity(l1, l3)
        s.line_circle_tangency(l2, circ)
        s.line_line_parallelism(l1, l2)            # duplicated
        s.point_point_distance(p[0], p[1], 2.5)    # contradictory
        if k == 0:
            s.fix(p[0])
    return s


@pytest.mark.parametrize("build", [lambda S: _triangles(S, 50), lambda S: _every_tag(S, 16)], ids=["triangles50", "every_tag16"])
def test_system_analyze_large(oracle, build):
    import fiksi_b200.system as fsys
    got, ref = build(fsys.System), build(oracle.System)
    assert got.variables.shape[0] * got.num_constraints() > 30000  # beyond the warp kernel
    assert got.analyze() == ref.analyze()
    assert len(ref.analyze()) > 0


# ---- 3. the kernels agree ----------------------------------------------------------------------------------------------
def _stress_topologies():
    out = [(name, w) for name, w in wl.stress_families(64)]
    out += [("truss257", wl.truss(257)), ("cad_mix515", wl.cad_mix(515))]
    return out


def test_warp_cta_group_agree_where_the_warp_kernel_fits():
    for name, w in _stress_topologies():
        topo = topology(w)
        assert topo.analyze_kernel(w.n) == "warp", name
        runs = {}
        for k in ("warp", "cta", "group"):
            with forced(k):
                assert topo.analyze_kernel(w.n) == k
                runs[k] = topo.batch_analyze(w.raw_vars, w.raw_param)
        assert np.array_equal(runs["warp"], runs["cta"]) and np.array_equal(runs["warp"], runs["group"]), name


def test_kernels_agree_across_the_shared_memory_boundary(oracle):
    seen = set()
    for k in range(40, 52):
        w = wl.hinged_triangles(k, n_sketches=2)
        w.raw_vars = w.raw_vars + 0.01 * np.sin(np.arange(w.raw_vars.size)).reshape(w.raw_vars.shape)
        topo = topology(w)
        auto = topo.analyze_kernel(w.n)
        seen.add(auto)
        m, n = len(w.kind), w.n_vars
        assert (auto == "warp") == (m * n * 8 + (m + n) * 4 <= 200 * 1024), k
        ref = oracle_flags(oracle, w)
        for kern in ("warp", "cta", "group") if auto == "warp" else ("cta", "group"):
            with forced(kern):
                assert np.array_equal(topo.batch_analyze(w.raw_vars, w.raw_param), ref), (k, kern)
        if auto != "warp":
            with forced("warp"), pytest.raises(fk.FiksiError) as e:
                topo.batch_analyze(w.raw_vars, w.raw_param)
            assert e.value.code == -5
    assert "warp" in seen and len(seen) > 1


def test_cta_and_group_agree_on_large_cases():
    for w in (lattice_batch(24, 20, 3), lattice_batch(32, 32, 1), wl.hinged_triangles(64, n_sketches=5)):
        topo = topology(w)
        with forced("cta"):
            a = topo.batch_analyze(w.raw_vars, w.raw_param)
        with forced("group"):
            b = topo.batch_analyze(w.raw_vars, w.raw_param)
        assert np.array_equal(a, b), w.name


# ---- 4. batches ---------------------------------------------------------------------------------------------------------
def test_flags_do_not_depend_on_batch_size_or_composition():
    w = lattice_batch(12, 10, 700)  # 700 sketches: more than the resident CTAs, so the persistent loop goes round
    topo = topology(w)
    assert topo.analyze_kernel(700) == "cta" and topo.analyze_kernel(1) == "group"
    full = topo.batch_analyze(w.raw_vars, w.raw_param)
    again = topo.batch_analyze(w.raw_vars, w.raw_param)
    assert np.array_equal(full, again)
    for sel in (slice(0, 0), slice(5, 6), slice(0, 100), slice(17, 300, 3), slice(699, 700)):
        part = topo.batch_analyze(w.raw_vars[sel], w.raw_param[sel])
        assert part.shape[0] == len(range(700)[sel])
        assert np.array_equal(part, full[sel]), sel
    rev = topo.batch_analyze(w.raw_vars[::-1].copy(), w.raw_param[::-1].copy())
    assert np.array_equal(rev, full[::-1])
    with forced("group"):
        assert np.array_equal(topo.batch_analyze(w.raw_vars[:40], w.raw_param[:40]), full[:40])


def test_batch_sizes_against_oracle(oracle):
    w = lattice_batch(16, 12, 400)
    topo = topology(w)
    full = topo.batch_analyze(w.raw_vars, w.raw_param)
    picks = [0, 1, 147, 148, 299, 399]
    assert np.array_equal(full[picks], oracle_flags(oracle, w, picks))
    for n in (1, 100, 400):
        assert np.array_equal(topo.batch_analyze(w.raw_vars[:n], w.raw_param[:n]), full[:n]), n


def test_workspace_budget_caps_the_ctas(oracle):
    """19.2 MB per sketch: 4 GiB holds 223 workspaces, fewer than the CTAs the device keeps resident (two per SM), so
    300 sketches go through the persistent loop on a capped grid."""
    w = chain_in_cloud(300)
    topo = topology(w)
    assert topo.analyze_kernel(300) == "cta"
    got = topo.batch_analyze(w.raw_vars, w.raw_param)
    assert np.array_equal(got[[0, 299]], oracle_flags(oracle, w, [0, 299]))
    assert np.array_equal(topo.batch_analyze(w.raw_vars[150:152], w.raw_param[150:152]), got[150:152])


def test_nan_sketch_is_isolated(oracle):
    w = lattice_batch(12, 10, 6)
    bad = w.raw_vars.copy()
    bad[3, 2:4] = bad[3, 0:2]  # points 0 and 1 coincide: the distance gradient is 0/0
    topo = topology(w)
    clean = topo.batch_analyze(w.raw_vars, w.raw_param)
    for kern in ("cta", "group"):
        with forced(kern):
            got = topo.batch_analyze(bad, w.raw_param)
        assert np.array_equal(got[3], oracle.analyze(bad[3], w.kind, w.idx, w.raw_param[3])), kern
        keep = [0, 1, 2, 4, 5]
        assert np.array_equal(got[keep], clean[keep]), kern


# ---- 5. limits ----------------------------------------------------------------------------------------------------------
def test_config3_is_refused_before_allocation():
    w = wl.lattice(400, 250)
    topo = topology(w)
    with pytest.raises(fk.FiksiError) as e:
        topo.analyze_kernel(1)
    assert e.value.code == -5
    msg = str(e.value)
    for part in ("320001600256 bytes", "4294967296", "n_vars = 200000", "26624"):
        assert part in msg, msg
    with pytest.raises(fk.FiksiError) as e2:
        topo.batch_analyze(w.raw_vars, w.raw_param)
    assert e2.value.code == -5 and str(e2.value) == msg


def test_64x50_is_accepted():
    w = wl.lattice(64, 50)
    assert topology(w).analyze_kernel(1) == "group"


# ---- 6. large goldens ---------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("nx,ny", [(48, 40), (64, 50)])
def test_large_lattice_golden(nx, ny):
    from golden.make_analyze_goldens import input_hashes, unpack_flags
    with open(os.path.join(GOLDEN, f"analyze_lattice{nx}x{ny}.json")) as f:
        g = json.load(f)
    w = wl.lattice(nx, ny)
    assert input_hashes(w) == g["sha256"]
    topo = topology(w)
    assert topo.analyze_kernel(1) == "group"
    got = topo.batch_analyze(w.raw_vars, w.raw_param)[0]
    ref = unpack_flags(g["flags"], g["n_expr"])
    assert int(got.sum()) == g["independent"]
    assert np.array_equal(got, ref)
