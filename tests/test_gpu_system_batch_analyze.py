"""fk_system_batch_analyze / fk_system_batch_residuals (System.batch_analyze / System.batch_residuals): System::analyze and
calculate_residual over n variants of one drawing in one call.  Every variant must equal the per-variant loop (set the
variant's numbers, System.analyze() / System.residuals(), restore) bit for bit; argument refusals are host logic and run
without a GPU."""
import ctypes as C
import os
import subprocess
import sys
import zlib

import numpy as np
import pytest

import scenarios as sc
import fiksi_b200 as fk
from fiksi_b200 import workloads as wl
from fiksi_b200._lib import lib, ptr

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
_PARAM_TAGS = (1, 2, 4, 7)  # constraints with a parameter: distances and angles


def _recording(S):
    """S whose constraint calls record (tag, parameter) in construction order, for fk.System and oracle.System alike."""
    methods = {"point_point_coincidence": 0, "point_point_distance": 1, "point_point_point_angle": 2, "point_line_incidence": 3,
               "point_line_distance": 4, "point_circle_incidence": 5, "segment_segment_length_equality": 6,
               "line_line_angle": 7, "line_line_parallelism": 8, "line_line_perpendicularity": 9, "line_circle_tangency": 10}

    class R(S):
        def __init__(self):
            super().__init__()
            self.tags, self.params = [], []

    def wrap(name, tag):
        base = getattr(S, name)

        def f(self, *args):
            self.tags.append(tag)
            self.params.append(float(args[-1]) if tag in _PARAM_TAGS else 0.0)
            return base(self, *args)
        return f
    for name, tag in methods.items():
        setattr(R, name, wrap(name, tag))
    return R


FkRec = _recording(fk.System)


def _build(builder, S=FkRec):
    b = builder(S)
    b["s"].point_vars = [b["s"].element_variable(p) for p in b.get("points", [])]
    return b["s"]


def _add_ppd(s, w):
    raw = w.raw_vars[0]
    pts = [s.add_point(float(raw[2 * i]), float(raw[2 * i + 1])) for i in range(len(raw) // 2)]
    for e in range(len(w.kind)):
        s.point_point_distance(pts[int(w.idx[e][0]) // 2], pts[int(w.idx[e][1]) // 2], float(w.raw_param[0][e]))
    return pts


def drawing_a(S=FkRec):
    """16 hinged chains of 4 triangles + 4 circle_triangle_line + a 20-point truss: 372 variables, beyond the warp kernel."""
    s = S()
    for _ in range(16):
        sc.hinged_triangles_bench(lambda: s, 4)
    for _ in range(4):
        sc.circle_triangle_line(lambda: s)
    _add_ppd(s, wl.truss(1, 20))
    return s


def drawing_b(S=FkRec):
    """A 30x20 lattice + 8 triangles: residuals of System.residuals() run on the global sparse path (fk_topology_eval)."""
    s = S()
    _add_ppd(s, wl.lattice(30, 20))
    for _ in range(8):
        sc.single_triangle(lambda: s)
    return s


def _variants(s, n, seed, specials=True):
    """n variable / parameter rows with seeded relative noise of 1e-3 on the variables and the distance / angle parameters.
    With `specials`: variant 1 a NaN variable, 2 an infinite variable, 3 a NaN parameter, 4 the first three points collinear
    (the rank drops), 5 the first two points coincident (NaN gradients)."""
    rng = np.random.default_rng(seed)
    v0 = s.variables.copy()
    p0 = np.array(s.params, dtype=np.float64)
    vars_ = v0[None, :] * (1.0 + 1e-3 * rng.standard_normal((n, len(v0))))
    noisy = np.array([t in _PARAM_TAGS for t in s.tags], dtype=bool)
    params = np.tile(p0, (n, 1))
    if len(p0):
        params[:, noisy] *= 1.0 + 1e-3 * rng.standard_normal((n, int(noisy.sum())))
    pv = getattr(s, "point_vars", [])
    if specials and n > 5:
        vars_[1, len(v0) // 2] = np.nan
        vars_[2, 0] = np.inf
        params[3, 0] = np.nan
        if len(pv) >= 3:
            a, b, c = pv[:3]
            vars_[4, c:c + 2] = 2.0 * vars_[4, b:b + 2] - vars_[4, a:a + 2]
        if len(pv) >= 2:
            vars_[5, pv[1]:pv[1] + 2] = vars_[5, pv[0]:pv[0] + 2]
    return vars_, params


def _loop(s, vars_, params, what=("analyze", "residuals")):
    """The per-variant reference: this system's numbers set to each variant's, then System.analyze() / residuals()."""
    v0, p0 = s.variables.copy(), list(s.params)
    an, res = [], []
    for k in range(len(vars_)):
        for i, x in enumerate(vars_[k]):
            s.set_variable(i, float(x))
        for c, x in enumerate(params[k]):
            s.set_parameter(c, float(x))
        if "analyze" in what:
            an.append(s.analyze())
        if "residuals" in what:
            res.append(s.residuals())
    for i, x in enumerate(v0):
        s.set_variable(i, float(x))
    for c, x in enumerate(p0):
        s.set_parameter(c, float(x))
    return an, np.array(res).reshape(len(res), s.num_constraints())


def _lists(dep):
    return [np.repeat(np.arange(dep.shape[1]), dep[v]).tolist() for v in range(len(dep))]


def _same(a, b):
    return np.array_equal(a, b, equal_nan=True)


# ---- host only: argument refusals --------------------------------------------------------------------------------------
def test_null_arguments_and_zero_variants():
    s = _build(sc.two_connected_components)
    assert lib().fk_system_batch_analyze(None, 2, None, None, None, 1) == -1
    assert lib().fk_system_batch_residuals(None, 2, None, None, None, 1) == -1
    assert lib().fk_system_batch_analyze(s._h, 2, None, None, None, 1) == -1
    assert lib().fk_system_batch_residuals(s._h, 2, None, None, None, 1) == -1
    assert lib().fk_system_batch_analyze(s._h, 0, None, None, None, 1) == 0
    assert lib().fk_system_batch_residuals(s._h, 0, None, None, None, 1) == 0
    assert s.batch_analyze(n=0).shape == (0, 2) and s.batch_residuals(n=0).shape == (0, 2)
    with pytest.raises(ValueError):
        s.batch_analyze(np.zeros((2, 8)), np.zeros((3, 2)))


# ---- on the device -----------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("name", sorted(sc.ALL))
def test_every_scenario_equals_the_per_variant_loop(oracle, name):
    s = _build(sc.ALL[name])
    vars_, params = _variants(s, 32, seed=zlib.crc32(name.encode()))
    tmpl_v, tmpl_r = s.variables.copy(), s.residuals()
    dep = s.batch_analyze(vars_, params)
    res = s.batch_residuals(vars_, params)
    assert dep.dtype == np.uint8 and dep.shape == res.shape == (32, s.num_constraints())
    assert np.array_equal(s.variables, tmpl_v) and _same(s.residuals(), tmpl_r)  # s is not modified
    ref_an, ref_res = _loop(s, vars_, params)
    assert _lists(dep) == ref_an, name
    assert _same(res, ref_res), (name, np.argwhere(~((res == ref_res) | (np.isnan(res) & np.isnan(ref_res))))[:5])
    for k in (0, 4, 5, 17, 31):  # the oracle: analyze exactly, residuals within the facade's tolerance
        so = _build(sc.ALL[name], _recording(oracle.System))
        for i, x in enumerate(vars_[k]):
            so.set_variable(i, float(x))
        for c, x in enumerate(params[k]):
            so.set_parameter(c, float(x))
        assert so.analyze() == ref_an[k], (name, k)
        ro = np.array([so.calculate_residual(c) for c in range(s.num_constraints())])
        assert np.array_equal(np.isnan(ro), np.isnan(res[k])), (name, k)
        fin = ~np.isnan(ro)
        scale = max(1.0, float(np.max(np.abs(vars_[k])))) ** 2
        assert np.all(np.abs(ro[fin] - res[k][fin]) <= 1e-7 * scale), (name, k, ro, res[k])


@pytest.mark.gpu
def test_over_constrained_scenarios_flag_the_reference_constraints():
    s = _build(sc.overconstrained)  # tests/basic.rs:90-112: the last distance over-constrains the frame
    assert _lists(s.batch_analyze(n=3)) == [[5]] * 3
    vars_, params = _variants(s, 8, seed=1, specials=False)
    assert _lists(s.batch_analyze(vars_, params)) == [[5]] * 8


@pytest.mark.gpu
def test_three_analyze_kernels_agree_on_a_small_drawing(monkeypatch):
    s = _build(lambda S: sc.hinged_triangles_bench(S, 16))
    vars_, params = _variants(s, 40, seed=21)
    got = {}
    for kernel in ("warp", "cta", "group"):
        monkeypatch.setenv("FK_ANALYZE_KERNEL", kernel)
        got[kernel] = s.batch_analyze(vars_, params)
    monkeypatch.delenv("FK_ANALYZE_KERNEL")
    assert np.array_equal(got["warp"], got["cta"]) and np.array_equal(got["warp"], got["group"])
    assert _lists(got["warp"]) == _loop(s, vars_, params, ("analyze",))[0]


@pytest.mark.gpu
def test_drawing_beyond_shared_memory_on_cta_and_group_kernels(monkeypatch):
    s = drawing_a()
    assert len(s.variables) == 372
    vars_, params = _variants(s, 2048, seed=0xA)
    big = s.batch_analyze(vars_, params)  # a batch that fills the device: one CTA per sketch
    small = s.batch_analyze(vars_[:3], params[:3])  # a few sketches: groups of CTAs
    assert np.array_equal(small, big[:3])
    for kernel in ("cta", "group"):
        monkeypatch.setenv("FK_ANALYZE_KERNEL", kernel)
        assert np.array_equal(s.batch_analyze(vars_[:64], params[:64]), big[:64]), kernel
    monkeypatch.delenv("FK_ANALYZE_KERNEL")
    sample = [0, 1, 2, 3, 4, 5, 1000, 2047]
    ref_an, ref_res = _loop(s, vars_[sample], params[sample])
    assert _lists(big[sample]) == ref_an
    assert _same(s.batch_residuals(vars_, params)[sample], ref_res)


def _drawing_b_path():
    """Path of the whole-drawing topology fk_system_residuals builds for drawing (b) (every variable free, every row): the
    lattice's distances, then per triangle the distances (0, 1), (0, 2), (1, 2) of its three points."""
    w = wl.lattice(30, 20)
    kind, idx = list(w.kind), [list(r) for r in w.idx]
    base = len(w.raw_vars[0])
    for k in range(8):
        v = base + 6 * k
        for a, b in ((0, 1), (0, 2), (1, 2)):
            kind.append(1)
            idx.append([v + 2 * a, v + 2 * b, 0, 0])
    n_vars = base + 48
    return fk.Topology.from_arrays(n_vars, kind, idx, np.arange(n_vars), np.arange(len(kind))).info["path"]


def test_drawing_b_residuals_run_on_the_global_sparse_path():
    # what test_drawing_on_the_global_sparse_path compares against: fk_topology_eval, not the K2 evaluation
    assert _drawing_b_path() == 2


@pytest.mark.gpu
def test_drawing_on_the_global_sparse_path():
    s = drawing_b()  # System.residuals() runs fk_topology_eval on it (test_drawing_b_residuals_run_on_the_global_sparse_path)
    vars_, params = _variants(s, 12, seed=0xB)
    res = s.batch_residuals(vars_, params)
    ref_res = _loop(s, vars_, params, ("residuals",))[1]  # System.residuals() runs fk_topology_eval here
    assert _same(res, ref_res)
    # every kind with an angle, a tangency or an incidence, beside the lattice: fk_topology_eval's bits too
    t = FkRec()
    _add_ppd(t, wl.lattice(30, 20))
    for builder in (sc.circle_triangle_line, sc.connected_triangles, sc.lib_doc_example, sc.distance_and_angle,
                    sc.triangle_inscribed_circle, sc.coincident_points):
        builder(lambda: t)
    tv, tp = _variants(t, 6, seed=0xC, specials=False)
    assert _same(t.batch_residuals(tv, tp), _loop(t, tv, tp, ("residuals",))[1])
    dep = s.batch_analyze(vars_[[0, 4, 7]], params[[0, 4, 7]])
    assert _lists(dep) == _loop(s, vars_[[0, 4, 7]], params[[0, 4, 7]], ("analyze",))[0]


@pytest.mark.gpu
def test_variants_are_independent_of_each_other_and_of_the_batch():
    s = _build(sc.ALL["circle_triangle_line"])
    vars_, params = _variants(s, 24, seed=4)
    dep, res = s.batch_analyze(vars_, params), s.batch_residuals(vars_, params)
    clean_v, clean_p = _variants(s, 24, seed=4, specials=False)
    cd, cr = s.batch_analyze(clean_v, clean_p), s.batch_residuals(clean_v, clean_p)
    keep = [k for k in range(24) if k not in (1, 2, 3, 4, 5)]
    assert np.array_equal(dep[keep], cd[keep]) and _same(res[keep], cr[keep])  # NaN / inf stay in their variant
    perm = np.random.default_rng(0).permutation(24)
    assert np.array_equal(s.batch_analyze(vars_[perm], params[perm]), dep[perm])
    assert _same(s.batch_residuals(vars_[perm], params[perm]), res[perm])
    assert np.array_equal(s.batch_analyze(vars_[7:9], params[7:9]), dep[7:9])
    assert _same(s.batch_residuals(vars_[7:8], params[7:8]), res[7:8])


_CHUNK_SCRIPT = """
import sys, numpy as np
sys.path.insert(0, {root!r}); sys.path.insert(0, {tests!r})
import test_gpu_system_batch_analyze as t, scenarios as sc
s = t._build(sc.ALL['hinged_triangles_bench_4'])
v, p = t._variants(s, 50, seed=5)
np.savez({path!r}, dep=s.batch_analyze(v, p), res=s.batch_residuals(v, p))
"""


@pytest.mark.gpu
def test_chunks_and_devices_do_not_change_results(tmp_path):
    s = _build(sc.ALL["hinged_triangles_bench_4"])
    vars_, params = _variants(s, 50, seed=5)
    dep, res = s.batch_analyze(vars_, params), s.batch_residuals(vars_, params)
    path = str(tmp_path / "chunked.npz")
    script = _CHUNK_SCRIPT.format(root=ROOT, tests=os.path.join(ROOT, "tests"), path=path)
    env = dict(os.environ, FK_SYSTEM_BATCH_CHUNK="3")
    subprocess.check_call([sys.executable, "-c", script], env=env, cwd=str(tmp_path))
    got = np.load(path)
    assert np.array_equal(got["dep"], dep) and _same(got["res"], res)
    if fk.device_count() < 2:
        pytest.skip("n_gpus=2 needs two devices")
    assert np.array_equal(s.batch_analyze(vars_, params, n_gpus=2), dep)
    assert _same(s.batch_residuals(vars_, params, n_gpus=2), res)


@pytest.mark.gpu
def test_template_rows_and_the_plan():
    s = _build(sc.ALL["lib_doc_example"])
    vars_, params = _variants(s, 3, seed=2, specials=False)
    tmpl_v, tmpl_p = s.variables.copy(), np.array(s.params)
    for v, p in ((None, None), (vars_, None), (None, params)):
        rv = np.tile(tmpl_v, (3, 1)) if v is None else v
        rp = np.tile(tmpl_p, (3, 1)) if p is None else p
        ref_an, ref_res = _loop(s, rv, rp)
        assert _lists(s.batch_analyze(v, p, n=3)) == ref_an
        assert _same(s.batch_residuals(v, p, n=3), ref_res)
    # new values keep the plan and show in the template rows of the next call
    s.set_variable(2, 0.25)
    s.set_parameter(0, 4.0)
    assert _same(s.batch_residuals(n=2), np.tile(s.residuals(), (2, 1)))
    assert _lists(s.batch_analyze(n=1)) == [s.analyze()]
    # a structural edit drops the plan: the new constraint shows
    p = s.add_point(0.3, 0.7)
    s.point_point_distance(p, 0, 1.0)
    s.point_point_distance(p, 0, 1.0)  # the same row twice: dependent
    res = s.batch_residuals(n=2)
    assert res.shape == (2, 5) and _same(res[0], s.residuals())
    dep = s.batch_analyze(n=1)
    assert _lists(dep) == [s.analyze()] and dep[0, 4] == 1


@pytest.mark.gpu
def test_diagnosing_a_solved_sweep():
    s = _build(sc.ALL["circle_triangle_line"])
    vars_, params = _variants(s, 16, seed=8, specials=False)
    vars_[3] = vars_[3] * 1e-9  # a degenerate start
    solved, _ = s.batch_solve(vars_, params)
    dep, res = s.batch_analyze(solved, params), s.batch_residuals(solved, params)
    ref_an, ref_res = _loop(s, solved, params)
    assert _lists(dep) == ref_an
    assert _same(res, ref_res)


def _big_lattice():
    s = FkRec()
    _add_ppd(s, wl.lattice(120, 112))
    return s


@pytest.mark.gpu
def test_analyze_size_limit():
    s = _big_lattice()
    nv, nc = len(s.variables), s.num_constraints()
    assert nv == 26880 > 26624
    out = np.full((2, nc), 7, np.uint8)
    assert lib().fk_system_batch_analyze(s._h, 2, None, None, ptr(out, C.c_uint8), 1) == -5
    assert "26624" in lib().fk_last_error().decode()
    assert np.all(out == 7)
    res = s.batch_residuals(n=2)  # every size: no topology, no front limit
    assert _same(res[0], s.residuals()) and _same(res[1], res[0])
