"""fk_system_batch_solve / System.batch_solve: System::solve over n variants of one drawing in one call.  Every variant must
equal a per-variant System.solve on the same numbers (bit for bit where both run the same batched kernels); the plan
probe and the refusals are host logic and run without a GPU."""
import ctypes as C
import os
import subprocess
import sys
import zlib

import numpy as np
import pytest

import cad_drawings as cd
import scenarios as sc
import fiksi_b200 as fk
from fiksi_b200 import workloads as wl
from fiksi_b200._lib import FkReport, FkSolvingOptions, lib, ptr

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
_PARAM_TAGS = (1, 2, 4, 7)  # constraints with a parameter: distances and angles


class RecSystem(fk.System):
    """fk.System that remembers every constraint's tag and parameter (the template of the variants' parameter rows)."""

    def __init__(self):
        super().__init__()
        self.tags, self.params = [], []

    def _c(self, tag, elements, param=0.0):
        cid = super()._c(tag, elements, param)
        self.tags.append(tag)
        self.params.append(param)
        return cid


def _variants(s, n, seed, specials=True):
    """n variables / parameter rows: seeded relative noise of 1e-3 on the variables and on the parameters of parameterised
    constraints; with `specials`, variants 1-3 carry a NaN variable, an infinite variable and a NaN parameter."""
    rng = np.random.default_rng(seed)
    v0 = s.variables.copy()
    p0 = np.array(s.params, dtype=np.float64)
    vars_ = v0[None, :] * (1.0 + 1e-3 * rng.standard_normal((n, len(v0))))
    noisy = np.array([t in _PARAM_TAGS for t in s.tags], dtype=bool)
    params = np.tile(p0, (n, 1))
    if len(p0):
        params[:, noisy] *= 1.0 + 1e-3 * rng.standard_normal((n, int(noisy.sum())))
    if specials and n > 3 and len(v0):
        vars_[1, len(v0) // 2] = np.nan
        vars_[2, 0] = np.inf
        if len(p0):
            params[3, 0] = np.nan
    return vars_, params


def _loop(s, vars_, params, optimizer="lm", perturb=True):
    """The per-variant reference: this system's numbers set to each variant's, then System.solve."""
    v0 = s.variables.copy()
    p0 = list(s.params)
    outs, reps = [], []
    for k in range(len(vars_)):
        for i, x in enumerate(vars_[k]):
            s.set_variable(i, float(x))
        for c, x in enumerate(params[k]):
            s.set_parameter(c, float(x))
        s.solve(perturb=perturb, optimizer=optimizer)
        outs.append(s.variables.copy())
        reps.append(s._reports.copy())
    for i, x in enumerate(v0):
        s.set_variable(i, float(x))
    for c, x in enumerate(p0):
        s.set_parameter(c, float(x))
    return np.array(outs).reshape(len(vars_), len(v0)), np.array(reps).reshape(len(vars_), -1)


def _same_reports(a, b):
    for f in a.dtype.names:
        if a[f].dtype.kind == "f":
            assert np.array_equal(a[f], b[f], equal_nan=True), f
        else:
            assert np.array_equal(a[f], b[f]), f


def _build(builder):
    return builder(RecSystem)["s"]


def _add_ppd(s, w, k=0):
    """Workload w's sketch k (all point-point distances) appended to s as its own component."""
    raw = w.raw_vars[k]
    pts = [s.add_point(float(raw[2 * i]), float(raw[2 * i + 1])) for i in range(len(raw) // 2)]
    for e in range(len(w.kind)):
        s.point_point_distance(pts[int(w.idx[e][0]) // 2], pts[int(w.idx[e][1]) // 2], float(w.raw_param[k][e]))
    return pts


def _grouping_drawing():
    s = RecSystem()
    for _ in range(12):
        sc.single_triangle(lambda: s)
    sc.circle_triangle_line(lambda: s)
    _add_ppd(s, wl.truss(1, 20))
    return s


def _cad_drawing(S):
    """Three components: a mixed-kind CAD grid on the one-CTA-per-sketch path (path 1), a smaller one with shared vertices
    on the tile path and a single triangle."""
    s = S()
    cd.cad_grid(lambda: s, *cd.PATH1_LOW, seed=3)
    cd.cad_grid(lambda: s, *cd.PATH0, seed=4)
    sc.single_triangle(lambda: s)
    return s


def _lattice_drawing(nx, ny):
    s = RecSystem()
    _add_ppd(s, wl.lattice(nx, ny))
    sc.single_triangle(lambda: s)
    return s


# ---- host only: the plan and the refusals ----------------------------------------------------------------------------
def test_layout_groups_identical_components():
    s = _grouping_drawing()
    assert s.batch_layout() == (14, 3, [12, 1, 1])
    assert _build(sc.two_connected_components).batch_layout() == (2, 1, [2])
    quirk = _build(sc.stale_component_quirk)
    assert quirk.batch_layout()[0] == sum(1 for elements, _ in quirk.components() if elements)
    free = RecSystem()
    free.add_point(1.0, 2.0)
    assert free.batch_layout() == (0, 0, [])


def test_structural_edit_drops_the_plan():
    s = _build(sc.two_connected_components)
    assert s.batch_layout() == (2, 1, [2])
    s.set_variable(0, 5.0)
    s.set_parameter(0, 2.0)
    assert s.batch_layout() == (2, 1, [2])
    p = s.add_point(9.0, 9.0)
    s.point_point_distance(p, 0, 3.0)  # joins the first component
    assert s.batch_layout() == (2, 2, [1, 1])


def _raw_call(s, opts, n, out):
    reps = np.zeros(max(1, n), dtype=fk.REPORT_DTYPE)
    got = C.c_uint32(0)
    return lib().fk_system_batch_solve(s._h, C.byref(opts), n, None, None, None if out is None else ptr(out, C.c_double),
                                       reps.ctypes.data_as(C.POINTER(FkReport)), 1, C.byref(got), 1)


def test_refusals_before_any_device_work():
    s = _build(sc.two_connected_components)
    out = np.full((2, len(s.variables)), 7.0)
    for dec in (1, 2):
        assert _raw_call(s, FkSolvingOptions(0, dec, 1, 0), 2, out) == -1
    assert _raw_call(s, FkSolvingOptions(2, 0, 1, 0), 2, out) == -1
    assert _raw_call(s, FkSolvingOptions(0, 0, 1, 1), 2, out) == -1
    assert _raw_call(s, FkSolvingOptions(0, 0, 1, 0), 2, None) == -1
    assert np.all(out == 7.0)
    big = _lattice_drawing(80, 60)  # largest front 260 rows: beyond the batched sparse kernel
    out = np.full((2, len(big.variables)), 7.0)
    assert _raw_call(big, FkSolvingOptions(0, 0, 1, 0), 2, out) == -5
    msg = lib().fk_last_error().decode()
    assert "component 0" in msg and "260" in msg, msg
    assert np.all(out == 7.0)


def test_zero_variants():
    s = _build(sc.two_connected_components)
    out, reps = s.batch_solve(n=0)
    assert out.shape == (0, 8) and reps.shape == (0, 2)


# ---- on the device ---------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("optimizer", ["lm", "lbfgs"])
@pytest.mark.parametrize("perturb", [True, False])
@pytest.mark.parametrize("name", sorted(sc.ALL))
def test_every_scenario_equals_the_per_variant_solve(name, perturb, optimizer):
    s = _build(sc.ALL[name])
    vars_, params = _variants(s, 64, seed=zlib.crc32(name.encode()))
    tmpl = s.variables.copy()
    out, reps = s.batch_solve(vars_, params, optimizer=optimizer, perturb=perturb)
    assert np.array_equal(s.variables, tmpl)  # the template is not modified
    ref_out, ref_reps = _loop(s, vars_, params, optimizer, perturb)
    assert reps.shape == ref_reps.shape
    assert np.array_equal(out, ref_out, equal_nan=True), (name, np.argwhere(~((out == ref_out) | (np.isnan(out) & np.isnan(ref_out))))[:5])
    _same_reports(reps, ref_reps)


@pytest.mark.gpu
@pytest.mark.parametrize("name", sorted(sc.REFERENCE_SOLVED))
def test_lm_variants_against_the_oracle(oracle, name):
    s = _build(sc.ALL[name])
    vars_, params = _variants(s, 16, seed=7, specials=False)
    out, reps = s.batch_solve(vars_, params)
    for k in (0, 5, 15):
        so = sc.ALL[name](oracle.System)["s"]
        for i, x in enumerate(vars_[k]):
            so.set_variable(i, float(x))
        for c, x in enumerate(params[k]):
            so.set_parameter(c, float(x))
        so.solve()
        ro = so.reports()
        assert len(ro) == reps.shape[1]
        for a, b in zip(ro, reps[k]):
            assert a["exit_reason"] == b["exit_reason"] and a["trace_hash"] == b["trace_hash"], (name, k, a, b)
        vo = so.variables
        assert np.max(np.abs(vo - out[k])) <= 1e-9 * np.max(np.abs(vo))


@pytest.mark.gpu
@pytest.mark.parametrize("optimizer", ["lm", "lbfgs"])
def test_grouped_structures(optimizer):
    s = _grouping_drawing()
    vars_, params = _variants(s, 40, seed=3)
    out, reps = s.batch_solve(vars_, params, optimizer=optimizer)
    assert reps.shape == (40, 14)
    ref_out, ref_reps = _loop(s, vars_, params, optimizer)
    assert np.array_equal(out, ref_out, equal_nan=True)
    _same_reports(reps, ref_reps)


@pytest.mark.gpu
def test_lattice_component_on_the_sparse_batch_kernel():
    s = _lattice_drawing(30, 20)
    vars_, params = _variants(s, 8, seed=11, specials=False)
    out, reps = s.batch_solve(vars_, params)
    ref_out, ref_reps = _loop(s, vars_, params)
    for f in ("exit_reason", "trace_hash", "outer_iters", "factorizations", "accepted"):
        assert np.array_equal(reps[f], ref_reps[f]), f
    assert np.max(np.abs(out - ref_out)) <= 1e-11 * np.max(np.abs(ref_out))
    out, reps = s.batch_solve(vars_, params, optimizer="lbfgs")
    ref_out, ref_reps = _loop(s, vars_, params, "lbfgs")
    assert np.array_equal(out, ref_out)
    _same_reports(reps, ref_reps)


def test_cad_drawing_components_take_paths_1_and_0(oracle):
    paths = [fk.Topology.from_arrays(len(k[0]), k[1], k[2], k[4], k[5]).info["path"]
             for _, _, k in _cad_drawing(oracle.System).prepare(perturb=False)]
    assert sorted(paths) == [0, 0, 1]
    assert _cad_drawing(RecSystem).batch_layout() == (3, 3, [1, 1, 1])


@pytest.mark.gpu
def test_cad_drawing_with_a_path1_component(oracle):
    """Mixed kinds, fixed points and duplicated slots in every batched component kernel the system batch has for small
    systems: 64 variants equal the per-variant solve bit for bit, three of them the oracle's System.solve."""
    s = _cad_drawing(RecSystem)
    vars_, params = _variants(s, 64, seed=17)
    out, reps = s.batch_solve(vars_, params)
    ref_out, ref_reps = _loop(s, vars_, params)
    assert np.array_equal(out, ref_out, equal_nan=True)
    _same_reports(reps, ref_reps)
    for k in (0, 10, 40):
        so = _cad_drawing(oracle.System)
        for i, x in enumerate(vars_[k]):
            so.set_variable(i, float(x))
        for c, x in enumerate(params[k]):
            so.set_parameter(c, float(x))
        so.solve()
        ro = so.reports()
        assert len(ro) == reps.shape[1] == 3
        for a, b in zip(ro, reps[k]):
            for f in ("exit_reason", "trace_hash", "outer_iters", "factorizations", "accepted", "lambda"):
                assert a[f] == b[f], (k, f, a, b)
            assert abs(a["ssr"] - b["ssr"]) <= 1e-9 * max(a["ssr"], 1.0)
        vo = so.variables
        assert np.max(np.abs(vo - out[k])) <= 1e-9 * np.max(np.abs(vo))


_CHUNK_SCRIPT = """
import sys, numpy as np
sys.path.insert(0, {root!r}); sys.path.insert(0, {tests!r})
import test_gpu_system_batch as t, scenarios as sc
s = t._build(sc.ALL['hinged_triangles_bench_4'])
v, p = t._variants(s, 50, seed=5)
out, reps = s.batch_solve(v, p)
np.savez({path!r}, out=out, reps=reps.view(np.uint8))
"""


@pytest.mark.gpu
def test_chunks_and_devices_do_not_change_results(tmp_path):
    s = _build(sc.ALL["hinged_triangles_bench_4"])
    vars_, params = _variants(s, 50, seed=5)
    out, reps = s.batch_solve(vars_, params)
    path = str(tmp_path / "chunked.npz")
    script = _CHUNK_SCRIPT.format(root=ROOT, tests=os.path.join(ROOT, "tests"), path=path)
    env = dict(os.environ, FK_SYSTEM_BATCH_CHUNK="7")
    subprocess.check_call([sys.executable, "-c", script], env=env, cwd=str(tmp_path))
    got = np.load(path)
    assert np.array_equal(got["out"], out, equal_nan=True)
    assert np.array_equal(got["reps"], reps.view(np.uint8))
    if fk.device_count() < 2:
        pytest.skip("n_gpus=2 needs two devices")
    out2, reps2 = s.batch_solve(vars_, params, n_gpus=2)
    assert np.array_equal(out2, out, equal_nan=True)
    _same_reports(reps2, reps)


@pytest.mark.gpu
def test_large_component_with_lbfgs():
    s = _lattice_drawing(80, 60)
    vars_, params = _variants(s, 2, seed=13, specials=False)
    out, reps = s.batch_solve(vars_, params, optimizer="lbfgs")
    ref_out, ref_reps = _loop(s, vars_[:1], params[:1], "lbfgs")
    assert np.array_equal(out[:1], ref_out)
    _same_reports(reps[:1], ref_reps)


@pytest.mark.gpu
def test_edges():
    # free points without constraints: no component, rows come back as they went in
    s = RecSystem()
    for k in range(4):
        s.add_point(float(k), 1.0 - k)
    vars_, params = _variants(s, 5, seed=1)
    out, reps = s.batch_solve(vars_, params)
    ref_out, ref_reps = _loop(s, vars_, params)
    assert reps.shape == ref_reps.shape == (5, 0)
    assert np.array_equal(out, ref_out, equal_nan=True)
    # vars=None / params=None: the template's own numbers
    s = _build(sc.circle_triangle_line)
    vars_, params = _variants(s, 3, seed=2, specials=False)
    tmpl_v, tmpl_p = s.variables.copy(), np.array(s.params)
    for v, p in ((None, None), (vars_, None), (None, params)):
        out, reps = s.batch_solve(v, p, n=3)
        ref_out, ref_reps = _loop(s, np.tile(tmpl_v, (3, 1)) if v is None else v, np.tile(tmpl_p, (3, 1)) if p is None else p)
        assert np.array_equal(out, ref_out)
        _same_reports(reps, ref_reps)
    assert np.array_equal(s.variables, tmpl_v)
    # a structural edit after a call: the next call solves the new structure
    s = _build(sc.two_connected_components)
    s.batch_solve(n=2)
    p = s.add_point(3.0, 3.0)
    s.point_point_distance(p, 0, 1.5)
    s.fix(p)
    vars_, params = _variants(s, 4, seed=9, specials=False)
    out, reps = s.batch_solve(vars_, params)
    ref_out, ref_reps = _loop(s, vars_, params)
    assert np.array_equal(out, ref_out)
    _same_reports(reps, ref_reps)
