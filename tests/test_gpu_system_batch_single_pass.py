"""fk_system_batch_solve_single_pass / System.batch_solve_single_pass: System::solve with Decomposer::SinglePass over n
variants of one drawing in one call.  Every variant must equal a per-variant System.solve_single_pass on the same numbers
(bit for bit where both run the same batched kernels); the plan probe (sets, waves, structures) and the refusals are host
logic and run without a GPU."""
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
from fiksi_b200._lib import FkReport, lib, ptr
from test_gpu_system_batch import RecSystem, _add_ppd, _build, _grouping_drawing, _lattice_drawing, _same_reports, _variants

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _loop(s, vars_, params, perturb=True):
    """The per-variant reference: this system's numbers set to each variant's, then System.solve_single_pass."""
    v0 = s.variables.copy()
    p0 = list(s.params)
    outs, reps = [], []
    for k in range(len(vars_)):
        for i, x in enumerate(vars_[k]):
            s.set_variable(i, float(x))
        for c, x in enumerate(params[k]):
            s.set_parameter(c, float(x))
        s.solve_single_pass(perturb=perturb)
        outs.append(s.variables.copy())
        reps.append(s._reports.copy())
    for i, x in enumerate(v0):
        s.set_variable(i, float(x))
    for c, x in enumerate(p0):
        s.set_parameter(c, float(x))
    return np.array(outs).reshape(len(vars_), len(v0)), np.array(reps).reshape(len(vars_), -1)


def _ring(nx, ny):
    """An nx x ny unit lattice (distances to the left, upper and upper-left neighbours) closed into a ring: the first column
    is tied to the last.  SinglePass finds one strongly connected set of every variable."""
    s = RecSystem()
    pts = [[s.add_point(x + 0.01 * ((7 * x + 3 * y) % 5), y + 0.01 * ((3 * x + 5 * y) % 7)) for x in range(nx)] for y in range(ny)]
    for y in range(ny):
        for x in range(nx):
            if x:
                s.point_point_distance(pts[y][x], pts[y][x - 1], 1.0)
            if y:
                s.point_point_distance(pts[y][x], pts[y - 1][x], 1.0)
            if x and y:
                s.point_point_distance(pts[y][x], pts[y - 1][x - 1], 2 ** 0.5)
    for y in range(ny):
        s.point_point_distance(pts[y][0], pts[y][nx - 1], 1.0)
        if y:
            s.point_point_distance(pts[y][0], pts[y - 1][nx - 1], 2 ** 0.5)
    return s


def _raw_call(s, perturb, n, out):
    reps = np.zeros(max(1, n), dtype=fk.REPORT_DTYPE)
    got = C.c_uint32(0)
    return lib().fk_system_batch_solve_single_pass(s._h, perturb, n, None, None, None if out is None else ptr(out, C.c_double),
                                                   reps.ctypes.data_as(C.POINTER(FkReport)), 1, C.byref(got), 1)


# ---- host only: the plan and the refusals ----------------------------------------------------------------------------
def test_layout_sets_waves_and_structures():
    s = _grouping_drawing()  # 12 identical triangles, circle_triangle_line and a 20-point truss
    n, nw, ns, wave, struct = s.single_pass_batch_layout()
    assert n == len(s.single_pass_plan()) == len(wave) == len(struct)
    assert ns < n and len(set(struct)) == ns
    tri = [struct[k] for k, (free, _) in enumerate(s.single_pass_plan()[:12]) if len(free) == 6]
    assert len(tri) == 12 and len(set(tri)) == 1  # the triangles' sets share one structure across components
    n, nw, ns, wave, _ = _build(sc.two_connected_components).single_pass_batch_layout()
    assert n == 2 and nw == 1 and wave == [0, 0]
    truss = RecSystem()
    _add_ppd(truss, wl.truss(1, 20))
    assert truss.single_pass_batch_layout()[:2] == (17, 17)
    lattice = RecSystem()
    _add_ppd(lattice, wl.lattice(30, 20))
    assert lattice.single_pass_batch_layout()[:2] == (462, 44)
    empty = RecSystem()
    empty.add_point(1.0, 2.0)
    assert empty.single_pass_batch_layout() == (0, 0, 0, [], [])


def test_stale_component_sets_wait_for_what_they_read():
    s = _build(sc.stale_component_quirk)
    plan = s.single_pass_plan()
    _, _, _, wave, _ = s.single_pass_batch_layout()
    solves_b2 = next(k for k, (free, _) in enumerate(plan) if 12 in free and 13 in free)
    fresh = next(k for k, (free, _) in enumerate(plan) if free == [14, 15])
    assert set(plan[solves_b2][1]) & set(plan[fresh][1])  # the {fresh} set reads b[2] as the first set solves it
    assert wave[fresh] > wave[solves_b2]


def test_structural_edit_drops_the_plan():
    s = _build(sc.two_connected_components)
    assert s.single_pass_batch_layout()[:3] == (2, 1, 1)
    s.set_variable(0, 5.0)
    s.set_parameter(0, 2.0)
    assert s.single_pass_batch_layout()[:3] == (2, 1, 1)
    p = s.add_point(9.0, 9.0)
    s.point_point_distance(p, 0, 3.0)  # joins the first component
    assert s.single_pass_batch_layout()[:3] == (2, 1, 2)
    s.fix(p)
    assert s.single_pass_batch_layout()[0] == len(s.single_pass_plan())


def test_refusals_before_any_device_work():
    s = _build(sc.two_connected_components)
    out = np.full((2, len(s.variables)), 7.0)
    assert _raw_call(s, 2, 2, out) == -1
    assert _raw_call(s, -1, 2, out) == -1
    assert _raw_call(s, 1, 2, None) == -1
    assert np.all(out == 7.0)
    big = _ring(80, 60)  # one set of 9,600 variables whose largest front (244 rows) is beyond the batched sparse kernel
    assert big.single_pass_batch_layout()[:3] == (1, 1, 1)
    out = np.full((2, len(big.variables)), 7.0)
    assert _raw_call(big, 1, 2, out) == -5
    msg = lib().fk_last_error().decode()
    assert "set 0" in msg and "first expression 0" in msg and "244" in msg, msg
    assert np.all(out == 7.0)


def test_zero_variants():
    s = _build(sc.two_connected_components)
    out, reps = s.batch_solve_single_pass(n=0)
    assert out.shape == (0, 8) and reps.shape == (0, 2)


# ---- on the device ---------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("perturb", [True, False])
@pytest.mark.parametrize("name", sorted(sc.ALL))
def test_every_scenario_equals_the_per_variant_solve(name, perturb):
    s = _build(sc.ALL[name])
    vars_, params = _variants(s, 48, seed=zlib.crc32(name.encode()) ^ 0x5F)
    tmpl = s.variables.copy()
    out, reps = s.batch_solve_single_pass(vars_, params, perturb=perturb)
    assert np.array_equal(s.variables, tmpl)  # the template is not modified
    ref_out, ref_reps = _loop(s, vars_, params, perturb)
    assert reps.shape == ref_reps.shape
    assert np.array_equal(out, ref_out, equal_nan=True), (name, np.argwhere(~((out == ref_out) | (np.isnan(out) & np.isnan(ref_out))))[:5])
    _same_reports(reps, ref_reps)


@pytest.mark.gpu
@pytest.mark.parametrize("name", sorted(sc.REFERENCE_SOLVED))
def test_variants_against_the_oracle(oracle, name):
    s = _build(sc.ALL[name])
    vars_, params = _variants(s, 16, seed=17, specials=False)
    out, reps = s.batch_solve_single_pass(vars_, params)
    for k in (0, 7, 15):
        so = sc.ALL[name](oracle.System)["s"]
        for i, x in enumerate(vars_[k]):
            so.set_variable(i, float(x))
        for c, x in enumerate(params[k]):
            so.set_parameter(c, float(x))
        so.solve_single_pass()
        ro = so.reports()
        assert len(ro) == reps.shape[1]
        for a, b in zip(ro, reps[k]):
            assert a["exit_reason"] == b["exit_reason"] and a["trace_hash"] == b["trace_hash"], (name, k, a, b)
        vo = so.variables
        assert np.max(np.abs(vo - out[k])) <= 1e-9 * max(np.max(np.abs(vo)), 1e-300)


@pytest.mark.gpu
def test_grouped_structures():
    s = _grouping_drawing()
    vars_, params = _variants(s, 40, seed=3)
    out, reps = s.batch_solve_single_pass(vars_, params)
    ref_out, ref_reps = _loop(s, vars_, params)
    assert np.array_equal(out, ref_out, equal_nan=True)
    _same_reports(reps, ref_reps)


@pytest.mark.gpu
def test_lattice_drawings():
    s = _lattice_drawing(30, 20)  # 30x20 lattice + a triangle
    for _ in range(7):
        sc.single_triangle(lambda: s)
    vars_, params = _variants(s, 12, seed=11)
    out, reps = s.batch_solve_single_pass(vars_, params)
    ref_out, ref_reps = _loop(s, vars_, params)
    assert np.array_equal(out, ref_out, equal_nan=True)
    _same_reports(reps, ref_reps)
    big = _lattice_drawing(80, 60)  # refused by fk_system_batch_solve with LM (largest front 260 rows)
    vars_, params = _variants(big, 3, seed=13, specials=False)
    out, reps = big.batch_solve_single_pass(vars_, params)
    ref_out, ref_reps = _loop(big, vars_, params)
    assert np.array_equal(out, ref_out)
    _same_reports(reps, ref_reps)


@pytest.mark.gpu
def test_set_on_the_sparse_batch_kernel():
    s = _ring(30, 20)  # one set of 1,200 variables on the global sparse path
    vars_, params = _variants(s, 4, seed=19, specials=False)
    out, reps = s.batch_solve_single_pass(vars_, params)
    ref_out, ref_reps = _loop(s, vars_, params)
    for f in ("exit_reason", "trace_hash", "outer_iters", "factorizations", "accepted"):
        assert np.array_equal(reps[f], ref_reps[f]), f
    assert np.max(np.abs(out - ref_out)) <= 1e-11 * np.max(np.abs(ref_out))


_CHUNK_SCRIPT = """
import sys, numpy as np
sys.path.insert(0, {root!r}); sys.path.insert(0, {tests!r})
import test_gpu_system_batch as t, scenarios as sc
s = t._build(sc.ALL['stale_component_quirk'])
v, p = t._variants(s, 50, seed=5)
out, reps = s.batch_solve_single_pass(v, p)
np.savez({path!r}, out=out, reps=reps.view(np.uint8))
"""


@pytest.mark.gpu
def test_chunks_and_devices_do_not_change_results(tmp_path):
    s = _build(sc.ALL["stale_component_quirk"])
    vars_, params = _variants(s, 50, seed=5)
    out, reps = s.batch_solve_single_pass(vars_, params)
    path = str(tmp_path / "chunked.npz")
    script = _CHUNK_SCRIPT.format(root=ROOT, tests=os.path.join(ROOT, "tests"), path=path)
    env = dict(os.environ, FK_SYSTEM_BATCH_CHUNK="7")
    subprocess.check_call([sys.executable, "-c", script], env=env, cwd=str(tmp_path))
    got = np.load(path)
    assert np.array_equal(got["out"], out, equal_nan=True)
    assert np.array_equal(got["reps"], reps.view(np.uint8))
    if fk.device_count() < 2:
        pytest.skip("n_gpus=2 needs two devices")
    out2, reps2 = s.batch_solve_single_pass(vars_, params, n_gpus=2)
    assert np.array_equal(out2, out, equal_nan=True)
    _same_reports(reps2, reps)


@pytest.mark.gpu
def test_edges():
    # free points without constraints: no set, rows come back as they went in
    s = RecSystem()
    for k in range(4):
        s.add_point(float(k), 1.0 - k)
    vars_, params = _variants(s, 5, seed=1)
    out, reps = s.batch_solve_single_pass(vars_, params)
    ref_out, ref_reps = _loop(s, vars_, params)
    assert reps.shape == ref_reps.shape == (5, 0)
    assert np.array_equal(out, ref_out, equal_nan=True)
    # vars=None / params=None: the template's own numbers
    s = _build(sc.circle_triangle_line)
    vars_, params = _variants(s, 3, seed=2, specials=False)
    tmpl_v, tmpl_p = s.variables.copy(), np.array(s.params)
    for v, p in ((None, None), (vars_, None), (None, params)):
        out, reps = s.batch_solve_single_pass(v, p, n=3)
        ref_out, ref_reps = _loop(s, np.tile(tmpl_v, (3, 1)) if v is None else v, np.tile(tmpl_p, (3, 1)) if p is None else p)
        assert np.array_equal(out, ref_out)
        _same_reports(reps, ref_reps)
    assert np.array_equal(s.variables, tmpl_v)
    # a structural edit after a call: the next call solves the new structure
    s = _build(sc.two_connected_components)
    s.batch_solve_single_pass(n=2)
    p = s.add_point(3.0, 3.0)
    s.point_point_distance(p, 0, 1.5)
    s.fix(p)
    vars_, params = _variants(s, 4, seed=9, specials=False)
    out, reps = s.batch_solve_single_pass(vars_, params)
    ref_out, ref_reps = _loop(s, vars_, params)
    assert np.array_equal(out, ref_out)
    _same_reports(reps, ref_reps)
