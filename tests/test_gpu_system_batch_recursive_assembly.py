"""fk_system_batch_solve_recursive_assembly / System.batch_solve_recursive_assembly: System::solve with
Decomposer::RecursiveAssembly over n variants of one drawing in one call, against the per-variant
System.solve_recursive_assembly.  Bit for bit on drawings whose plan moves no point; where a step moves the points a cluster
owns, the device's sincos and glibc's sin / cos may differ in the last place, so every step's decisions must agree and
coordinates within 1e-11 of the variant's largest |value|.  The plan probe (steps, waves, structures) and the refusals are
host logic and run without a GPU."""
import ctypes as C
import os
import subprocess
import sys
import zlib

import numpy as np
import pytest

import scenarios as sc
import fiksi_b200 as fk
from fiksi_b200._lib import FkReport, lib, ptr
from test_gpu_system_batch import RecSystem, _build, _same_reports, _variants
from test_recursive_assembly import _random_system

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
# the planner's search is exhaustive: the two long benchmark chains are left out, as in test_recursive_assembly
SOLVABLE = ["coincident_points", "collinear_points", "distance_and_angle", "fixed_point_and_circle_center_incidence",
            "fixed_with_coincidence", "hinged_triangles", "hinged_triangles_bench_4", "large_order_of_magnitude", "lib_doc_example",
            "metric_and_singular", "near_degenerate_isosceles_triangle", "overconstrained", "overconstrained_triangle_line_incidence",
            "single_triangle", "single_triangle_fixed_p1", "triangle_inscribed_circle", "two_connected_components",
            "underconstrained_triangle"]
PANICS = ["circle_triangle_line", "connected_triangles", "stale_component_quirk"]
NO_MOVES = ["coincident_points", "fixed_point_and_circle_center_incidence", "two_connected_components", "underconstrained_triangle"]
REPORT_DECISIONS = ("exit_reason", "outer_iters", "factorizations", "trace_hash")


def _loop(s, vars_, params, perturb=True):
    """The per-variant reference: this system's numbers set to each variant's, then System.solve_recursive_assembly."""
    v0 = s.variables.copy()
    p0 = list(s.params)
    outs, reps = [], []
    for k in range(len(vars_)):
        for i, x in enumerate(vars_[k]):
            s.set_variable(i, float(x))
        for c, x in enumerate(params[k]):
            s.set_parameter(c, float(x))
        s.solve_recursive_assembly(perturb=perturb)
        outs.append(s.variables.copy())
        reps.append(s._reports.copy())
    for i, x in enumerate(v0):
        s.set_variable(i, float(x))
    for c, x in enumerate(p0):
        s.set_parameter(c, float(x))
    return np.array(outs).reshape(len(vars_), len(v0)), np.array(reps).reshape(len(vars_), -1)


def _agree(out, reps, ref_out, ref_reps):
    """The contract where steps move points: equal decisions per step, coordinates within 1e-11 of the variant's largest
    finite |value| (non-finite values equal).  Returns the fraction of variants that are bit-identical anyway."""
    assert reps.shape == ref_reps.shape
    for f in REPORT_DECISIONS:
        assert np.array_equal(reps[f], ref_reps[f]), f
    same = (out == ref_out) | (np.isnan(out) & np.isnan(ref_out))
    fin = np.where(np.isfinite(ref_out), np.abs(ref_out), 0.0)
    tol = 1e-11 * np.max(fin, axis=1, initial=0.0)[:, None]
    with np.errstate(invalid="ignore"):
        close = np.isfinite(out) & np.isfinite(ref_out) & (np.abs(out - ref_out) <= tol)
    assert np.all(same | close), np.argwhere(~same)[:5]
    return float(np.mean(np.all(same, axis=1))) if len(out) else 1.0


def _chains_drawing(chains=16, triangles=8, circles=4):
    """16 hinged 4-triangle chains + 8 single triangles + 4 triangle_inscribed_circle: 28 components, 240 steps."""
    s = RecSystem()
    for _ in range(chains):
        sc.hinged_triangles_bench(lambda: s, 4)
    for _ in range(triangles):
        sc.single_triangle(lambda: s)
    for _ in range(circles):
        sc.triangle_inscribed_circle(lambda: s)
    return s


def _no_moves_drawing():
    s = RecSystem()
    for name in NO_MOVES:
        sc.ALL[name](lambda: s)
    return s


def _raw_call(s, perturb, n, out):
    reps = np.zeros(max(1, n), dtype=fk.REPORT_DTYPE)
    got = C.c_uint32(0)
    return lib().fk_system_batch_solve_recursive_assembly(s._h, perturb, n, None, None, None if out is None else ptr(out, C.c_double),
                                                          reps.ctypes.data_as(C.POINTER(FkReport)), 1, C.byref(got), 1)


# ---- host only: the plan and the refusals ----------------------------------------------------------------------------
@pytest.mark.parametrize("name", SOLVABLE)
def test_layout_steps_equal_the_plan(name):
    s = _build(sc.ALL[name])
    n, nw, ns, wave, struct = s.recursive_assembly_batch_layout()
    assert n == s.recursive_assembly_plan()[0] == len(wave) == len(struct) >= 1
    assert 1 <= nw <= n and 1 <= ns <= n and max(wave) == nw - 1 and sorted(set(struct)) == list(range(ns))


def test_layout_of_the_chains_drawing():
    s = _chains_drawing()
    assert len([c for c in s.components() if c[0]]) == 28
    n, nw, ns, wave, struct = s.recursive_assembly_batch_layout()
    assert n == 240
    chain = 12  # steps of one 4-triangle chain
    for c in range(16):  # step k of every chain: one structure, one wave
        assert struct[c * chain:(c + 1) * chain] == struct[:chain] and wave[c * chain:(c + 1) * chain] == wave[:chain]
    assert len(set(struct[:chain])) == chain
    tri = struct[16 * chain:16 * chain + 24]
    assert tri == tri[:3] * 8  # the single triangles' steps share theirs too
    assert nw == max(wave) + 1 <= chain and ns < 40


def test_plan_kept_by_values_dropped_by_structural_edits():
    s = _build(sc.two_connected_components)
    assert s.recursive_assembly_batch_layout() == (2, 1, 1, [0, 0], [0, 0])
    s.set_variable(0, 5.0)
    s.set_parameter(0, 2.0)
    assert s.recursive_assembly_batch_layout() == (2, 1, 1, [0, 0], [0, 0])
    p = s.add_point(9.0, 9.0)
    s.point_point_distance(p, 0, 3.0)  # joins the first component
    n = s.recursive_assembly_batch_layout()[0]
    assert n == s.recursive_assembly_plan()[0] and n > 2
    s.fix(p)
    assert s.recursive_assembly_batch_layout()[0] == s.recursive_assembly_plan()[0]
    q = s.add_point(1.0, 1.0)
    s.point_point_distance(q, p, 1.0)
    assert s.recursive_assembly_batch_layout()[0] == s.recursive_assembly_plan()[0] == n + 1


def test_refusals_before_any_device_work():
    s = _build(sc.two_connected_components)
    out = np.full((2, len(s.variables)), 7.0)
    assert _raw_call(s, 2, 2, out) == -1
    assert _raw_call(s, -1, 2, out) == -1
    assert _raw_call(s, 1, 2, None) == -1
    assert np.all(out == 7.0)
    for name in PANICS:  # the reference panics on these plans
        s = _build(sc.ALL[name])
        out = np.full((2, len(s.variables)), 7.0)
        assert _raw_call(s, 1, 2, out) == -1, name
        assert "the reference panics" in lib().fk_last_error().decode()
        assert np.all(out == 7.0)
    s = _random_system(RecSystem, np.random.default_rng(377))  # its last step reads a point a contraction took away
    out = np.full((2, len(s.variables)), 7.0)
    assert _raw_call(s, 1, 2, out) == -1
    assert "an expression reads a variable outside its step" in lib().fk_last_error().decode()
    assert np.all(out == 7.0)


def test_zero_variants():
    s = _build(sc.two_connected_components)
    out, reps = s.batch_solve_recursive_assembly(n=0)
    assert out.shape == (0, 8) and reps.shape == (0, 2)


# ---- on the device ---------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("perturb", [True, False])
@pytest.mark.parametrize("name", SOLVABLE)
def test_every_scenario_against_the_per_variant_solve(name, perturb):
    s = _build(sc.ALL[name])
    vars_, params = _variants(s, 48, seed=zlib.crc32(name.encode()) ^ 0x2A)
    tmpl = s.variables.copy()
    out, reps = s.batch_solve_recursive_assembly(vars_, params, perturb=perturb)
    assert np.array_equal(s.variables, tmpl)  # the template is not modified
    ref_out, ref_reps = _loop(s, vars_, params, perturb)
    if name in NO_MOVES:
        assert np.array_equal(out, ref_out, equal_nan=True)
        _same_reports(reps, ref_reps)
    else:
        print(f"{name} perturb={perturb}: bit-identical variants {_agree(out, reps, ref_out, ref_reps):.3f}")


@pytest.mark.gpu
@pytest.mark.parametrize("perturb", [True, False])
def test_drawing_without_moves_is_bit_identical(perturb):
    s = _no_moves_drawing()
    vars_, params = _variants(s, 64, seed=23)
    out, reps = s.batch_solve_recursive_assembly(vars_, params, perturb=perturb)
    ref_out, ref_reps = _loop(s, vars_, params, perturb)
    assert np.array_equal(out, ref_out, equal_nan=True)
    _same_reports(reps, ref_reps)


@pytest.mark.gpu
def test_chains_drawing_against_the_loop():
    s = _chains_drawing()
    vars_, params = _variants(s, 256, seed=29)
    out, reps = s.batch_solve_recursive_assembly(vars_, params)
    sample = [0, 1, 2, 3, 77, 255]
    ref_out, ref_reps = _loop(s, vars_[sample], params[sample])
    print(f"chains drawing: bit-identical variants {_agree(out[sample], reps[sample], ref_out, ref_reps):.3f}")


@pytest.mark.gpu
@pytest.mark.parametrize("name", SOLVABLE)
def test_variants_against_the_oracle(oracle, name):
    """Traces and exits equal to the oracle's restatement.  Coordinates within 1e-9 where every step is consistent; on a
    self-contradicting drawing (a step ends with a sum of squares above the LM threshold) the least-squares compromise is
    rounded differently by the normal equations here and the oracle's QR (SURVEY H1), so there the final sums of squares
    must agree instead, as in test_recursive_assembly."""
    s = _build(sc.ALL[name])
    vars_, params = _variants(s, 16, seed=31, specials=False)
    out, reps = s.batch_solve_recursive_assembly(vars_, params)
    for k in (0, 9):
        so = sc.ALL[name](oracle.System)["s"]
        for i, x in enumerate(vars_[k]):
            so.set_variable(i, float(x))
        for c, x in enumerate(params[k]):
            so.set_parameter(c, float(x))
        so.solve_recursive_assembly()
        ro = so.reports()
        assert len(ro) == reps.shape[1]
        for a, b in zip(ro, reps[k]):
            assert a["exit_reason"] == b["exit_reason"] and a["trace_hash"] == b["trace_hash"], (name, k, a, b)
        vo = np.asarray(so.variables)
        if all(a["ssr"] < 1e-8 for a in ro):
            assert np.max(np.abs(vo - out[k])) <= 1e-9 * max(np.max(np.abs(vo)), 1e-300)
        else:
            for a, b in zip(ro, reps[k]):
                assert abs(a["ssr"] - b["ssr"]) <= 1e-7 * max(a["ssr"], 1.0), (name, k, a, b)


_CHUNK_SCRIPT = """
import sys, numpy as np
sys.path.insert(0, {root!r}); sys.path.insert(0, {tests!r})
import test_gpu_system_batch_recursive_assembly as t, test_gpu_system_batch as b
s = t._chains_drawing(2, 2, 1)
v, p = b._variants(s, 50, seed=5)
out, reps = s.batch_solve_recursive_assembly(v, p)
np.savez({path!r}, out=out, reps=reps.view(np.uint8))
"""


@pytest.mark.gpu
def test_chunks_do_not_change_results(tmp_path):
    s = _chains_drawing(2, 2, 1)
    vars_, params = _variants(s, 50, seed=5)
    out, reps = s.batch_solve_recursive_assembly(vars_, params)
    path = str(tmp_path / "chunked.npz")
    script = _CHUNK_SCRIPT.format(root=ROOT, tests=os.path.join(ROOT, "tests"), path=path)
    env = dict(os.environ, FK_SYSTEM_BATCH_CHUNK="3")
    subprocess.check_call([sys.executable, "-c", script], env=env, cwd=str(tmp_path))
    got = np.load(path)
    assert np.array_equal(got["out"], out, equal_nan=True)
    assert np.array_equal(got["reps"], reps.view(np.uint8))


@pytest.mark.gpu
def test_two_devices_do_not_change_results():
    if fk.device_count() < 2:
        pytest.skip("n_gpus=2 needs two devices")
    s = _chains_drawing(2, 2, 1)
    vars_, params = _variants(s, 50, seed=5)
    out, reps = s.batch_solve_recursive_assembly(vars_, params)
    out2, reps2 = s.batch_solve_recursive_assembly(vars_, params, n_gpus=2)
    assert np.array_equal(out2, out, equal_nan=True)
    _same_reports(reps2, reps)


@pytest.mark.gpu
def test_edges():
    # free points without constraints: no step, rows come back as they went in
    s = RecSystem()
    for k in range(4):
        s.add_point(float(k), 1.0 - k)
    vars_, params = _variants(s, 5, seed=1)
    out, reps = s.batch_solve_recursive_assembly(vars_, params)
    ref_out, ref_reps = _loop(s, vars_, params)
    assert reps.shape == ref_reps.shape == (5, 0)
    assert np.array_equal(out, ref_out, equal_nan=True)
    # vars=None / params=None: the template's own numbers
    s = _build(sc.triangle_inscribed_circle)
    vars_, params = _variants(s, 3, seed=2, specials=False)
    tmpl_v, tmpl_p = s.variables.copy(), np.array(s.params)
    for v, p in ((None, None), (vars_, None), (None, params)):
        out, reps = s.batch_solve_recursive_assembly(v, p, n=3)
        ref_out, ref_reps = _loop(s, np.tile(tmpl_v, (3, 1)) if v is None else v, np.tile(tmpl_p, (3, 1)) if p is None else p)
        _agree(out, reps, ref_out, ref_reps)
    assert np.array_equal(s.variables, tmpl_v)
