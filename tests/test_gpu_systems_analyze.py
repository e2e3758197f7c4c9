"""fk_systems_analyze / fk_systems_residuals (fiksi_b200.analyze_systems / systems_residuals): System::analyze and
calculate_residual over many different drawings in one call.  Every drawing must equal its own System.analyze() /
System.residuals(), bit for bit."""
import ctypes as C
import os
import subprocess
import sys

import numpy as np
import pytest

import systems_mix as mix
import fiksi_b200 as fk
from fiksi_b200._lib import lib, ptr

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def henneberg(n_points, seed):
    """A drawing of n_points built by seeded random Henneberg steps: every new point tied to two random earlier points."""
    def build(S):
        rng = np.random.default_rng(seed)
        s = S()
        p = [s.add_point(*rng.uniform(-5, 5, 2)) for _ in range(n_points)]
        s.point_point_distance(p[0], p[1], float(rng.uniform(1, 3)))
        for i in range(2, n_points):
            a, b = rng.choice(i, 2, replace=False)
            s.point_point_distance(p[i], p[int(a)], float(rng.uniform(1, 3)))
            s.point_point_distance(p[i], p[int(b)], float(rng.uniform(1, 3)))
        return s
    return build


def _check(systems, counts=None, res=None):
    """Every drawing's counts give its own analyze() list; every drawing's residuals are its own residuals()."""
    counts = fk.analyze_systems(systems) if counts is None else counts
    res = fk.systems_residuals(systems) if res is None else res
    assert len(counts) == len(res) == len(systems)
    for i, s in enumerate(systems):
        assert counts[i].dtype == np.uint8 and len(counts[i]) == s.num_constraints(), i
        assert np.repeat(np.arange(s.num_constraints()), counts[i]).tolist() == s.analyze(), i
        assert np.array_equal(res[i], s.residuals(), equal_nan=True), i
    return counts, res


@pytest.mark.gpu
@pytest.mark.parametrize("seed", [3, 4])
def test_mix_equals_every_drawings_own_analyze_and_residuals(seed):
    systems = [b(fk.System) for b in mix.mixed(seed)]
    assert set(fk.systems_analyze_layout(systems)[2]) == {0, 1}
    counts, _ = _check(systems)
    assert any(c.any() for c in counts)  # the over-constrained scenarios are in the mix


@pytest.mark.gpu
def test_many_distinct_structures_in_one_heterogeneous_launch():
    rng = np.random.default_rng(11)
    systems = [henneberg(int(rng.integers(4, 13)), seed=k)(fk.System) for k in range(500)]
    ns, inst, kind = fk.systems_analyze_layout(systems)
    assert kind.count(0) > 200
    _check(systems)


@pytest.mark.gpu
def test_footprint_classes_in_one_call():
    builders = [mix.lone_point, mix.hinged_chain(1, seed=1), mix.hinged_chain(45, seed=2), mix.scenario(sorted(mix.sc.ALL)[0])]
    builders += [mix.hinged_chain(n, seed=n) for n in range(2, 12)] + [mix.hinged_chain(45, seed=3)]
    systems = [b(fk.System) for b in builders]
    assert set(fk.systems_analyze_layout(systems)[2]) == {0}
    _check(systems)


@pytest.mark.gpu
def test_beyond_the_warp_kernel_every_kernel_agrees(monkeypatch):
    builders = [mix.hinged_chain(46, seed=k) for k in range(4)] + [mix.cad_drawing, mix.hinged_chain(2, seed=9)]
    systems = [b(fk.System) for b in builders]
    ns, inst, kind = fk.systems_analyze_layout(systems)
    assert any(k == 1 and i > 1 for i, k in zip(inst, kind))  # one structure with several instances through kind 1
    counts, _ = _check(systems)
    for kernel in ("cta", "group"):
        monkeypatch.setenv("FK_ANALYZE_KERNEL", kernel)
        assert set(fk.systems_analyze_layout(systems)[2]) == {1}
        forced = fk.analyze_systems(systems)
        for a, b in zip(forced, counts):
            assert np.array_equal(a, b), kernel


@pytest.mark.gpu
def test_drawing_beyond_the_analyze_limit_is_refused():
    systems = [b(fk.System) for b in mix.mixed(seed=7)[:10]] + [mix.lattice_drawing(120, 112)(fk.System)]
    total = sum(s.num_constraints() for s in systems)
    out = np.full(total, 7, np.uint8)
    handles = (C.c_void_p * len(systems))(*[s._h for s in systems])
    assert lib().fk_systems_analyze(len(systems), handles, ptr(out, C.c_uint8), total, 1) == -5
    assert "drawing 10: " in lib().fk_last_error().decode()
    assert (out == 7).all()
    res = fk.systems_residuals(systems)
    for i, s in enumerate(systems):
        assert np.array_equal(res[i], s.residuals(), equal_nan=True), i


@pytest.mark.gpu
def test_nan_stays_in_its_drawing():
    builders = mix.mixed(seed=5)[:40]
    clean, dirty = [b(fk.System) for b in builders], [b(fk.System) for b in builders]
    k = next(i for i, s in enumerate(dirty) if len(s.variables) > 2 and s.num_constraints() > 0)
    dirty[k].set_variable(1, float("nan"))
    a, b = fk.analyze_systems(clean), fk.analyze_systems(dirty)
    ra, rb = fk.systems_residuals(clean), fk.systems_residuals(dirty)
    assert np.isnan(rb[k]).any()
    for i in range(len(builders)):
        if i != k:
            assert np.array_equal(a[i], b[i]) and np.array_equal(ra[i], rb[i], equal_nan=True), i
    _check(dirty, b, rb)


@pytest.mark.gpu
def test_duplicates_are_accepted_and_no_system_changes():
    systems = [b(fk.System) for b in mix.mixed(seed=8)[:30]]
    before = [(s.variables.copy(), s.residuals().copy()) for s in systems]
    twice = systems + systems[:10] + [systems[3]]
    counts, res = _check(twice)
    for s, (v, r) in zip(systems, before):
        assert np.array_equal(s.variables, v, equal_nan=True)
        assert np.array_equal(s.residuals(), r, equal_nan=True)  # (the parameters too)
    for j, i in enumerate(list(range(10)) + [3]):
        assert np.array_equal(counts[30 + j], counts[i]) and np.array_equal(res[30 + j], res[i], equal_nan=True)


_CHUNK_SCRIPT = """
import sys; sys.path[:0] = [{root!r}, {tests!r}]
import numpy as np, fiksi_b200 as fk, systems_mix as mix
systems = [b(fk.System) for b in mix.mixed(seed=6)]
np.save({dep!r}, np.concatenate(fk.analyze_systems(systems)))
np.save({res!r}, np.concatenate(fk.systems_residuals(systems)))
"""


@pytest.mark.gpu
def test_chunks_and_devices_change_nothing(tmp_path):
    systems = [b(fk.System) for b in mix.mixed(seed=6)]
    dep = np.concatenate(fk.analyze_systems(systems))
    res = np.concatenate(fk.systems_residuals(systems))
    assert np.array_equal(np.concatenate(fk.analyze_systems(systems, n_gpus=0)), dep)
    assert np.array_equal(np.concatenate(fk.systems_residuals(systems, n_gpus=0)), res, equal_nan=True)
    d, r = str(tmp_path / "dep.npy"), str(tmp_path / "res.npy")
    code = _CHUNK_SCRIPT.format(root=ROOT, tests=os.path.join(ROOT, "tests"), dep=d, res=r)
    subprocess.run([sys.executable, "-c", code], env=dict(os.environ, FK_SYSTEM_BATCH_CHUNK="3"), check=True)
    assert np.array_equal(np.load(d), dep)
    assert np.array_equal(np.load(r), res, equal_nan=True)


@pytest.mark.gpu
def test_diagnosing_a_solved_sweep():
    builders = mix.mixed(seed=9)
    systems, twins = [b(fk.System) for b in builders], [b(fk.System) for b in builders]
    fk.solve_systems(systems)
    for t in twins:
        t.solve()
    counts, res = fk.analyze_systems(systems), fk.systems_residuals(systems)
    for s, t in zip(systems, twins):
        assert np.array_equal(s.variables, t.variables, equal_nan=True)
    _check(twins, counts, res)
