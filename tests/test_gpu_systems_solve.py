"""fk_systems_solve / fiksi_b200.solve_systems: System::solve over many different drawings in one call.  Every drawing must
equal its own System.solve on an identically built twin, bit for bit (LM on the global sparse path: equal decisions,
coordinates within 1e-11)."""
import os
import subprocess
import sys

import numpy as np
import pytest

import systems_mix as mix
import fiksi_b200 as fk

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
_DECISIONS = ("exit_reason", "trace_hash", "outer_iters", "factorizations", "accepted")


@pytest.fixture
def twins():
    """build(builders) -> (systems for the batch call, identically built twins for the per-drawing solve)."""
    return lambda builders: ([b(fk.System) for b in builders], [b(fk.System) for b in builders])


def _solve_twins(twins, optimizer, perturb):
    out = []
    for t in twins:
        t.solve(perturb=perturb, optimizer=optimizer)
        out.append(t._reports.copy())
    return out


def _same(a, b):
    for f in a.dtype.names:
        assert np.array_equal(a[f], b[f], equal_nan=a[f].dtype.kind == "f"), f


@pytest.mark.gpu
@pytest.mark.parametrize("optimizer", ["lm", "lbfgs"])
@pytest.mark.parametrize("perturb", [True, False])
def test_mix_equals_every_drawings_own_solve(twins, optimizer, perturb):
    systems, ref = twins(mix.mixed(seed=3))
    kinds = set(fk.systems_layout(systems, optimizer)[3])
    assert kinds == ({0, 1} if optimizer == "lm" else {1})
    reps = fk.solve_systems(systems, optimizer=optimizer, perturb=perturb)
    ref_reps = _solve_twins(ref, optimizer, perturb)
    for i, (s, t) in enumerate(zip(systems, ref)):
        assert np.array_equal(s.variables, t.variables, equal_nan=True), i
        assert len(reps[i]) == len(ref_reps[i]), i
        _same(reps[i], ref_reps[i])


@pytest.mark.gpu
def test_lattice_in_the_mix_runs_the_sparse_batch_kernel(twins):
    builders = mix.mixed(seed=4)[:20] + [mix.lattice_drawing(30, 20)]
    systems, ref = twins(builders)
    assert 2 in fk.systems_layout(systems)[3]
    reps = fk.solve_systems(systems)
    ref_reps = _solve_twins(ref, "lm", True)
    for s, t, r, q in zip(systems[:-1], ref[:-1], reps[:-1], ref_reps[:-1]):
        assert np.array_equal(s.variables, t.variables, equal_nan=True)
        _same(r, q)
    for f in _DECISIONS:
        assert np.array_equal(reps[-1][f], ref_reps[-1][f]), f
    a, b = systems[-1].variables, ref[-1].variables
    assert np.max(np.abs(a - b)) <= 1e-11 * np.max(np.abs(b))
    systems, ref = twins(builders)  # L-BFGS: bit for bit on every size
    reps = fk.solve_systems(systems, optimizer="lbfgs")
    ref_reps = _solve_twins(ref, "lbfgs", True)
    for s, t, r, q in zip(systems, ref, reps, ref_reps):
        assert np.array_equal(s.variables, t.variables, equal_nan=True)
        _same(r, q)


@pytest.mark.gpu
def test_nan_stays_in_its_drawing(twins):
    builders = mix.mixed(seed=5)[:40]
    clean, dirty = twins(builders)
    k = next(i for i, s in enumerate(dirty) if len(s.variables) > 2 and fk.systems_layout([s])[0])
    dirty[k].set_variable(1, float("nan"))
    fk.solve_systems(clean)
    reps = fk.solve_systems(dirty)
    assert np.isnan(dirty[k].variables).any()
    for i, (a, b) in enumerate(zip(clean, dirty)):
        if i != k:
            assert np.array_equal(a.variables, b.variables), i
    assert len(reps) == len(dirty)


_CHUNK_SCRIPT = """
import sys; sys.path[:0] = [{root!r}, {tests!r}]
import numpy as np, fiksi_b200 as fk, systems_mix as mix
systems = [b(fk.System) for b in mix.mixed(seed=6)]
reps = fk.solve_systems(systems, optimizer={opt!r})
np.save({out!r}, np.concatenate([s.variables for s in systems]))
np.save({rep!r}, np.concatenate(reps))
"""


@pytest.mark.gpu
@pytest.mark.parametrize("optimizer", ["lm", "lbfgs"])
def test_chunks_and_devices_change_nothing(twins, tmp_path, optimizer):
    systems, every_device = twins(mix.mixed(seed=6))
    reps = fk.solve_systems(systems, optimizer=optimizer)
    vars_ = np.concatenate([s.variables for s in systems])
    all_reps = np.concatenate(reps)
    reps0 = fk.solve_systems(every_device, optimizer=optimizer, n_gpus=0)
    assert np.array_equal(np.concatenate([s.variables for s in every_device]), vars_, equal_nan=True)
    _same(np.concatenate(reps0), all_reps)
    out, rep = str(tmp_path / "vars.npy"), str(tmp_path / "reps.npy")
    code = _CHUNK_SCRIPT.format(root=ROOT, tests=os.path.join(ROOT, "tests"), opt=optimizer, out=out, rep=rep)
    subprocess.run([sys.executable, "-c", code], env=dict(os.environ, FK_SYSTEM_BATCH_CHUNK="3"), check=True)
    assert np.array_equal(np.load(out), vars_, equal_nan=True)
    _same(np.load(rep), all_reps)


@pytest.mark.gpu
def test_front_beyond_the_sparse_batch_kernel_is_refused(twins):
    systems, _ = twins(mix.mixed(seed=7)[:10] + [mix.lattice_drawing(80, 60)])
    before = [s.variables.copy() for s in systems]
    with pytest.raises(fk.FiksiError) as e:
        fk.solve_systems(systems)
    assert e.value.code == -5
    assert "drawing 10" in str(e.value) and "component 0" in str(e.value) and "260" in str(e.value), str(e.value)
    for s, v in zip(systems, before):
        assert np.array_equal(s.variables, v, equal_nan=True)
