"""fk_systems_layout / fiksi_b200.systems_layout and the refusals of fk_systems_solve: the plan across different drawings and
every refusal are host logic, checked here without a GPU."""
import ctypes as C
import os
import subprocess
import sys

import numpy as np
import pytest

import scenarios as sc
import systems_mix as mix
import fiksi_b200 as fk
from fiksi_b200._lib import FkReport, FkSolvingOptions, lib, ptr

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _triangles(n):
    rng = np.random.default_rng(5)
    out = []
    for _ in range(n):
        s = fk.System()
        a, b, c = s.add_point(*rng.uniform(-2, 2, 2)), s.add_point(*rng.uniform(-2, 2, 2)), s.add_point(*rng.uniform(-2, 2, 2))
        s.point_point_distance(a, b, 1.0)
        s.point_point_distance(b, c, 1.5)
        s.point_point_distance(a, c, 2.0)
        out.append(s)
    return out


def test_identical_structures_merge_across_drawings():
    assert fk.systems_layout(_triangles(100)) == (100, 1, [100], [1])  # 64 and more: one uniform launch
    assert fk.systems_layout(_triangles(3)) == (3, 1, [3], [0])        # fewer: the heterogeneous launch
    assert fk.systems_layout(_triangles(3), optimizer="lbfgs") == (3, 1, [3], [1])


def test_mix_counts_equal_the_drawings_own_layouts():
    systems = [b(fk.System) for b in mix.mixed(seed=1)]
    n_comp, n_struct, inst, kind = fk.systems_layout(systems)
    own = [s.batch_layout() for s in systems]
    assert n_comp == sum(o[0] for o in own) == sum(inst)
    assert max(o[1] for o in own) <= n_struct <= sum(o[1] for o in own)
    assert 80 in inst and kind[inst.index(80)] == 1  # the truss sketches: one structure across 80 drawings
    assert 0 in kind
    # twice the same drawings (other objects): the same structures, twice the instances
    twice = systems + [b(fk.System) for b in mix.mixed(seed=1)]
    assert fk.systems_layout(twice, optimizer="lbfgs") == (2 * n_comp, n_struct, [2 * k for k in inst], [1] * n_struct)
    assert fk.systems_layout([]) == (0, 0, [], [])


def test_merging_does_not_rely_on_the_topology_cache():
    code = ("import sys; sys.path[:0] = [%r, %r]\n"
            "import fiksi_b200 as fk, systems_mix as mix\n"
            "print(fk.systems_layout([b(fk.System) for b in mix.mixed(seed=1)]))\n") % (ROOT, os.path.join(ROOT, "tests"))
    env = dict(os.environ, FK_TOPOLOGY_CACHE="0")
    off = subprocess.run([sys.executable, "-c", code], env=env, capture_output=True, text=True, check=True).stdout.strip()
    assert off == str(fk.systems_layout([b(fk.System) for b in mix.mixed(seed=1)]))


def _raw_solve(systems, opts, handles=None):
    n = len(systems)
    if handles is None:
        handles = (C.c_void_p * max(n, 1))(*[s._h for s in systems])
    reps = np.zeros(64, dtype=fk.REPORT_DTYPE)
    solved = np.zeros(max(n, 1), np.uint32)
    return lib().fk_systems_solve(n, handles, None if opts is None else C.byref(opts), reps.ctypes.data_as(C.POINTER(FkReport)), len(reps),
                                  ptr(solved, C.c_uint32), 1)


def test_refusals_modify_no_system():
    systems = [sc.two_connected_components(fk.System)["s"], sc.single_triangle(fk.System)["s"]]
    before = [s.variables.copy() for s in systems]
    for dec in (1, 2):
        assert _raw_solve(systems, FkSolvingOptions(0, dec, 1, 0)) == -1
    for bad in (FkSolvingOptions(2, 0, 1, 0), FkSolvingOptions(0, 0, 2, 0), FkSolvingOptions(0, 0, 1, 1)):
        assert _raw_solve(systems, bad) == -1
    assert _raw_solve(systems, None) == -1
    ok = FkSolvingOptions(0, 0, 1, 0)
    assert _raw_solve(systems, ok, (C.c_void_p * 2)(systems[0]._h, None)) == -1
    assert _raw_solve(systems + [systems[0]], ok) == -1
    assert "twice" in lib().fk_last_error().decode()
    assert lib().fk_systems_solve(2, None, C.byref(ok), None, 0, None, 1) == -1
    assert lib().fk_systems_solve(0, None, C.byref(ok), None, 0, None, 1) == 0
    for s, v in zip(systems, before):
        assert np.array_equal(s.variables, v)
    with pytest.raises(fk.FiksiError):
        fk.solve_systems([systems[0], systems[0]])
    assert fk.solve_systems([]) == []
