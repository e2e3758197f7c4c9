"""fk_systems_analyze_layout / fiksi_b200.systems_analyze_layout and the FK_ERR_INVALID refusals of fk_systems_analyze and
fk_systems_residuals: the plan across different drawings and the argument checks are host logic, checked here without a GPU."""
import ctypes as C

import numpy as np

import scenarios as sc
import systems_mix as mix
import fiksi_b200 as fk
from fiksi_b200._lib import lib, ptr


def test_identical_drawings_are_one_structure():
    chains = [mix.hinged_chain(3, seed=1)(fk.System) for _ in range(5)]
    assert fk.systems_analyze_layout(chains) == (1, [5], [0])
    fixed = mix.hinged_chain(3, seed=1)(fk.System)
    fixed.fix(0)  # fixing an element keeps every variable a column: the same structure
    assert fk.systems_analyze_layout(chains + [fixed]) == (1, [6], [0])
    other = mix.hinged_chain(3, seed=2)(fk.System)  # other coordinates and parameters, same structure
    assert fk.systems_analyze_layout(chains + [other, chains[0]]) == (1, [7], [0])
    assert fk.systems_analyze_layout([mix.hinged_chain(4, seed=1)(fk.System)] + chains) == (2, [1, 5], [0, 0])
    assert fk.systems_analyze_layout([]) == (0, [], [])


def test_many_instances_get_a_launch_of_their_own():
    chains = [mix.hinged_chain(3, seed=k)(fk.System) for k in range(64)]
    assert fk.systems_analyze_layout(chains[:63]) == (1, [63], [0])  # fewer than 64: the heterogeneous warp launch
    assert fk.systems_analyze_layout(chains) == (1, [64], [1])
    lone = mix.hinged_chain(4, seed=1)(fk.System)
    assert fk.systems_analyze_layout([lone] + chains) == (2, [1, 64], [0, 1])


def test_launch_kind_follows_the_warp_footprint():
    fits, beyond = mix.hinged_chain(45, seed=1)(fk.System), mix.hinged_chain(46, seed=1)(fk.System)
    assert (len(fits.variables), fits.num_constraints()) == (182, 135)  # 193 KiB per warp
    assert (len(beyond.variables), beyond.num_constraints()) == (186, 138)  # 201 KiB
    assert fk.systems_analyze_layout([fits, beyond, beyond]) == (2, [1, 2], [0, 1])


def test_forced_kernel_sends_every_structure_to_one_launch(monkeypatch):
    systems = [mix.hinged_chain(n, seed=n)(fk.System) for n in (1, 3, 46)]
    assert fk.systems_analyze_layout(systems)[2] == [0, 0, 1]
    for kernel in ("cta", "group"):
        monkeypatch.setenv("FK_ANALYZE_KERNEL", kernel)
        assert fk.systems_analyze_layout(systems)[2] == [1, 1, 1]
    monkeypatch.setenv("FK_ANALYZE_KERNEL", "warp")
    assert fk.systems_analyze_layout(systems)[2] == [0, 0, 1]


def test_mix_counts_every_drawing_once():
    systems = [b(fk.System) for b in mix.mixed(seed=1)]
    ns, inst, kind = fk.systems_analyze_layout(systems)
    assert sum(inst) == len(systems) and ns == len(inst)
    assert kind[inst.index(80)] == 1  # the truss sketches: 80 instances, a launch of their own
    assert set(kind) == {0, 1}


def _call(fn, systems, out, cap, handles=None):
    n = len(systems)
    if handles is None:
        handles = (C.c_void_p * max(n, 1))(*[s._h for s in systems])
    return fn(n, handles, out, cap, 1)


def test_refusals_leave_the_outputs_untouched():
    systems = [sc.two_connected_components(fk.System)["s"], sc.single_triangle(fk.System)["s"], mix.empty(fk.System)]
    total = sum(s.num_constraints() for s in systems)
    before = [s.variables.copy() for s in systems]
    dep = np.full(total + 1, 7, np.uint8)
    res = np.full(total + 1, 7.0)
    for fn, out in ((lib().fk_systems_analyze, ptr(dep, C.c_uint8)), (lib().fk_systems_residuals, ptr(res, C.c_double))):
        assert fn(2, None, out, total, 1) == -1
        assert "null systems" in lib().fk_last_error().decode()
        assert _call(fn, systems, out, total, (C.c_void_p * 3)(systems[0]._h, None, systems[2]._h)) == -1
        assert "index 1" in lib().fk_last_error().decode()
        assert _call(fn, systems, None, total) == -1
        assert "null output" in lib().fk_last_error().decode()
        assert _call(fn, systems, out, total - 1) == -1
        assert str(total) in lib().fk_last_error().decode()
        assert fn(0, None, None, 0, 1) == 0
        assert _call(fn, [systems[2]], None, 0) == 0  # no constraints: nothing to compute, no output needed
    assert (dep == 7).all() and (res == 7.0).all()
    for s, v in zip(systems, before):
        assert np.array_equal(s.variables, v)
    null_sys = (C.c_void_p * 1)(None)
    assert lib().fk_systems_analyze_layout(1, null_sys, None, None, None) == -1
    assert fk.analyze_systems([]) == [] and fk.systems_residuals([]) == []
    counts = fk.analyze_systems([systems[2], mix.lone_point(fk.System)])
    assert [len(c) for c in counts] == [0, 0]
