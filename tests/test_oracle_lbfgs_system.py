"""The reference for System::solve with Optimizer::LBfgs (tests/oracle_system.py) is composed from System.prepare and a
per-component solve.  With LM as the optimizer the same composition must reproduce the oracle's own System::solve bit for
bit -- variables and reports -- which pins the composition (scale, perturbation snapshots, write-back) itself."""
import numpy as np
import pytest

import oracle_system
import scenarios as sc

FIELDS = ("exit_reason", "outer_iters", "factorizations", "accepted", "ssr", "lambda", "trace_hash")


@pytest.mark.parametrize("name", sorted(sc.ALL))
@pytest.mark.parametrize("perturb", [True, False])
def test_composition_reproduces_system_solve(oracle, name, perturb):
    a, b = sc.ALL[name](oracle.System), sc.ALL[name](oracle.System)
    variables, reps = oracle_system.solve(oracle, a["s"], perturb=perturb, optimizer="lm")
    b["s"].solve(perturb=perturb)
    assert np.array_equal(variables, b["s"].variables)
    ref = b["s"].reports()
    assert len(reps) == len(ref)
    for r, q in zip(reps, ref):
        assert all(r[f] == q[f] or (r[f] != r[f] and q[f] != q[f]) for f in FIELDS), (r, q)


@pytest.mark.parametrize("name", sorted(sc.ALL))
def test_lbfgs_composition_solves_each_component(oracle, name):
    """optimizer="lbfgs": one oracle.lbfgs_solve per prepared component, nothing else moves."""
    a = sc.ALL[name](oracle.System)
    before = a["s"].variables.copy()
    variables, reps = oracle_system.solve(oracle, a["s"], optimizer="lbfgs")
    assert len(reps) == len(a["s"].prepare())
    touched = np.zeros(len(before), bool)
    for prob, scale, keep in a["s"].prepare():
        vars_, _, _, _, free_vars, _ = keep
        x, rep = oracle.lbfgs_solve(prob, vars_[free_vars])
        assert np.array_equal(variables[free_vars], scale * x)
        touched[free_vars] = True
    assert np.array_equal(variables[~touched], before[~touched])
