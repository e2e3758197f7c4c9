"""System::solve with Decomposer::None composed from the oracle's own pieces (assemble/mod.rs:127-167): the per-component
problems of ``System.prepare`` (scaled, seeded perturbation, each a snapshot of the transformed variables), each solved by
the optimizer from its current free values, written back as ``variables[free] = scale * x``.  With ``optimizer="lm"``
this reproduces ``oracle.System.solve`` (checked on the CPU); with ``"lbfgs"`` it is the reference for the GPU's
``System.solve(optimizer="lbfgs")``."""
import numpy as np


def solve(oracle, s, perturb=True, optimizer="lbfgs"):
    """Returns (variables after the solve, one report dict per solved component)."""
    fn = {"lm": oracle.lm_solve, "lbfgs": oracle.lbfgs_solve}[optimizer]
    variables = s.variables.copy()
    reports = []
    for prob, scale, keep in s.prepare(perturb=perturb):
        vars_, _, _, _, free_vars, _ = keep
        out = fn(prob, vars_[free_vars])
        x, rep = out[0], out[1]
        variables[free_vars] = scale * x
        reports.append(rep)
    return variables, reports
