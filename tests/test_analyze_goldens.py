"""The analyze goldens (tests/golden/analyze_lattice*.json) were made from workloads.lattice's single sketch: its raw
variables and parameters must still hash to what the goldens recorded, or the goldens no longer describe these inputs."""
import json
import os

import numpy as np
import pytest

from fiksi_b200 import workloads as wl
from golden.make_analyze_goldens import input_hashes, unpack_flags

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


@pytest.mark.parametrize("nx,ny", [(48, 40), (64, 50)])
def test_golden_inputs_match_the_generator(nx, ny):
    with open(os.path.join(GOLDEN, f"analyze_lattice{nx}x{ny}.json")) as f:
        g = json.load(f)
    w = wl.lattice(nx, ny)
    assert (g["nx"], g["ny"], g["n_vars"], g["n_expr"]) == (nx, ny, w.n_vars, len(w.kind))
    assert input_hashes(w) == g["sha256"]
    flags = unpack_flags(g["flags"], g["n_expr"])
    assert flags.shape == (len(w.kind),) and int(flags.sum()) == g["independent"]
    assert not flags[min(w.n_vars, len(w.kind)):].any()  # rows beyond min(m, n) are never examined
