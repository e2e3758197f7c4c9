"""Generates the golden flags that pin System::analyze on lattices too large for the oracle inside a test run.

    python tests/golden/make_analyze_goldens.py 48x40 64x50

For every lattice the oracle (``oracle/``, the pinned CPU restatement of the reference) runs find_overconstraints
(analyze/numerical/mod.rs:123-147) once on the single sketch of ``workloads.lattice(nx, ny)``, about 1 minute for 48x40
and 5 minutes for 64x50 on one core, and the script stores tests/golden/analyze_lattice<nx>x<ny>.json:

  shape          nx, ny, n_vars, n_expr
  sha256         of the raw variables and of the parameters the generator produced (float64 bytes), so that a change
                 of the generator shows up as a failed hash rather than as a wrong golden
  flags          the per-expression "independent" flags, packed MSB first (numpy.packbits), as hex
  independent    the number of independent expressions (the rank)
"""
import hashlib
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)

import oracle  # noqa: E402
from fiksi_b200 import workloads as wl  # noqa: E402


def input_hashes(w):
    return {"raw_vars": hashlib.sha256(np.ascontiguousarray(w.raw_vars[0]).tobytes()).hexdigest(),
            "raw_param": hashlib.sha256(np.ascontiguousarray(w.raw_param[0]).tobytes()).hexdigest()}


def unpack_flags(hexstr, n_expr):
    return np.unpackbits(np.frombuffer(bytes.fromhex(hexstr), dtype=np.uint8))[:n_expr].astype(bool)


def main():
    here = os.path.dirname(os.path.abspath(__file__))
    for case in sys.argv[1:]:
        nx, ny = (int(s) for s in case.split("x"))
        w = wl.lattice(nx, ny)
        t0 = time.time()
        flags = oracle.analyze(w.raw_vars[0], w.kind, w.idx, w.raw_param[0])
        seconds = time.time() - t0
        meta = {"case": f"lattice{nx}x{ny}", "nx": nx, "ny": ny, "n_vars": int(w.n_vars), "n_expr": int(len(w.kind)),
                "sha256": input_hashes(w), "flags": np.packbits(flags.astype(np.uint8)).tobytes().hex(),
                "independent": int(flags.sum())}
        with open(os.path.join(here, f"analyze_lattice{nx}x{ny}.json"), "w") as f:
            json.dump(meta, f, indent=1, sort_keys=True)
        print(case, "independent", meta["independent"], "of", meta["n_expr"], f"{seconds:.1f} s", flush=True)


if __name__ == "__main__":
    main()
