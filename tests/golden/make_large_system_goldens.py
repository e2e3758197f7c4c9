"""Generates the golden fixtures that pin the large single-system path (BASELINE config 3) against the
oracle at sizes the oracle cannot finish inside a test run.

    python tests/golden/make_large_system_goldens.py lattice150x120 irregular12000 lattice400x250

For every case: the oracle (``oracle/``, the pinned CPU restatement of the reference) runs the whole
Levenberg-Marquardt solve in its bit-identical fast QR mode (``oracle.qr_fast``; identity with the
reference-cost mode is checked by tests/test_oracle_fast_mode.py) and the script stores

  tests/golden/large_<case>.json   sizes, sha256 of the augmented CSC pattern / COLAMD permutation /
                                   etree / R pattern, the accept-reject trace, exit, counts, ssr, lambda
  tests/golden/large_<case>_x.npy  the converged free variables (float64); above X_FULL_MAX variables a
                                   seeded sample of them, described by the JSON's "x_sample"

The inputs come from fiksi_b200.workloads generators (pure numpy, deterministic), so the GPU tests
rebuild them from the case name.  lattice400x250 needs ~35 GB of RAM and a few hours on one core.
"""
import hashlib
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import oracle  # noqa: E402
from large_cases import X_FULL_MAX, X_SAMPLE_SIZE, build_case, x_sample_indices  # noqa: E402


def sha(a):
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


def main():
    here = os.path.dirname(os.path.abspath(__file__))
    os.environ.setdefault("ORC_PROGRESS", "1")
    for case in sys.argv[1:]:
        args = build_case(case)
        op, keep = oracle.make_problem(*args)
        x0 = args[0][args[4]]
        t0 = time.time()
        sym = oracle.symbolic(op)
        t_sym = time.time() - t0
        meta = {
            "case": case, "n_free": int(op.n_free), "n_rows": int(op.n_rows),
            "aug_nnz": int(len(sym["aug_rowidx"])), "r_nnz": int(len(sym["r_rowidx"])),
            "sha256": {k: sha(v) for k, v in sym.items()},
            "dtypes": {k: str(v.dtype) for k, v in sym.items()},
            "oracle_symbolic_seconds": round(t_sym, 2),
        }
        print(case, "symbolic done", round(t_sym, 1), "s, r_nnz", meta["r_nnz"], flush=True)
        with oracle.qr_fast(True):
            t0 = time.time()
            x, rep, trace = oracle.lm_solve(op, x0)
            meta["oracle_lm_seconds"] = round(time.time() - t0, 1)
        meta["trace"] = trace
        meta["report"] = {k: (float(v).hex() if isinstance(v, float) else int(v)) for k, v in rep.items()}
        if len(x) > X_FULL_MAX:
            # the tests normalise by the largest coordinate of the whole solution, so it is kept beside the sample
            meta["x_sample"] = {"size": X_SAMPLE_SIZE, "seed": 0, "max_abs": float(np.max(np.abs(x))).hex()}
            x = x[x_sample_indices(len(x), X_SAMPLE_SIZE, 0)]
        np.save(os.path.join(here, f"large_{case}_x.npy"), x)
        with open(os.path.join(here, f"large_{case}.json"), "w") as f:
            json.dump(meta, f, indent=1, sort_keys=True)
        print(case, "done:", trace, rep, meta["oracle_lm_seconds"], "s", flush=True)


if __name__ == "__main__":
    main()
