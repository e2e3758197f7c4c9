"""bench.py --dump-outputs: the arrays written after the timed steps are what the library's own calls return for the
same seeded inputs, and --steps sets the number of timed steps of both the device-resident and the end-to-end loop."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

import fiksi_b200 as fk
from fiksi_b200 import workloads as wl

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_dumped_outputs_are_the_solves_of_the_bench_inputs(tmp_path):
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "2", "--warmup", "0", "--no-extras",
                        "--dump-outputs", str(tmp_path)], capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stderr[-4000:]
    line = json.loads(r.stdout.strip().splitlines()[-1])
    assert line["steps"] == 2 and line["e2e"]["steps"] == 2
    out = {f[:-len(".npy")]: np.load(tmp_path / f) for f in os.listdir(tmp_path)}
    assert all(a.dtype == np.float64 for a in out.values()) and sum(a.nbytes for a in out.values()) <= 64 << 20

    w = wl.truss(65536)
    v, p, scale = w.prepare()
    assert np.all(w.raw_param == w.raw_param[0])  # bench.py sends one shared row of distances
    topo = fk.Topology.from_arrays(w.n_vars, w.kind, w.idx, w.free_vars, w.rows)
    x, rep = topo.batch_solve(v, p)
    xs, _scales, reps = topo.batch_system_solve(w.raw_vars, w.raw_param[0], shared_param=True)
    for prefix, want_x, want_rep in (("", x, rep), ("e2e_", xs, reps)):
        assert np.array_equal(out[prefix + "x"], want_x), prefix + "x"
        for key in ("exit_reason", "outer_iters", "factorizations", "accepted", "ssr", "lambda"):
            assert np.array_equal(out[prefix + key], want_rep[key].astype(np.float64)), prefix + key
        hi, lo = (out[prefix + h].astype(np.uint64) for h in ("trace_hash_hi", "trace_hash_lo"))
        assert np.array_equal((hi << np.uint64(32)) | lo, want_rep["trace_hash"]), prefix + "trace_hash"
