"""The host-buffer chunk pipeline of a (topology, device), which fk_batch_system_solve and fk_batch_solve_device (and their
_begin / _wait halves) share: both kinds of call mixed on one pipeline, a synchronous call between two halves, plans regrown
by one kind of call and reused by the other, and the FK_E2E_TRACE chunk timeline."""
import math
import os
import subprocess
import sys

import numpy as np
import pytest

import fiksi_b200 as fk
from fiksi_b200 import workloads as wl

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
KEYS = ("exit_reason", "outer_iters", "factorizations", "accepted", "trace_hash", "lambda", "ssr")
REP_WORDS = fk.REPORT_DTYPE.itemsize // 8


def _topology(w):
    return fk.Topology.from_arrays(w.n_vars, w.kind, w.idx, w.free_vars, w.rows)


def _pinned(a):
    import torch
    return torch.from_numpy(np.ascontiguousarray(a)).pin_memory()


def _batch(kind, w, ref, shared=True):
    """One batch of truss workload `w` for a call of `kind` ("system": fk_batch_system_solve on the raw values, "device":
    fk_batch_solve_device on the prepared ones): pinned input and output buffers, and the result of the one-call form,
    computed on `ref` (another topology object, so another pipeline)."""
    if kind == "system":
        par = w.raw_param[0] if shared else w.raw_param
        x, _, rep = ref.batch_system_solve(w.raw_vars, par, perturb=True, shared_param=shared)
        inputs = (w.raw_vars, par)
    else:
        v, p, _ = w.prepare()
        x, rep = ref.batch_solve(v, p)
        inputs = (v, p)
    bufs = tuple(_pinned(a) for a in inputs) + (_pinned(np.zeros_like(x)), _pinned(np.zeros((len(x), REP_WORDS))))
    return {"kind": kind, "shared": shared, "bufs": bufs, "x": x, "rep": rep}


def _ptrs(b):
    return [t.data_ptr() for t in b["bufs"]]


def _begin(topo, b):
    if b["kind"] == "system":
        return topo.batch_system_solve_begin(0, len(b["x"]), *_ptrs(b), shared_param=b["shared"])
    return topo.batch_solve_begin(0, len(b["x"]), *_ptrs(b))


def _wait(topo, b, token):
    (topo.batch_system_solve_wait if b["kind"] == "system" else topo.batch_solve_wait)(token)


def _check(b):
    assert np.array_equal(b["bufs"][2].numpy(), b["x"]), b["kind"]
    rep = b["bufs"][3].numpy().view(fk.REPORT_DTYPE).reshape(len(b["x"]))
    for key in KEYS:
        assert np.array_equal(rep[key], b["rep"][key]), (b["kind"], key)


def test_both_kinds_of_call_two_in_flight_on_one_pipeline():
    """System::solve-level and device-level halves alternate on one truss topology, two batches in flight, each with its own
    output buffers: every batch returns exactly what its one-call form returns."""
    n = 20000
    ws = [wl.truss(n, first=k * n) for k in range(5)]
    topo, ref = _topology(ws[0]), _topology(ws[0])
    batches = [_batch(kind, w, ref) for kind, w in zip(("system", "device", "system", "device", "system"), ws)]
    tokens = []
    for k, b in enumerate(batches):
        tokens.append(_begin(topo, b))
        if k >= 1:
            _wait(topo, batches[k - 1], tokens[k - 1])
    _wait(topo, batches[-1], tokens[-1])
    for b in batches:
        _check(b)


@pytest.mark.parametrize("kind", ["system", "device"])
def test_a_synchronous_call_between_two_halves(kind):
    """begin(A), a synchronous fk_batch_system_solve of B, begin(C), wait(A), wait(C): all three bit-identical to their one-call
    forms (C takes A's token slot), and a token no call has handed out is still rejected."""
    n = 20000
    ws = [wl.truss(n, first=k * n) for k in range(3)]
    topo, ref = _topology(ws[0]), _topology(ws[0])
    a, b, c = _batch(kind, ws[0], ref), _batch("system", ws[1], ref, shared=False), _batch(kind, ws[2], ref)
    ta = _begin(topo, a)
    topo.batch_system_solve_into(0, n, *_ptrs(b), shared_param=False)
    tc = _begin(topo, c)
    _wait(topo, a, ta)
    _wait(topo, c, tc)
    for x in (a, b, c):
        _check(x)
    with pytest.raises(fk.FiksiError):
        _wait(topo, c, tc + 1)


def test_plans_regrown_by_one_kind_of_call_serve_the_other():
    """A device-level call on a small batch sizes the plans; a System::solve-level call with larger chunks regrows them (the
    new plans get their unscaled-input and scale buffers from it); device-level calls on the large and the small batch and a
    System::solve-level call again run on whatever plans are there.  Every result equals its reference bit for bit."""
    small, large = 3000, 100000
    w = wl.truss(large)
    v, p, _ = w.prepare()
    topo, ref = _topology(w), _topology(w)
    want_small, want_large = ref.batch_solve(v[:small], p[:small]), ref.batch_solve(v, p)
    want_sys = ref.batch_system_solve(w.raw_vars, w.raw_param[0], perturb=True, shared_param=True)

    def same(got, want):
        assert all(np.array_equal(g, r) for g, r in zip(got[:-1], want[:-1]))
        for key in KEYS:
            assert np.array_equal(got[-1][key], want[-1][key]), key
    same(topo.batch_solve(v[:small], p[:small]), want_small)
    same(topo.batch_system_solve(w.raw_vars, w.raw_param[0], perturb=True, shared_param=True), want_sys)
    same(topo.batch_solve(v, p), want_large)
    same(topo.batch_solve(v[:small], p[:small]), want_small)
    same(topo.batch_system_solve(w.raw_vars, w.raw_param[0], perturb=True, shared_param=True), want_sys)


_TRACE_SCRIPT = r"""
import sys, numpy as np, torch
sys.path.insert(0, %r)
import fiksi_b200 as fk
from fiksi_b200 import workloads as wl
n_sys, n_dev = %d, %d
w = wl.truss(n_sys)
v, p, _ = w.prepare()
topo = fk.Topology.from_arrays(w.n_vars, w.kind, w.idx, w.free_vars, w.rows)
out = {}
for kind, n, ins in (("system", n_sys, (w.raw_vars, w.raw_param[0])), ("device", n_dev, (v[:n_dev], p[:n_dev]))):
    bufs = [torch.from_numpy(np.ascontiguousarray(a)).pin_memory() for a in ins]
    bufs += [torch.zeros((n, topo.info["n_free"]), dtype=torch.float64).pin_memory(),
             torch.zeros((n, fk.REPORT_DTYPE.itemsize // 8), dtype=torch.float64).pin_memory()]
    ptrs = [b.data_ptr() for b in bufs]
    if kind == "system":
        token = topo.batch_system_solve_begin(0, n, *ptrs, shared_param=True)
    else:
        token = topo.batch_solve_begin(0, n, *ptrs)
    out[kind + "_x"], out[kind + "_rep"] = bufs[2].numpy().copy(), bufs[3].numpy().copy()  # as _begin left them
    assert token != 0
    (topo.batch_system_solve_wait if kind == "system" else topo.batch_solve_wait)(token)
    print("[call done]", kind, file=sys.stderr, flush=True)
np.savez(sys.argv[1], **out)
"""


def test_trace_timeline_of_both_kinds_of_call(tmp_path):
    """FK_E2E_TRACE=1 (read once per process, hence the subprocess): one timeline line per chunk of every call, the _begin
    halves complete before returning (their outputs are in place when they return), _wait succeeds, and the results are
    those of this process, which runs untraced."""
    n_sys, n_dev = 30000, 12000
    w = wl.truss(n_sys)
    v, p, _ = w.prepare()
    topo = _topology(w)
    want = {"system": topo.batch_system_solve(w.raw_vars, w.raw_param[0], perturb=True, shared_param=True)[::2],
            "device": topo.batch_solve(v[:n_dev], p[:n_dev])}
    path = str(tmp_path / "trace.npz")
    env = dict(os.environ, FK_E2E_TRACE="1")
    env.pop("FK_E2E_CHUNKS", None)
    r = subprocess.run([sys.executable, "-c", _TRACE_SCRIPT % (ROOT, n_sys, n_dev), path], env=env, capture_output=True,
                       text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    got = np.load(path)
    for kind, n in (("system", n_sys), ("device", n_dev)):
        assert np.array_equal(got[kind + "_x"], want[kind][0]), kind
        rep = got[kind + "_rep"].view(fk.REPORT_DTYPE).reshape(n)
        for key in KEYS:
            assert np.array_equal(rep[key], want[kind][1][key]), (kind, key)
    # 2,048 sketches per chunk for both: the pipeline's minimum chunk (n / 16 and n / 8 are smaller), which is below half a
    # wave of the sketch kernel (at least 32 x 148 sketches) and so is not rounded to waves
    calls, lines = [], []
    for line in r.stderr.splitlines():
        if line.startswith("[e2e trace] chunk"):
            lines.append(int(line.split()[3].rstrip(":")))
        elif line.startswith("[call done]"):
            calls.append((line.split()[-1], lines))
            lines = []
    assert calls == [("system", list(range(math.ceil(n_sys / 2048)))), ("device", list(range(math.ceil(n_dev / 2048))))], r.stderr[-2000:]
