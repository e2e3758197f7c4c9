"""workloads.lattice with several sketches: the default call stays config 3's single sketch, byte for byte, and sketch 0 of a
batch is that sketch."""
import math

import numpy as np

from fiksi_b200 import workloads as wl


def _single_sketch_arrays(nx, ny, noise=0.02, seed=0xF1C50003):
    """The single-sketch lattice as config 3, the goldens and the large-system tests have always generated it."""
    pts = np.array([[x, y] for y in range(ny) for x in range(nx)], dtype=np.float64)
    kind, idx, dist = [], [], []
    for y in range(ny):
        for x in range(nx):
            i = y * nx + x
            for dx, dy in ((-1, 0), (0, -1), (-1, -1)):
                xx, yy = x + dx, y + dy
                if xx < 0 or yy < 0:
                    continue
                kind.append(1)
                idx.append([2 * i, 2 * (yy * nx + xx), 0, 0])
                dist.append(math.hypot(dx, dy))
    u = wl.uniform_pm1(wl.splitmix64(np.array([seed], dtype=np.uint64), 2 * nx * ny))
    return np.array(kind, np.uint8), np.array(idx, np.uint32), pts.reshape(1, -1) + noise * u, np.array(dist).reshape(1, -1)


def test_default_lattice_is_unchanged():
    for nx, ny in ((5, 4), (30, 20), (64, 50)):
        kind, idx, raw, dist = _single_sketch_arrays(nx, ny)
        w = wl.lattice(nx, ny)
        assert w.kind.tobytes() == kind.tobytes() and w.idx.tobytes() == idx.tobytes()
        assert w.raw_vars.tobytes() == raw.tobytes() and w.raw_param.tobytes() == dist.tobytes()
        assert np.array_equal(w.free_vars, np.arange(2 * nx * ny)) and np.array_equal(w.rows, np.arange(len(kind)))


def test_batch_sketch_zero_is_the_single_sketch_and_the_others_differ():
    one = wl.lattice(12, 9)
    many = wl.lattice(12, 9, n_sketches=5)
    assert many.raw_vars.shape == (5, one.n_vars) and many.raw_param.shape == (5, one.raw_param.shape[1])
    assert many.raw_vars[0].tobytes() == one.raw_vars[0].tobytes()
    assert all(many.raw_param[k].tobytes() == one.raw_param[0].tobytes() for k in range(5))
    assert len({many.raw_vars[k].tobytes() for k in range(5)}) == 5
    # sketch k of a batch starting at `first` is sketch first + k of a batch starting at 0
    tail = wl.lattice(12, 9, n_sketches=2, first=3)
    assert tail.raw_vars.tobytes() == many.raw_vars[3:5].tobytes()
