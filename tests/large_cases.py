"""Inputs of the large single-system parity cases (shared by the golden generator and the GPU tests):
case name -> (vars, kind, idx, param, free_vars, rows), everything numpy and deterministic."""
import numpy as np

from fiksi_b200 import workloads as wl

# Golden coordinate files stay well under 1 MB: a case with more than X_FULL_MAX free variables (512 KB)
# stores a seeded sample of X_SAMPLE_SIZE of them.
X_FULL_MAX = 65536
X_SAMPLE_SIZE = 16384


def x_sample_indices(n_free, size, seed):
    """Sorted indices of the converged coordinates that a sampled golden stores."""
    return np.sort(np.random.default_rng(seed).choice(n_free, size=size, replace=False))


def irregular_graph(n_pts, seed=11, ties=4, window=400, extent=100.0, noise=0.01):
    """Random points in sweep order, every point tied to its `ties` nearest earlier points inside a window
    (over-constrained, consistent, well conditioned); the first two points are fixed."""
    rng = np.random.default_rng(seed)
    pts = rng.uniform(0.0, extent, size=(n_pts, 2))
    order = np.argsort(pts[:, 0] + 0.37 * pts[:, 1], kind="stable")
    pts = pts[order]
    edges = [(0, 1)]
    for k in range(2, n_pts):
        lo = max(0, k - window)
        d = np.sum((pts[lo:k] - pts[k]) ** 2, axis=1)
        near = np.argsort(d, kind="stable")[:ties] + lo
        edges += [(int(a), k) for a in near]
    kind = np.ones(len(edges), np.uint8)
    idx = np.array([[2 * a, 2 * b, 0, 0] for a, b in edges], np.uint32)
    dist = np.array([np.hypot(*(pts[a] - pts[b])) for a, b in edges])
    noisy = pts + rng.uniform(-noise, noise, size=pts.shape)
    free_vars = np.arange(4, 2 * n_pts, dtype=np.uint32)
    return wl.Workload("irregular", kind, idx, free_vars, np.arange(len(edges)), noisy.reshape(1, -1), dist.reshape(1, -1))


def build_case(name):
    if name.startswith("lattice"):
        nx, ny = (int(t) for t in name[len("lattice"):].split("x"))
        w = wl.lattice(nx, ny)
    elif name.startswith("irregular"):
        w = irregular_graph(int(name[len("irregular"):]))
    else:
        raise ValueError(name)
    v, p, _scale = w.prepare()
    return v[0], w.kind, w.idx, p[0], w.free_vars, w.rows
