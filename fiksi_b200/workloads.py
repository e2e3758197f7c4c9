"""Synthetic sketch generators for BASELINE.json's configs (SURVEY.md App. D) and the host-side
pre/post-processing of ``assemble::solve`` for batches of single-component sketches.

Everything here is input generation and bookkeeping in numpy: PRNG streams, coordinates, the
flattened topology arrays (kinds / indices / free set / rows), and the bit-exact restatement of
the reference's scale + perturbation step (fiksi/src/assemble/mod.rs:32-124) vectorised over
sketches so that 65,536- and 1,000,000-sketch batches can be prepared in seconds.  No residual,
Jacobian, ordering or factorisation is computed here.
"""
from __future__ import annotations

import math

import numpy as np

MASK64 = np.uint64(0xFFFFFFFFFFFFFFFF)


def splitmix64(seed, n_draws):
    """splitmix64 streams: seed[k] -> n_draws uint64 each.  Returns [len(seed)][n_draws]."""
    with np.errstate(over="ignore"):
        state = np.asarray(seed, dtype=np.uint64).copy()
        out = np.empty((state.shape[0], n_draws), dtype=np.uint64)
        for d in range(n_draws):
            state = state + np.uint64(0x9E3779B97F4A7C15)
            z = state.copy()
            z = (z ^ (z >> np.uint64(30))) * np.uint64(0xBF58476D1CE4E5B9)
            z = (z ^ (z >> np.uint64(27))) * np.uint64(0x94D049BB133111EB)
            out[:, d] = z ^ (z >> np.uint64(31))
    return out


def uniform_pm1(bits):
    """Uniform in [-1, 1) from the top 53 bits (SURVEY App. D)."""
    return (bits >> np.uint64(11)).astype(np.float64) * (2.0 / 9007199254740992.0) - 1.0


# ---- LCG of the reference (fiksi/src/rand.rs:24-39), used for the perturbation stream ---------
def lcg_f64(seed, n):
    out = np.empty(n, dtype=np.float64)
    state = seed & 0xFFFFFFFF
    c = 1.0 / 4294967295.0
    for k in range(n):
        state = (state * 1664525 + 1013904223) & 0xFFFFFFFF
        out[k] = c * float(state)
    return out


class Workload:
    """A uniform batch: one topology + per-sketch raw variables / parameters."""

    def __init__(self, name, kind, idx, free_vars, rows, raw_vars, raw_param, perturb_vars=None):
        self.name = name
        # variables that draw from the solve's RNG stream, ascending (all free variables of the
        # system's components in component order); defaults to this problem's free variables
        self.perturb_vars = None if perturb_vars is None else np.ascontiguousarray(perturb_vars, dtype=np.uint32)
        self.kind = np.ascontiguousarray(kind, dtype=np.uint8)
        self.idx = np.ascontiguousarray(idx, dtype=np.uint32).reshape(-1, 4)
        self.free_vars = np.ascontiguousarray(free_vars, dtype=np.uint32)
        self.rows = np.ascontiguousarray(rows, dtype=np.uint32)
        self.raw_vars = np.ascontiguousarray(raw_vars, dtype=np.float64)    # [n][n_vars]
        self.raw_param = np.ascontiguousarray(raw_param, dtype=np.float64)  # [n][n_expr]

    @property
    def n(self):
        return self.raw_vars.shape[0]

    @property
    def n_vars(self):
        return self.raw_vars.shape[1]

    def prepare(self, perturb=True):
        """Scale + perturb exactly as assemble::solve does for a system whose elements all sit in
        one connected component (fiksi/src/assemble/mod.rs:32-124).  Returns (vars, param, scale)."""
        v, p = self.raw_vars, self.raw_param
        is_len = (self.kind == 1) | (self.kind == 4)  # PPD / PLD distances take part in the scale
        s = np.zeros(self.n)
        for k in range(v.shape[1]):                    # sequential, left to right (utils.rs:12-19)
            s = s + v[:, k] * v[:, k]
        cnt = v.shape[1]
        for e in np.nonzero(is_len)[0]:
            s = s + p[:, e] * p[:, e]
            cnt += 1
        scale = np.sqrt(s / float(cnt))
        recip = 1.0 / scale
        vs = v * recip[:, None]
        ps = p.copy()
        ps[:, is_len] = recip[:, None] * p[:, is_len]
        if perturb:
            order = self.free_vars if self.perturb_vars is None else self.perturb_vars
            draws = lcg_f64(42, 2 * len(order))   # Rng::from_seed(42) per solve (mod.rs:47)
            c1, c2 = 1.0 / 8196.0, 1.0 / 65568.0
            for j, fv in enumerate(order if self.perturb_vars is not None else np.sort(order)):  # ascending BTreeSet order
                col = vs[:, fv]
                vs[:, fv] = col + (col * c1 * draws[2 * j] + c2 * draws[2 * j + 1])
        return np.ascontiguousarray(vs), np.ascontiguousarray(ps), scale

    def write_back(self, raw_vars, free_values, scale):
        """system.variables[var] = system_scale * x[k] (assemble/mod.rs:161-166)."""
        out = raw_vars.copy()
        out[:, self.free_vars] = scale[:, None] * free_values
        return out


def truss(n_sketches, n_points=20, noise=0.05, seed=0xF1C50002, first=0):
    """Config 2: zig-zag equilateral strip, Henneberg edges (0,1), then (i,i-1),(i,i-2)."""
    q = np.array([[0.5 * i, (i % 2) * math.sqrt(3.0) / 2.0] for i in range(n_points)])
    edges = [(0, 1)] + [e for i in range(2, n_points) for e in ((i, i - 1), (i, i - 2))]
    dist = np.array([math.hypot(*(q[a] - q[b])) for a, b in edges])
    ids = np.arange(first, first + n_sketches, dtype=np.uint64)
    u = uniform_pm1(splitmix64(np.uint64(seed) + ids, 2 * n_points))
    raw = q.reshape(1, -1) + noise * u
    kind = np.full(len(edges), 1, np.uint8)
    idx = np.zeros((len(edges), 4), np.uint32)
    for e, (a, b) in enumerate(edges):
        idx[e, 0], idx[e, 1] = 2 * a, 2 * b
    return Workload(f"truss{n_points}", kind, idx, np.arange(2 * n_points), np.arange(len(edges)), raw,
                    np.tile(dist, (n_sketches, 1)))


RAD = math.pi / 180.0

# circle_triangle_line (examples/fiksi_svg_tests/src/main.rs:12-45): the five points are created
# first (variables 0..9), the radius Length after the triangle constraints (variable 10);
# expressions in file order.
_CTL_BASE = np.array([10., 0., 20., 10., 30., -10., -40., -50., 40., -50., 5.])
_CTL_KIND = [2, 2, 1, 10, 7, 3, 1, 1]
_CTL_IDX = [[0, 2, 4, 0], [2, 4, 0, 0], [0, 2, 0, 0], [0, 2, 4, 10], [0, 4, 6, 8], [4, 6, 8, 0], [4, 6, 0, 0], [6, 8, 0, 0]]
_CTL_PARAM = np.array([40. * RAD, 70. * RAD, 70., 0., -90. * RAD, 0., 40., 80.])
_CTL_LEN = np.array([0, 0, 1, 0, 0, 0, 1, 1], dtype=bool)


def cad_mix(n_sketches, seed=0xF1C50004, first=0):
    """Config 4: circle_triangle_line topology; per sketch a scale s in [0.5, 2], coordinates
    s*(c + 0.05*|c|*U), distances s*d, radius 5s."""
    ids = np.arange(first, first + n_sketches, dtype=np.uint64)
    bits = splitmix64(np.uint64(seed) + ids, 11)
    u = uniform_pm1(bits)
    s = 1.25 + 0.75 * u[:, 10]
    coords = np.tile(_CTL_BASE, (n_sketches, 1))
    coords[:, :10] = coords[:, :10] + 0.05 * np.abs(coords[:, :10]) * u[:, :10]
    raw = coords * s[:, None]
    param = np.tile(_CTL_PARAM, (n_sketches, 1))
    param[:, _CTL_LEN] = param[:, _CTL_LEN] * s[:, None]
    return Workload("cad_mix", _CTL_KIND, _CTL_IDX, np.arange(11), np.arange(8), raw, param)


def lattice(nx=400, ny=250, noise=0.02, seed=0xF1C50003, n_sketches=1, first=0):
    """Config 3: nx*ny unit lattice, raster order; PPD to left, up, up-left neighbours.  Sketch k of a batch draws its
    noise from splitmix64(seed + first + k) (as truss does); the default single sketch is config 3 itself."""
    pts = np.array([[x, y] for y in range(ny) for x in range(nx)], dtype=np.float64)
    kind, idx, dist = [], [], []
    for y in range(ny):
        for x in range(nx):
            i = y * nx + x
            for dx, dy in ((-1, 0), (0, -1), (-1, -1)):
                xx, yy = x + dx, y + dy
                if xx < 0 or yy < 0:
                    continue
                j = yy * nx + xx
                kind.append(1)
                idx.append([2 * i, 2 * j, 0, 0])
                dist.append(math.hypot(dx, dy))
    n_pts = nx * ny
    ids = np.arange(first, first + n_sketches, dtype=np.uint64)
    u = uniform_pm1(splitmix64(np.uint64(seed) + ids, 2 * n_pts))
    raw = pts.reshape(1, -1) + noise * u
    return Workload(f"lattice{nx}x{ny}", kind, idx, np.arange(2 * n_pts), np.arange(len(kind)), raw,
                    np.tile(np.array(dist), (n_sketches, 1)))


def hinged_triangles(n_triangles, n_sketches=1):
    """fiksi/benches/fiksi_bench.rs:15-40."""
    coords = [0., 0.]
    kind, idx, dist = [], [], []
    for k in range(n_triangles):
        p1, p2 = len(coords), len(coords) + 2
        coords += [-1., float(k), 1., float(k)]
        for a, b, d in ((0, p1, 2.), (0, p2, 2.), (p1, p2, 3.)):
            kind.append(1)
            idx.append([a, b, 0, 0])
            dist.append(d)
    raw = np.tile(np.array(coords), (n_sketches, 1))
    return Workload(f"hinged{n_triangles}", kind, idx, np.arange(len(coords)), np.arange(len(kind)), raw,
                    np.tile(np.array(dist), (n_sketches, 1)))


def _ppd(edges):
    kind = [1] * len(edges)
    idx = [[2 * a, 2 * b, 0, 0] for a, b in edges]
    return kind, idx


def stress_families(n_each=8192, seed=0xF1C50005):
    """Config 5: under-/over-constrained, singular and badly scaled sketches built from the
    reference's own scenarios (SURVEY App. D), each varied per sketch by a random size factor and a
    little coordinate noise.  Returns [(family name, Workload)]."""
    ids = np.arange(n_each, dtype=np.uint64)
    out = []

    def draws(k, n_draws):
        return uniform_pm1(splitmix64(np.uint64(seed + 0x1000 * k) + ids, n_draws))

    def family(k, name, pts, kind, idx, param, is_len, free=None, noise=1e-3, size=(0.5, 2.0), perturb_vars=None):
        pts = np.asarray(pts, dtype=np.float64).reshape(-1)
        u = draws(k, len(pts) + 1)
        s = 0.5 * (size[0] + size[1]) + 0.5 * (size[1] - size[0]) * u[:, -1]
        raw = (pts.reshape(1, -1) + noise * u[:, :-1]) * s[:, None]
        par = np.tile(np.asarray(param, dtype=np.float64), (n_each, 1))
        is_len = np.asarray(is_len, dtype=bool)
        par[:, is_len] = par[:, is_len] * s[:, None]
        free = np.arange(len(pts)) if free is None else np.asarray(free)
        out.append((name, Workload(name, kind, idx, free, np.arange(len(kind)), raw, par, perturb_vars=perturb_vars)))

    tri = [(0, 1), (0, 2), (1, 2)]
    # 1 collinear singular start (tests/singular.rs:19-40): exactly collinear, no noise
    k, i = _ppd(tri)
    family(1, "collinear_singular_start", [0, 0, 3, 0, 6, 0], k, i, [1., 1., 1.], [1, 1, 1], noise=0.0)
    # 2 impossible angles + incidence (tests/basic.rs:56-87)
    family(2, "impossible_angles_incidence", [0, 0, 1, .5, 2, 1, 3, 1.5], [2, 2, 2, 3],
           [[0, 2, 4, 0], [2, 4, 0, 0], [4, 0, 2, 0], [2, 4, 6, 0]], [40 * RAD, 80 * RAD, 100 * RAD, 0.], [0, 0, 0, 0])
    # 3 under-constrained triangle (tests/basic.rs:36-52)
    family(3, "underconstrained_triangle", [0, 0, 1, .5, 2, 1], [2, 2], [[0, 2, 4, 0], [2, 4, 0, 0]], [40 * RAD, 80 * RAD], [0, 0])
    # 4 over-constrained four points, six distances, one inconsistent (tests/basic.rs:90-112)
    k, i = _ppd([(0, 1), (0, 2), (1, 3), (2, 3), (1, 2), (0, 3)])
    family(4, "overconstrained_inconsistent", [.123, .1, 1.2, 0, -.5, 1.1, 1.599, 1.2], k, i, [1., 1.5, 1.7, 1.2, 2., 5.], [1] * 6)
    # 5 duplicated constraint: rank-deficient rows
    k, i = _ppd(tri + [(1, 2)])
    family(5, "duplicated_constraint", [0, 0, 1, .5, 2, 1], k, i, [1., 1., 1., 1.], [1] * 4)
    # 6 large magnitude 1e20 (tests/magnitude.rs:13-36)
    k, i = _ppd(tri)
    family(6, "scale_1e20", np.array([1.5, 6.5, 3.2, .8, 2.2, -1.5]) * 1e20, k, i, np.array([5., 3., 4.]) * 1e20, [1] * 3, noise=1e17)
    # 7 near-degenerate isosceles triangle at 1e13 (tests/magnitude.rs:143-166)
    k, i = _ppd([(0, 1), (1, 2), (0, 2)])
    family(7, "near_degenerate_1e13", [1.5e13, 6.5e13, 3.2e13, .8e13, 2.2, -1.5], k, i, [4e13 + 1., 4e13 + 1., 1.], [1] * 3,
           noise=0.0, size=(1.0, 1.0))
    # 8 triangle with a fixed point (tests/fixed.rs:9-43)
    k, i = _ppd(tri)
    family(8, "fixed_point_triangle", [0, 0, 1, .5, 2, 1], k, i, [1., 1., 1.], [1] * 3, free=[0, 1, 4, 5])
    # 9 two disconnected components in one system (tests/basic.rs:152-170): two problems per sketch
    # that share the variables and the solve's RNG stream
    k, i = _ppd([(0, 1), (2, 3)])
    pts = [.123, .1, 1.2, 0, -.5, 1.1, 1.599, 1.2]
    family(9, "two_components_a", pts, k, i, [1., 1.2], [1, 1], free=[0, 1, 2, 3], perturb_vars=np.arange(8))
    family(9, "two_components_b", pts, k, i, [1., 1.2], [1, 1], free=[4, 5, 6, 7], perturb_vars=np.arange(8))
    out[-2][1].rows = np.array([0], dtype=np.uint32)
    out[-1][1].rows = np.array([1], dtype=np.uint32)
    # 10 coincident points under a distance constraint: 1/0 -> NaN, the reference never returns
    k, i = _ppd([(0, 1)])
    family(10, "nan_coincident_points", [1, 1, 1, 1], k, i, [1.], [1], noise=0.0)
    return out
