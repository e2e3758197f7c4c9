"""Lists of different drawings for fk_systems_solve / solve_systems: every builder takes the System class (fk.System or
oracle.System) and returns one drawing, so that a test or a benchmark can build the same list twice."""
import numpy as np

import cad_drawings as cd
import scenarios as sc
from fiksi_b200 import workloads as wl


def add_ppd(s, w, k=0):
    """Workload w's sketch k (all point-point distances) appended to s as its own component."""
    raw = w.raw_vars[k]
    pts = [s.add_point(float(raw[2 * i]), float(raw[2 * i + 1])) for i in range(len(raw) // 2)]
    for e in range(len(w.kind)):
        s.point_point_distance(pts[int(w.idx[e][0]) // 2], pts[int(w.idx[e][1]) // 2], float(w.raw_param[k][e]))
    return pts


def scenario(name):
    return lambda S: sc.ALL[name](S)["s"]


def empty(S):
    return S()


def lone_point(S):
    s = S()
    s.add_point(1.0, 2.0)
    return s


def ppd(w, k):
    """Sketch k of the point-point-distance workload w as a drawing of its own."""
    def build(S):
        s = S()
        add_ppd(s, w, k)
        return s
    return build


def hinged_chain(n, seed):
    """hinged_triangles_bench with n triangles whose points sit at seeded offsets."""
    def build(S):
        rng = np.random.default_rng(seed)
        s = S()
        hinge = s.add_point(0.0, 0.0)
        for k in range(n):
            dx, dy = 0.2 * rng.standard_normal(2)
            p1, p2 = s.add_point(-1.0 + dx, k + dy), s.add_point(1.0 - dx, k - dy)
            s.point_point_distance(hinge, p1, 2.0)
            s.point_point_distance(hinge, p2, 2.0)
            s.point_point_distance(p1, p2, 3.0)
        return s
    return build


def scaled_ctl(seed):
    """circle_triangle_line at a seeded scale with seeded noise on its points."""
    def build(S):
        rng = np.random.default_rng(seed)
        return sc.circle_triangle_line(S, scale=float(rng.uniform(0.5, 20.0)), noise=list(rng.uniform(-1, 1, 10)))["s"]
    return build


def cad(nx, ny, seed):
    """cad_grid with the first seed from `seed` on (steps of 7919) whose ground truth keeps every angle off +-pi."""
    def build(S):
        for k in range(100):
            try:
                return cd.cad_grid(S, nx, ny, seed=seed + 7919 * k)["s"]
            except AssertionError:
                continue
        raise ValueError(f"no usable cad_grid seed from {seed}")
    return build


def cad_drawing(S):
    """Three components: a mixed-kind CAD grid on path 1, a smaller one with shared vertices on path 0, a single triangle."""
    s = S()
    cd.cad_grid(lambda: s, *cd.PATH1_LOW, seed=3)
    cd.cad_grid(lambda: s, *cd.PATH0, seed=4)
    sc.single_triangle(lambda: s)
    return s


def lattice_drawing(nx, ny):
    def build(S):
        s = S()
        add_ppd(s, wl.lattice(nx, ny))
        sc.single_triangle(lambda: s)
        return s
    return build


def mixed(seed):
    """The equality mix: every scenario (stale-index and fixed-point drawings among them), an empty drawing, a lone point,
    CAD drawings, 80 different sketches of one truss (one uniform structure) and singleton structures (heterogeneous),
    shuffled."""
    truss = wl.truss(80, 20)
    b = [scenario(name) for name in sorted(sc.ALL)]
    b += [empty, lone_point, cad_drawing, cad(*cd.PATH0, seed=9)]
    b += [ppd(truss, k) for k in range(80)]
    b += [hinged_chain(n, seed=100 + n) for n in (1, 3, 5, 7)] + [scaled_ctl(200 + k) for k in range(3)]
    order = np.random.default_rng(seed).permutation(len(b))
    return [b[i] for i in order]
