"""Mixed-kind CAD drawings with a known exact solution, written against the System interface shared by
``oracle.System`` and ``fiksi_b200.System`` (as tests/scenarios.py is).

``cad_grid`` lays out a jittered, triangulated grid of points, ties it together with distances and adds, cell by cell,
every constraint-level kind: coincidences (kind 0 rows), angles at a corner, point-line incidences and distances,
circles with a free radius (point on circle, line tangency), segment-length equalities between adjacent and far-apart
segments, line-line angles, parallels and perpendiculars.  Every parameter is measured on the ground truth, and every
auxiliary point is placed where its constraints hold, so the ground truth solves the drawing.  Two grid points are
fixed, which removes the rigid motions: J has full column rank there.

With ``shared_vertices=True`` the rows between adjacent edges name the shared corner twice (the Jacobian entries of
such a row are sums); with ``shared_vertices=False`` no row names a free variable twice, so the sketch-per-thread
kernel takes the drawing."""
import math

import numpy as np

H = 1.0          # grid spacing of the ground truth
JITTER = 0.15    # grid points sit within +-JITTER * H of the lattice
ANGLE_MARGIN = 0.1  # every angle row's ground-truth angle stays this far (rad) from +-pi

# (nx, ny) of the drawings the path tests use; tests/test_gpu_mixed_kinds.py pins the path, tile and shared-memory
# footprint each one reaches.
PATH0 = (4, 4)             # the smallest grid with every kind: tile kernel with shared vertices, sketch kernel without
PATH1_LOW = (8, 7)         # one CTA per sketch, just above the 24 KB of the tile kernel
PATH1_MID = (12, 11)
PATH1_HIGH = (16, 17)      # just under 200 KB
PATH2_NATURAL = (26, 26)   # global sparse path by size, ~2,100 free variables
FAR_ROWS = 3               # segment-length equalities between far-apart cells (widen the fronts)


def _rot(v, a):
    c, s = math.cos(a), math.sin(a)
    return np.array([c * v[0] - s * v[1], s * v[0] + c * v[1]])


def _angle(u, w):
    """Signed angle from u to w in (-pi, pi]."""
    return math.atan2(u[0] * w[1] - u[1] * w[0], u[0] * w[0] + u[1] * w[1])


def _cross(u, w):
    return float(u[0] * w[1] - u[1] * w[0])


def cad_grid(S, nx, ny, *, seed, shared_vertices=True):
    """One connected drawing on an nx x ny grid (nx, ny >= 3).  Returns dict(s, points, truth, fixed, constraints,
    kinds, params): `truth` maps every point handle to its ground-truth position, `kinds` / `params` list the
    constraint-level kind and raw parameter of each constraint in creation order."""
    assert nx >= 3 and ny >= 3
    rng = np.random.default_rng(seed)
    s = S()
    truth, kinds, params, cons = {}, [], [], []

    def point(xy):
        xy = np.asarray(xy, dtype=np.float64)
        p = s.add_point(float(xy[0]), float(xy[1]))
        truth[p] = xy
        return p

    def add(kind, param, c):
        kinds.append(kind)
        params.append(param)
        cons.append(c)

    def dist(a, b):
        d = float(np.hypot(*(truth[a] - truth[b])))
        add(1, d, s.point_point_distance(a, b, d))

    def line(a, b):
        return s.add_line(a, b)

    def angle3(a, b, c):  # kind 2: angle at b from (a - b) to (c - b)
        ang = _angle(truth[a] - truth[b], truth[c] - truth[b])
        assert abs(ang) < math.pi - ANGLE_MARGIN
        add(2, ang, s.point_point_point_angle(a, b, c, ang))

    def angle_ll(a, b, c, d):  # kind 7: angle from (b - a) to (d - c)
        ang = _angle(truth[b] - truth[a], truth[d] - truth[c])
        assert abs(ang) < math.pi - ANGLE_MARGIN
        add(7, ang, s.line_line_angle(line(a, b), line(c, d), ang))

    grid = [[None] * nx for _ in range(ny)]
    for j in range(ny):
        for i in range(nx):
            grid[j][i] = point([i * H + JITTER * H * rng.uniform(-1, 1), j * H + JITTER * H * rng.uniform(-1, 1)])
    fixed = [int(grid[0][0]), int(grid[0][2])]  # no row between them: every row has a free slot
    for p in fixed:
        s.fix(p)

    # the triangulated grid, point by point in raster order: every constraint touches the component built so far
    cells = []
    for j in range(ny):
        for i in range(nx):
            k = grid[j][i]
            if i > 0:
                dist(grid[j][i - 1], k)
            if j > 0:
                dist(grid[j - 1][i], k)
            if i > 0 and j > 0:
                dist(grid[j - 1][i - 1], k)
                cells.append((i, j))

    # per cell (corners a b / d c, counter-clockwise from the lower left) one feature, cycling through the kinds
    for t, (i, j) in enumerate(cells):
        a, b, c, d = grid[j - 1][i - 1], grid[j - 1][i], grid[j][i], grid[j][i - 1]
        A, B, C, D = (truth[q] for q in (a, b, c, d))
        f = t % 10
        if f == 0:  # kind 2 at a corner, kind 0 rows: an extra point coincident with c that a distance reads
            angle3(a, b, c)
            e = point(C)
            add(0, 0.0, s.point_point_coincidence(e, c))
            dist(e, a)
        elif f == 1:  # kind 7 between adjacent edges (shared corner b) or opposite edges
            if shared_vertices:
                angle_ll(a, b, b, c)
            else:
                angle_ll(a, b, d, c)
        elif f == 2:  # kind 9: an extra point on the perpendicular to ab through b (or through c)
            base = b if shared_vertices else c
            e = point(truth[base] + 0.6 * _rot(B - A, math.pi / 2))
            add(9, 0.0, s.line_line_perpendicularity(line(a, b), line(base, e)))
            dist(base, e)
        elif f == 3:  # kind 8: an extra point on the parallel to ab through b (collinear) or through d
            base = b if shared_vertices else d
            e = point(truth[base] + 0.7 * (B - A))
            add(8, 0.0, s.line_line_parallelism(line(a, b), line(base, e)))
            dist(base, e)
        elif f == 4:  # kind 6 between adjacent segments ab, be (or ab, ce); kind 2 fixes the direction of e
            base = b if shared_vertices else c
            e = point(truth[base] + _rot(B - A, 0.9))
            add(6, 0.0, s.segment_segment_length_equality(a, b, base, e))
            angle3(c if shared_vertices else b, base, e)
        elif f == 5:  # kind 3: an extra point on the diagonal ac, kind 4: d's signed distance to line ab
            e = point(A + 0.3 * (C - A))
            add(3, 0.0, s.point_line_incidence(e, line(a, c)))
            dist(a, e)
            sd = _cross(B - A, D - A) / float(np.hypot(*(B - A)))
            add(4, sd, s.point_line_distance(d, line(a, b), sd))
        elif f == 6:  # kind 5: a circle about c through d, its radius a free Length
            r = s.add_length(float(np.hypot(*(D - C))))
            add(5, 0.0, s.point_circle_incidence(d, s.add_circle(c, r)))
        elif f == 7:  # kind 10: a circle about d tangent to line ab
            r = s.add_length(abs(_cross(B - A, D - A)) / float(np.hypot(*(B - A))))
            add(10, 0.0, s.line_circle_tangency(line(a, b), s.add_circle(d, r)))
        elif f == 8:  # kind 7 between the two diagonals of the cell
            angle_ll(a, c, b, d)
        else:  # kind 4: a's signed distance to line bc
            sd = _cross(C - B, A - B) / float(np.hypot(*(C - B)))
            add(4, sd, s.point_line_distance(a, line(b, c), sd))

    # a few segment-length equalities between far-apart cells: segment ab of a cell near the start against a new
    # segment hung off a cell near the end (a kind-2 angle fixes its direction)
    for q in range(FAR_ROWS):
        i0, j0 = 1 + q % (nx - 1), 1
        i1, j1 = nx - 1 - q % (nx - 1), ny - 1
        a, b = grid[j0 - 1][i0 - 1], grid[j0 - 1][i0]
        p, c = grid[j1 - 1][i1], grid[j1][i1]
        e = point(truth[c] + _rot(truth[b] - truth[a], 2.0 + 0.3 * q))
        add(6, 0.0, s.segment_segment_length_equality(a, b, c, e))
        angle3(p, c, e)
    return dict(s=s, points=list(truth), truth=truth, fixed=fixed, constraints=cons, kinds=kinds, params=params)


# ---- flattened arrays ----------------------------------------------------------------------------------------------
def prepared(nx, ny, *, seed, shared_vertices=True):
    """The drawing's one component as System::solve flattens it (scaled, unperturbed): dict(keep=(vars, kind, idx,
    param, free_vars, rows), scale, spacing (H in scaled units), drawing (cad_grid's dict over oracle.System))."""
    import oracle
    d = cad_grid(oracle.System, nx, ny, seed=seed, shared_vertices=shared_vertices)
    (problem, scale, keep), = d["s"].prepare(perturb=False)
    return dict(keep=keep, scale=scale, spacing=H / scale, drawing=d, problem=problem)


def start_variants(prep, n, seed, amount=1e-2):
    """n start rows of the prepared problem: seeded uniform noise of +-amount grid spacings on every free entry (scaled
    units), the parameters unchanged.  Returns (vars [n][n_vars], param [n][n_expr])."""
    vars_, kind, idx, param, free_vars, rows = prep["keep"]
    rng = np.random.default_rng(seed)
    v = np.tile(np.asarray(vars_, np.float64), (n, 1))
    v[:, free_vars] += amount * prep["spacing"] * rng.uniform(-1.0, 1.0, size=(n, len(free_vars)))
    return np.ascontiguousarray(v), np.ascontiguousarray(np.tile(np.asarray(param, np.float64), (n, 1)))


def workload(nx, ny, n, *, seed, shared_vertices=True, amount=1e-2):
    """The drawing as a uniform batch of n sketches (fiksi_b200.workloads.Workload over raw, unscaled numbers): sketch k
    starts from the ground truth plus seeded noise of +-amount grid spacings on the free coordinates."""
    from fiksi_b200 import workloads as wl
    prep = prepared(nx, ny, seed=seed, shared_vertices=shared_vertices)
    vars_, kind, idx, param, free_vars, rows = prep["keep"]
    d = prep["drawing"]
    raw = np.tile(d["s"].variables, (n, 1))
    raw[:, free_vars] += amount * H * np.random.default_rng(seed + 1).uniform(-1.0, 1.0, size=(n, len(free_vars)))
    raw_param = np.repeat(d["params"], [2 if k == 0 else 1 for k in d["kinds"]]).astype(np.float64)
    name = f"cad{nx}x{ny}{'' if shared_vertices else 'd'}"
    return wl.Workload(name, kind, idx, free_vars, rows, raw, np.tile(raw_param, (n, 1)))


def duplicated_free_slots(keep):
    """Number of rows that name some free variable in two slots."""
    vars_, kind, idx, param, free_vars, rows = keep
    free = set(int(q) for q in free_vars)
    out = 0
    for r in rows:
        vi = slot_vars(int(kind[r]), idx[r])
        fv = [q for q in vi if q in free]
        out += len(fv) != len(set(fv))
    return out


def slot_vars(kind, idx):
    """Variable index of every slot of one expression (expressions.rs:48-182)."""
    i = [int(x) for x in idx]
    pt = lambda q: [q, q + 1]  # noqa: E731
    if kind == 0:
        return [i[0], i[1]]
    if kind == 1:
        return pt(i[0]) + pt(i[1])
    if kind in (2, 3, 4):
        return pt(i[0]) + pt(i[1]) + pt(i[2])
    if kind == 5:
        return pt(i[0]) + pt(i[1]) + [i[2]]
    if kind in (6, 7, 8, 9):
        return pt(i[0]) + pt(i[1]) + pt(i[2]) + pt(i[3])
    if kind == 10:
        return pt(i[0]) + pt(i[1]) + pt(i[2]) + [i[3]]
    raise ValueError(kind)
