"""Independent model of mr_triangulate_earclip (the rules of include/myrenderer_b200.h), its named wrong variants, and
the case generators of tests/test_earclip_cpu.py and tests/test_gpu_earclip.py.

The model works on one polygon (an [n, 2] float32 array) and returns (status, triangles as corner-id triples).  Its
orientation is exact rational arithmetic (fractions.Fraction); its ring walk is a plain loop over Python lists."""
from fractions import Fraction

import numpy as np

NO_EAR = 256
F32 = np.float32


def orient_exact(a, b, c):
    ax, ay, bx, by, cx, cy = (Fraction(float(v)) for v in (a[0], a[1], b[0], b[1], c[0], c[1]))
    d = (bx - ax) * (cy - ay) - (by - ay) * (cx - ax)
    return (d > 0) - (d < 0)


def orient_f32(a, b, c):
    with np.errstate(all="ignore"):
        d = F32(F32(F32(b[0]) - F32(a[0])) * F32(F32(c[1]) - F32(a[1]))) - F32(F32(F32(b[1]) - F32(a[1])) * F32(F32(c[0]) - F32(a[0])))
    return int(d > 0) - int(d < 0)


def orient_f64(a, b, c):
    d = (float(b[0]) - float(a[0])) * (float(c[1]) - float(a[1])) - (float(b[1]) - float(a[1])) * (float(c[0]) - float(a[0]))
    return (d > 0) - (d < 0)


VARIANTS = (
    "orient_f32",            # orient in f32
    "orient_f64",            # naive f64 determinant, no exact fallback
    "convex_blockers",       # strictly convex vertices counted as blockers
    "straight_not_blocker",  # orient = 0 vertices not counted as blockers
    "open_triangle",         # open instead of closed triangle
    "no_point_eq",           # no point-equality exclusion
    "cursor_at_q",           # cursor continues at q after an ear
    "no_zero_edge",          # no zero-length-edge rule
    "winding_shoelace",      # winding from an f64 shoelace sum
    "emit_ignores_winding",  # (p, c, q) whatever the winding
    "fallback_clips_next",   # the no-ear fallback clips next(c)
    "fallback_no_bit",       # the no-ear fallback does not set the bit
    "lowest_tie_last",       # lowest-vertex tie broken by the last index
)


def triangulate(P, variant=None):
    """(status, [(i, j, k), ...]) of one polygon with n >= 3 finite points."""
    P = np.asarray(P, dtype=np.float32)
    n = len(P)
    o = orient_f32 if variant == "orient_f32" else orient_f64 if variant == "orient_f64" else orient_exact
    pts = [(P[i, 0], P[i, 1]) for i in range(n)]

    def same(i, j):
        return pts[i][0] == pts[j][0] and pts[i][1] == pts[j][1]

    key = [(float(p[1]), float(p[0])) for p in pts]
    lo = min(key)
    m = max(i for i in range(n) if key[i] == lo) if variant == "lowest_tie_last" else key.index(lo)
    if variant == "winding_shoelace":
        x, y = P[:, 0].astype(np.float64), P[:, 1].astype(np.float64)
        a = float(np.sum(x * np.roll(y, -1) - np.roll(x, -1) * y))
        s = -1 if a < 0 else 1
    else:
        s = 1
        pm = next((m - d) % n for d in range(1, n) if not same((m - d) % n, m)) if any(not same(i, m) for i in range(n)) else None
        if pm is not None:
            nm = next((m + d) % n for d in range(1, n) if not same((m + d) % n, m))
            s = o(pts[pm], pts[m], pts[nm]) or 1
    prv = [(i - 1) % n for i in range(n)]
    nxt = [(i + 1) % n for i in range(n)]
    tris, status = [], 0

    def emit(p, c, q):
        tris.append((p, c, q) if s > 0 or variant == "emit_ignores_winding" else (q, c, p))

    def is_ear(p, c, q):
        if variant != "no_zero_edge" and (same(c, p) or same(c, q)):
            return True
        if s * o(pts[p], pts[c], pts[q]) <= 0:
            return False
        r = nxt[q]
        while r != p:
            w = s * o(pts[prv[r]], pts[r], pts[nxt[r]])
            nonconvex = True if variant == "convex_blockers" else (w < 0 if variant == "straight_not_blocker" else w <= 0)
            excluded = variant != "no_point_eq" and (same(r, p) or same(r, c) or same(r, q))
            if nonconvex and not excluded:
                t = (s * o(pts[p], pts[c], pts[r]), s * o(pts[c], pts[q], pts[r]), s * o(pts[q], pts[p], pts[r]))
                if (min(t) > 0) if variant == "open_triangle" else (min(t) >= 0):
                    return False
            r = nxt[r]
        return True

    c = stop = 0
    k = n
    while k > 3:
        while not is_ear(prv[c], c, nxt[c]):
            c = nxt[c]
            if c == stop:
                if variant != "fallback_no_bit":
                    status |= NO_EAR
                if variant == "fallback_clips_next":
                    c = nxt[c]
                break
        p, q = prv[c], nxt[c]
        emit(p, c, q)
        nxt[p], prv[q] = q, p
        k -= 1
        c = q if variant == "cursor_at_q" else nxt[q]
        stop = c
    emit(prv[c], c, nxt[c])
    return status, tris


# ---- exact geometry of the properties -------------------------------------------------------------------------
def _fr(p):
    return Fraction(float(p[0])), Fraction(float(p[1]))


def area2(P, tri=None):
    """Twice the exact signed area of the polygon (or of the triangle tri)."""
    idx = range(len(P)) if tri is None else tri
    pts = [_fr(P[i]) for i in idx]
    return sum(pts[i][0] * pts[(i + 1) % len(pts)][1] - pts[(i + 1) % len(pts)][0] * pts[i][1] for i in range(len(pts)))


def is_simple(P):
    """Exact test: no two non-adjacent edges meet, adjacent edges meet only at their shared vertex (no overlap)."""
    n = len(P)
    pts = [_fr(p) for p in P]

    def ori(a, b, c):
        d = (b[0] - a[0]) * (c[1] - a[1]) - (b[1] - a[1]) * (c[0] - a[0])
        return (d > 0) - (d < 0)

    def on_seg(a, b, c):
        return min(a[0], b[0]) <= c[0] <= max(a[0], b[0]) and min(a[1], b[1]) <= c[1] <= max(a[1], b[1])

    def meet(a, b, c, d):
        o1, o2, o3, o4 = ori(a, b, c), ori(a, b, d), ori(c, d, a), ori(c, d, b)
        if o1 * o2 < 0 and o3 * o4 < 0:
            return True
        return (o1 == 0 and on_seg(a, b, c)) or (o2 == 0 and on_seg(a, b, d)) or (o3 == 0 and on_seg(c, d, a)) or (o4 == 0 and on_seg(c, d, b))

    if len(set(pts)) != n:
        return False
    for i in range(n):
        a, b = pts[i], pts[(i + 1) % n]
        for j in range(i + 1, n):
            c, d = pts[j], pts[(j + 1) % n]
            if j == i + 1 or (i == 0 and j == n - 1):
                shared = b if j == i + 1 else a
                other = d if j == i + 1 else c
                far = a if j == i + 1 else b
                if ori(far, shared, other) == 0 and (on_seg(far, shared, other) or on_seg(shared, other, far)):
                    return False
                continue
            if meet(a, b, c, d):
                return False
    return True


# ---- generators ---------------------------------------------------------------------------------------------------
def random_ring(rng, n, scale=100.0):
    return (rng.random((n, 2)) * scale).astype(np.float32)


def random_simple(rng, n, tries=200):
    """A random simple polygon: a star-shaped ring of distinct angles (jittered radii), or a 2-opt untangled ring."""
    ang = np.sort(rng.random(n) * 2 * np.pi)
    r = 10 + rng.random(n) * 90
    P = np.stack([100 + r * np.cos(ang), 100 + r * np.sin(ang)], 1).astype(np.float32)
    return P


def grid_polygon(rng, n):
    """Integer-grid ring with collinear runs, repeated points and signed zeros: a staircase-comb walked around."""
    w = max(2, n // 4)
    pts = [(F32(-0.0), F32(0))] + [(F32(x), F32(0)) for x in range(1, w + 1)] + \
          [(F32(w), F32(y)) for y in range(1, 3)] + [(F32(x), F32(3 + (x % 3 == 0))) for x in range(w, -1, -1)] + \
          [(F32(0), F32(2)), (F32(0), F32(1))]
    P = np.array(pts, dtype=np.float32)
    if rng.random() < 0.5:  # a repeated point
        i = int(rng.integers(0, len(P)))
        P = np.insert(P, i, P[i], axis=0)
    return P


def mirror(P):
    """Clockwise copy: x -> -x (and reversed never: the winding rule must find it)."""
    Q = P.copy()
    Q[:, 0] = -Q[:, 0]
    return Q


def spiral(n):
    """A thick spiral: outer arm out, inner arm back; n points, simple, strongly non-convex."""
    h = n // 2
    t = np.linspace(0, 6 * np.pi, h)
    r1 = 10 + 8 * t
    r2 = 4 + 8 * t
    outer = np.stack([r1 * np.cos(t), r1 * np.sin(t)], 1)
    inner = np.stack([r2 * np.cos(t), r2 * np.sin(t)], 1)[::-1]
    P = np.concatenate([outer, inner])
    if len(P) < n:
        P = np.concatenate([P, P[-1:] * 0.999])
    P = P[:n].astype(np.float32)
    if area2(P) < 0:
        P = P[::-1].copy()
    return P


def near_collinear(rng, scale_exp=0):
    """A 6-gon whose first vertex lies a few ulps off the line of its neighbours (its convexity needs the exact sign)."""
    a = np.array([rng.uniform(1, 3), rng.uniform(1, 3)], dtype=np.float32)
    b = np.array([rng.uniform(5, 9), rng.uniform(5, 9)], dtype=np.float32)
    t = F32(rng.uniform(0.3, 0.7))
    c = (a + t * (b - a)).astype(np.float32)
    steps = int(rng.integers(-3, 4))
    for _ in range(abs(steps)):
        c[1] = np.nextafter(c[1], F32(np.inf) if steps > 0 else F32(-np.inf))
    # ring: c, b, then around the far side back to a; c is vertex 0 between a (last) and b
    P = np.array([c, b, [b[0] + 1, b[1] - 6], [a[0] + 4, a[1] - 6], [a[0] + 1, a[1] - 3], a], dtype=np.float32)
    return (P * F32(2.0 ** scale_exp)).astype(np.float32)


def f64_trap(rng):
    """A 4-gon whose vertex 0 lies exactly on the line y = 3x through its neighbours, at coordinates 2^-60..2^60 apart:
    the exact orientation is 0, a plain f64 determinant of the same points is not."""
    while True:
        xs = [float(rng.integers(1 << 20, 1 << 21)) * 2.0 ** int(e) for e in (rng.integers(-10, 10), rng.integers(20, 60), rng.integers(-60, -20))]
        c, b, a = [np.array([x, 3 * x], dtype=np.float32) for x in xs]
        if orient_f64(a, c, b) != 0:
            return np.array([c, b, [b[0], b[0]], a], dtype=np.float32)


def int_ring(rng, n, k=4):
    """Random ring on a k x k integer grid: self-intersecting, with straight vertices, repeated points and -0."""
    P = rng.integers(0, k, (n, 2)).astype(np.float32)
    P[P == 0] = np.where(rng.random(int((P == 0).sum())) < 0.5, np.float32(-0.0), np.float32(0.0))
    return P


def scaled(P, e):
    return (P.astype(np.float64) * 2.0 ** (e - 2)).astype(np.float32)  # coordinates below 256: finite at 2^121


def kill_cases(rng):
    """Inputs on which the model is compared with every variant (and the GPU with the oracle)."""
    cases = []
    for n in (3, 4, 5, 6, 7, 8, 10, 13):
        for _ in range(6):
            cases.append(random_ring(rng, n))          # mostly self-intersecting
            cases.append(random_simple(rng, n))
    for n in (8, 12, 20):
        g = grid_polygon(rng, n)
        cases += [g, mirror(g)]
    for e in (-140, -75, 121):
        cases.append(scaled(random_simple(rng, 12), e))
        cases.append(scaled(grid_polygon(rng, 12), e))
    for _ in range(40):
        cases.append(near_collinear(rng, int(rng.choice([0, 60, -60, 100]))))
    for _ in range(10):
        cases.append(f64_trap(rng))
    for n in (4, 5, 6, 7, 9):
        for _ in range(12):
            cases.append(int_ring(rng, n))
    cases += [spiral(40), mirror(spiral(40))]
    # hand-made: zero-length edges, a straight vertex on a diagonal, ties of the lowest vertex, a bow-tie
    cases.append(np.array([[0, 0], [0, 0], [4, 0], [4, 4], [4, 4], [0, 4]], np.float32))
    cases.append(np.array([[0, 0], [2, 0], [4, 0], [4, 4], [2, 1], [0, 4]], np.float32))
    cases.append(np.array([[0, 0], [4, 0], [2, 2], [4, 4], [0, 4], [2, 2]], np.float32))
    cases.append(np.array([[4, 0], [0, 4], [0, 0], [4, 4]], np.float32))
    cases.append(np.array([[2, 0], [4, 0], [4, 4], [0, 4], [0, 0]], np.float32))
    cases.append(np.array([[0, 0], [3, 0], [3, 3], [2, 1], [1, 3], [0, 0], [0, 3]], np.float32))
    return cases


def pack(polys):
    fp = np.zeros(len(polys) + 1, dtype=np.uint64)
    fp[1:] = np.cumsum([len(p) for p in polys])
    xy = np.concatenate([np.asarray(p, np.float32).reshape(-1, 2) for p in polys]) if polys else np.zeros((0, 2), np.float32)
    return xy.astype(np.float32), fp
