"""Independent model of mr_triangulate_earclip_holes (the bridge rule of include/myrenderer_b200.h), its named wrong
variants, and the case generators of tests/test_earclip_holes_cpu.py and tests/test_gpu_earclip_holes.py.

A polygon is an [N, 2] float32 array of points and a list of ring starts (ring 0 is the outer boundary, the others are
holes).  merge() bridges the holes into one ring of N + 2H points; triangulate() clips that ring with
_earclip.triangulate, unchanged.  Every predicate is exact (fractions.Fraction)."""
from fractions import Fraction

import numpy as np

import _earclip as E

BAD_HOLE = 512
NO_EAR = E.NO_EAR
orient = E.orient_exact

VARIANTS = (
    "holes_wrong_order",     # holes merged in increasing order of their rightmost vertex
    "crossing_f64",          # the crossing comparison evaluated in f64
    "no_reflex_check",       # always bridge to the crossing edge's max-x endpoint
    "nearest_by_distance",   # bridge to the nearest ring vertex right of M, no visibility test
    "first_copy",            # the first copy of a repeated bridge point instead of the wedge test
    "same_winding_kept",     # holes whose winding equals the outer ring's are not reversed
    "tie_last",              # equal crossings keep the last edge instead of the first
    "bad_hole_no_bit",       # the no-crossing fallback does not set MR_POLY_BAD_HOLE
)


def _f(v):
    return Fraction(float(v))


def winding(pts):
    """The lowest-vertex rule of mr_triangulate_earclip on one ring (list of (x, y) float pairs)."""
    n = len(pts)
    key = [(float(p[1]), float(p[0])) for p in pts]
    m = key.index(min(key))

    def same(i, j):
        return pts[i][0] == pts[j][0] and pts[i][1] == pts[j][1]

    if all(same(i, m) for i in range(n)):
        return 1
    pm = next((m - d) % n for d in range(1, n) if not same((m - d) % n, m))
    nm = next((m + d) % n for d in range(1, n) if not same((m + d) % n, m))
    return orient(pts[pm], pts[m], pts[nm]) or 1


def crossing_sign(a1, b1, a2, b2, my):
    """Exact sign of (b2.y - my) * orient(a1, b1, a2) + (my - a2.y) * orient(a1, b1, b2): > 0 when edge 2 crosses the
    line y = my left of edge 1 (both edges running the same way in y)."""
    def o(a, b, c):
        return (_f(b[0]) - _f(a[0])) * (_f(c[1]) - _f(a[1])) - (_f(b[1]) - _f(a[1])) * (_f(c[0]) - _f(a[0]))
    d = (_f(b2[1]) - _f(my)) * o(a1, b1, a2) + (_f(my) - _f(a2[1])) * o(a1, b1, b2)
    return (d > 0) - (d < 0)


def crossing_sign_f64(a1, b1, a2, b2, my):
    def o(a, b, c):
        return (float(b[0]) - float(a[0])) * (float(c[1]) - float(a[1])) - (float(b[1]) - float(a[1])) * (float(c[0]) - float(a[0]))
    d = (float(b2[1]) - float(my)) * o(a1, b1, a2) + (float(my) - float(a2[1])) * o(a1, b1, b2)
    return (d > 0) - (d < 0)


def rightmost(pts):
    """First index largest in (x, y)."""
    key = [(float(p[0]), float(p[1])) for p in pts]
    return key.index(max(key))


def bridge(pts, ring, M, s, variant=None):
    """Ring position the hole vertex M (a point) is bridged to, and whether an edge crossed the ray (False: fallback)."""
    L = len(ring)
    my = M[1]

    def P(k):
        return pts[ring[k % L]]

    if variant == "nearest_by_distance":
        best = None
        for k in range(L):
            q = P(k)
            if q[0] >= M[0]:
                d = (_f(q[0]) - _f(M[0])) ** 2 + (_f(q[1]) - _f(M[1])) ** 2
                if best is None or d < best[0]:
                    best = (d, k)
        return (best[1], True) if best else (0, False)
    cross = crossing_sign_f64 if variant == "crossing_f64" else crossing_sign
    e = None
    for k in range(L):
        a, b = P(k), P(k + 1)
        if s * (int(b[1] > a[1]) - int(b[1] < a[1])) <= 0 or not (min(a[1], b[1]) <= my <= max(a[1], b[1])):
            continue
        if s * orient(a, b, M) < 0:
            continue
        if e is None:
            e = k
            continue
        c = cross(P(e), P(e + 1), a, b, my)
        if c > 0 or (c == 0 and variant == "tie_last"):
            e = k
    if e is None:
        return 0, False
    a, b = P(e), P(e + 1)
    if a[1] == my:
        t = e
    elif b[1] == my:
        t = (e + 1) % L
    else:
        t = e if a[0] >= b[0] else (e + 1) % L
        if variant != "no_reflex_check":
            pt = P(t)
            u = 1 if pt[1] > my else -1
            for r in range(L):
                pr = P(r)
                if (pr[0] == M[0] and pr[1] == M[1]) or s * orient(P(r - 1), pr, P(r + 1)) > 0:
                    continue
                if u * (int(pr[1] > my) - int(pr[1] < my)) < 0 or s * orient(a, b, pr) < 0 or u * orient(M, pt, pr) > 0:
                    continue
                w = u * orient(M, pr, P(t))
                if w > 0 or (w == 0 and pr[0] < P(t)[0]):
                    t = r
    T = P(t)
    if variant == "first_copy":
        return next(k for k in range(L) if P(k)[0] == T[0] and P(k)[1] == T[1]), True
    for k in range(L):
        if P(k)[0] != T[0] or P(k)[1] != T[1]:
            continue
        pp, pn = P(k - 1), P(k + 1)
        if s * orient(pp, T, pn) > 0:
            ok = s * orient(pp, T, M) > 0 and s * orient(T, pn, M) > 0
        else:
            ok = s * orient(pp, T, M) > 0 or s * orient(T, pn, M) > 0
        if ok:
            return k, True
    return t, True


def merge(P, starts, variant=None):
    """(merged ring as point ids, status bits) of a valid-size polygon."""
    P = np.asarray(P, np.float32)
    pts = [(P[i, 0], P[i, 1]) for i in range(len(P))]
    ends = list(starts[1:]) + [len(P)]
    rings = [list(range(a, b)) for a, b in zip(starts, ends)]
    s = winding([pts[i] for i in rings[0]])
    ring = list(rings[0])
    holes = []
    for h in rings[1:]:
        j = rightmost([pts[i] for i in h])
        holes.append(((float(pts[h[j]][0]), float(pts[h[j]][1])), h, j))
    # decreasing (x, y) of the rightmost vertex, ties by hole index (the sort is stable)
    holes.sort(key=lambda t: t[0], reverse=variant != "holes_wrong_order")
    status = 0
    for _, h, j in holes:
        M = pts[h[j]]
        k, ok = bridge(pts, ring, M, s, variant)
        if not ok and variant != "bad_hole_no_bit":
            status |= BAD_HOLE
        sh = winding([pts[i] for i in h])
        n = len(h)
        if sh == s and variant != "same_winding_kept":
            seq = [h[(j - d) % n] for d in range(n)]
        else:
            seq = [h[(j + d) % n] for d in range(n)]
        ring = ring[: k + 1] + seq + [h[j], ring[k]] + ring[k + 1:]
    return ring, status


def triangulate(P, starts, variant=None):
    """(status, triangles as point ids of P) of one polygon with finite points, valid ring starts and N + 2H <= 4096."""
    ring, st = merge(P, starts, variant)
    st2, tris = E.triangulate(np.asarray(P, np.float32)[ring])
    return st | st2, [tuple(ring[i] for i in t) for t in tris]


# ---- generators ---------------------------------------------------------------------------------------------------
def star(rng, c, r0, r1, n, cw=False):
    ang = np.sort(rng.random(n) * 2 * np.pi)
    r = r0 + rng.random(n) * (r1 - r0)
    pts = np.stack([c[0] + r * np.cos(ang), c[1] + r * np.sin(ang)], 1).astype(np.float32)
    return pts[::-1].copy() if cw else pts


def _inside_strict(outer, p):
    """Exact: p strictly inside the simple ring outer (crossing number; on the boundary counts as outside)."""
    x, y = _f(p[0]), _f(p[1])
    n = len(outer)
    c = False
    for i in range(n):
        a, b = outer[i], outer[(i + 1) % n]
        ax, ay, bx, by = _f(a[0]), _f(a[1]), _f(b[0]), _f(b[1])
        if min(ay, by) <= y <= max(ay, by) and min(ax, bx) <= x <= max(ax, bx):
            if (bx - ax) * (y - ay) - (by - ay) * (x - ax) == 0:
                return False
        if (ay > y) != (by > y) and x < ax + (y - ay) * (bx - ax) / (by - ay):
            c = not c
    return c


def _segments_meet(a, b, c, d):
    def o(p, q, r):
        return orient(p, q, r)

    def on(p, q, r):
        return min(_f(p[0]), _f(q[0])) <= _f(r[0]) <= max(_f(p[0]), _f(q[0])) and min(_f(p[1]), _f(q[1])) <= _f(r[1]) <= max(_f(p[1]), _f(q[1]))
    o1, o2, o3, o4 = o(a, b, c), o(a, b, d), o(c, d, a), o(c, d, b)
    if o1 * o2 < 0 and o3 * o4 < 0:
        return True
    return (o1 == 0 and on(a, b, c)) or (o2 == 0 and on(a, b, d)) or (o3 == 0 and on(c, d, a)) or (o4 == 0 and on(c, d, b))


def valid_polygon(outer, holes):
    """outer and every hole simple, holes strictly inside outer and pairwise disjoint (exact; O(total^2))."""
    if not E.is_simple(outer) or not all(E.is_simple(h) for h in holes):
        return False
    for h in holes:
        if not all(_inside_strict(outer, q) for q in h):
            return False
    rings = [outer] + list(holes)
    for i in range(len(rings)):
        for j in range(i + 1, len(rings)):
            A, B = rings[i], rings[j]
            for u in range(len(A)):
                for v in range(len(B)):
                    if _segments_meet(A[u], A[(u + 1) % len(A)], B[v], B[(v + 1) % len(B)]):
                        return False
            if i > 0 and (_inside_strict(A, B[0]) or _inside_strict(B, A[0])):
                return False
    return True


def build(outer, holes):
    """(P, starts) of a polygon from its rings."""
    rings = [np.asarray(outer, np.float32)] + [np.asarray(h, np.float32) for h in holes]
    starts = [0]
    for r in rings[:-1]:
        starts.append(starts[-1] + len(r))
    return np.concatenate(rings).astype(np.float32), starts


def random_float(rng, max_holes=5):
    """Star outer ring and star holes, each hole kept only if the polygon stays valid."""
    while True:
        outer = star(rng, (100, 100), 50, 90, int(rng.integers(12, 40)))
        if E.is_simple(outer):
            break
    holes = []
    for _ in range(int(rng.integers(1, max_holes + 1))):
        c = 100 + (rng.random(2) - 0.5) * 60
        rr = 2 + rng.random() * 6
        h = star(rng, c, rr * 0.4, rr, int(rng.integers(3, 10)), cw=bool(rng.random() < 0.7))
        if valid_polygon(outer, holes + [h]):
            holes.append(h)
    return build(outer, holes)


def lattice(rng):
    """Comb outer ring on a small integer lattice, holes sharing y levels with outer vertices and with each other (rays
    through vertices and through earlier bridges)."""
    w = 16
    top = []
    for x in range(w, -1, -2):
        top += [(x, 12), (x - 1, 12 + int(rng.integers(1, 4)))] if x > 0 else [(x, 12)]
    outer = np.array([(0, 0), (w, 0)] + top, np.float32)
    holes = []
    for cx in range(1, w - 2, 3):
        for cy in range(1, 10, 3):
            if rng.random() < 0.6:
                k = int(rng.integers(0, 4))
                h = [[(cx, cy), (cx, cy + 2), (cx + 2, cy + 2), (cx + 2, cy)],
                     [(cx, cy), (cx + 1, cy + 2), (cx + 2, cy)],
                     [(cx, cy + 1), (cx + 1, cy + 2), (cx + 2, cy + 1), (cx + 1, cy)],
                     [(cx, cy), (cx, cy + 2), (cx + 1, cy + 1), (cx + 2, cy + 2), (cx + 2, cy)]][k]
                h = np.array(h, np.float32)
                if rng.random() < 0.5:
                    h = h[::-1].copy()
                holes.append(h)
    return build(outer, holes)


def grid_holes(rng):
    """Jagged integer rectangle with small rectangle / triangle holes on a lattice of cells."""
    w = 24
    top = [(x, w + int(rng.integers(0, 3))) for x in range(w, -1, -4)]
    bot = [(x, -int(rng.integers(0, 3))) for x in range(0, w + 1, 4)]
    outer = np.array(bot + top, np.float32)
    holes = []
    for cx in range(2, w - 2, 5):
        for cy in range(2, w - 2, 5):
            if rng.random() < 0.5:
                kind = int(rng.integers(0, 3))
                if kind == 0:
                    h = [(cx, cy), (cx, cy + 2), (cx + 2, cy + 2), (cx + 2, cy)]
                elif kind == 1:
                    h = [(cx, cy), (cx + 1, cy + 3), (cx + 3, cy)]
                else:
                    h = [(cx, cy + 1), (cx + 1, cy + 3), (cx + 3, cy + 3), (cx + 2, cy + 1), (cx + 3, cy)][::-1]
                h = np.array(h, np.float32)
                if rng.random() < 0.5:
                    h = h[::-1].copy()
                holes.append(h)
    return build(outer, holes)


def chain(rng, k=6):
    """A row of holes at one y level, left to right: each hole's ray hits the hole merged just before it."""
    outer = np.array([(0, 0), (10 * k + 10, 0), (10 * k + 10, 20), (0, 20)], np.float32)
    holes = []
    for i in range(k):
        x = 5 + 10 * i
        dy = float(rng.integers(-2, 3))
        holes.append(np.array([(x, 10 + dy), (x + 3, 8), (x + 6, 10), (x + 3, 12)], np.float32)[::-1].copy())
    return build(outer, holes)


def many_holes(nx, ny):
    """A square with nx * ny small square holes (alternating orientation)."""
    outer = np.array([(0, 0), (4 * nx + 2, 0), (4 * nx + 2, 4 * ny + 2), (0, 4 * ny + 2)], np.float32)
    holes = []
    for i in range(nx):
        for j in range(ny):
            x, y = 2 + 4 * i, 2 + 4 * j
            h = np.array([(x, y), (x, y + 2), (x + 2, y + 2), (x + 2, y)], np.float32)
            holes.append(h if (i + j) % 2 else h[::-1].copy())
    return build(outer, holes)


def scaled(P, e):
    return (P.astype(np.float64) * 2.0 ** (e - 8)).astype(np.float32)  # coordinates below 2^8: finite at 2^121


def mirrored(P):
    Q = P.copy()
    Q[:, 0] = -Q[:, 0]
    return Q


def invalid_cases(rng):
    """Touching, overlapping and outside holes (defined output, possibly NO_EAR / BAD_HOLE)."""
    sq = np.array([(0, 0), (10, 0), (10, 10), (0, 10)], np.float32)
    out = []
    out.append(build(sq, [np.array([(20, 2), (22, 2), (22, 4)], np.float32)]))            # outside: no crossing
    out.append(build(sq, [np.array([(2, 2), (2, 4), (10, 3)], np.float32)]))              # touches the outer edge
    out.append(build(sq, [np.array([(2, 2), (2, 6), (6, 6), (6, 2)], np.float32),
                          np.array([(4, 4), (4, 8), (8, 8), (8, 4)], np.float32)]))      # overlapping holes
    out.append(build(sq, [np.array([(2, 2), (2, 4), (4, 4), (4, 2)], np.float32),
                          np.array([(4, 4), (4, 6), (6, 6), (6, 4)], np.float32)]))      # holes sharing a corner
    out.append(build(sq, [np.array([(-5, 5), (-3, 7), (-3, 3)], np.float32)]))             # left of the outer ring
    out.append(build(sq, [np.array([(2, 2), (8, 8), (2, 8), (8, 2)], np.float32)]))        # self-intersecting hole
    out.append(build(sq, [np.array([(3, 3), (3, 3), (3, 3)], np.float32)]))                # all points equal
    tri = np.array([(0, 4), (0, 6), (1, 5)], np.float32)
    # two ring edges crossing each other on the hole's ray: equal crossings, different targets
    out.append(build(np.array([(4, 0), (6, 10), (7, 11), (7, -1), (6, 0), (4, 10), (3, 11), (3, -1)], np.float32), [tri]))
    # an edge spanning +-2^70 crosses the ray 10 * 2^-92 right of another: an f64 evaluation calls it a tie
    e = 2.0 ** -21
    out.append(build(np.array([(5 - e, -2.0 ** 70), (5 + e, 2.0 ** 70), (7, 2.0 ** 71), (7, -2.0 ** 71), (4, 0), (6, 10),
                               (3, 2.0 ** 71), (3, -2.0 ** 71)], np.float32), [tri]))
    for _ in range(12):
        outer = E.random_ring(rng, int(rng.integers(4, 9)), 10)
        holes = [E.random_ring(rng, int(rng.integers(3, 6)), 10) for _ in range(int(rng.integers(1, 4)))]
        out.append(build(outer, holes))
    return out


def kill_cases(rng):
    """(P, starts) cases on which the model is compared with every variant (and the GPU with the oracle)."""
    cases = []
    for _ in range(40):
        cases.append(random_float(rng))
    for _ in range(25):
        cases.append(lattice(rng))
        cases.append(grid_holes(rng))
    for k in (2, 4, 7):
        cases.append(chain(rng, k))
    cases.append(many_holes(3, 2))
    for P, st in list(cases[:12]):
        cases.append((mirrored(P), st))
    for e in (-140, -75, 121):
        for P, st in cases[40:46]:
            cases.append((scaled(P, e), st))
    cases += invalid_cases(rng)
    return cases


def pack(polys):
    """(xy, first_point, first_ring, ring_start) of a batch of (P, starts)."""
    fp = [0]
    fr = [0]
    rs = []
    for P, st in polys:
        rs += [fp[-1] + s for s in st]
        fp.append(fp[-1] + len(P))
        fr.append(fr[-1] + len(st))
    xy = np.concatenate([np.asarray(P, np.float32).reshape(-1, 2) for P, _ in polys]) if polys else np.zeros((0, 2), np.float32)
    return xy, np.array(fp, np.uint64), np.array(fr, np.uint64), np.array(rs, np.uint64)
