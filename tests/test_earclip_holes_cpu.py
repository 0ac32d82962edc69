"""CPU tests of ear clipping with holes: the C oracle against the Fraction model, the kill table of the model's wrong
variants, the exact crossing predicate against fractions, and the header's properties on valid polygons with holes (no
MR_POLY_NO_EAR or MR_POLY_BAD_HOLE, N + 2H - 2 triangles of orientation >= 0 that tile the polygon exactly)."""
import json
from collections import Counter
from fractions import Fraction

import numpy as np
import pytest

import _earclip as E
import _earclip_holes as H
import _earclip_holes_oracle as HO
import _earclip_oracle as EO


def oracle_tris(P, starts):
    xy, fp, fr, rs = H.pack([(P, starts)])
    r = HO.triangulate_earclip_holes(xy, fp, fr, rs)
    T = int(r["first_tri"][1])
    return int(r["status"][0]), [tuple(int(v) for v in r["ids"][3 * t: 3 * t + 3]) for t in range(T)]


@pytest.fixture(scope="module")
def cases():
    return H.kill_cases(np.random.default_rng(20261022))


def test_oracle_equals_model(cases):
    for P, st in cases:
        assert oracle_tris(P, st) == H.triangulate(P, st), (P.tolist(), st)


def test_kill_table(cases):
    ref = [H.triangulate(P, st) for P, st in cases]
    table = Counter()
    for v in H.VARIANTS:
        for (P, st), r in zip(cases, ref):
            if H.triangulate(P, st, v) != r:
                table[v] += 1
    print("\nkill table (cases on which each wrong variant differs): " + json.dumps({v: table[v] for v in H.VARIANTS}))
    assert all(table[v] > 0 for v in H.VARIANTS), [v for v in H.VARIANTS if not table[v]]


def _quads(rng, count):
    """Adversarial crossing comparisons: edge pairs through nearly the same point of the ray, at mixed scales."""
    out = np.empty((count, 9), np.float32)
    for i in range(count):
        e = int(rng.integers(-140, 100))
        s = 2.0 ** e
        my = rng.standard_normal() * s
        x0 = rng.standard_normal() * s
        q = []
        for _ in range(2):
            h1, h2 = s * 2.0 ** int(rng.integers(-20, 20)), s * 2.0 ** int(rng.integers(-20, 20))
            dx = rng.standard_normal() * s
            q += [x0 - dx * h1 / (h1 + h2), my - h1, x0 + dx * h2 / (h1 + h2), my + h2]
        out[i, :8] = q
        out[i, 8] = my
        for _ in range(int(rng.integers(0, 3))):
            k = int(rng.integers(0, 9))
            out[i, k] = np.nextafter(out[i, k], np.float32(np.inf) if rng.random() < 0.5 else np.float32(-np.inf))
        if rng.random() < 0.05:
            out[i, int(rng.integers(0, 9))] = np.float32(-0.0)
    out[~np.isfinite(out)] = np.float32(1.0)
    return out


def test_crossing_predicate_against_fractions():
    rng = np.random.default_rng(8)
    qs = _quads(rng, 4000)
    seen = Counter()
    for q in qs:
        ref = H.crossing_sign(q[0:2], q[2:4], q[4:6], q[6:8], q[8])
        assert HO.crossing_sign(q) == ref, q.tolist()
        seen[ref] += 1
    # triples: a crossing against itself and against an edge sharing an endpoint
    for q in qs[:500]:
        t = np.concatenate([q[0:4], q[0:4], q[8:9]])
        assert HO.crossing_sign(t) == 0
        t = np.concatenate([q[0:4], q[0:2], q[6:8], q[8:9]])
        assert HO.crossing_sign(t) == H.crossing_sign(t[0:2], t[2:4], t[4:6], t[6:8], t[8])
    assert min(seen[-1], seen[1]) > 1000 and seen[0] > 0, seen


def test_crossing_predicate_orders_crossings():
    """On edges that both run up, cross() > 0 exactly when edge 2 meets the line y = my left of edge 1."""
    rng = np.random.default_rng(9)
    for _ in range(2000):
        a1, b1, a2, b2 = (rng.integers(-50, 50, 2).astype(np.float32) for _ in range(4))
        my = np.float32(rng.integers(-10, 10))
        a1[1], b1[1], a2[1], b2[1] = my - rng.integers(1, 20), my + rng.integers(0, 20), my - rng.integers(0, 20), my + rng.integers(1, 20)

        def cx(a, b):
            return Fraction(float(a[0])) + (Fraction(float(my)) - Fraction(float(a[1]))) * (Fraction(float(b[0])) - Fraction(float(a[0]))) / (Fraction(float(b[1])) - Fraction(float(a[1])))
        d = cx(a1, b1) - cx(a2, b2)
        assert HO.crossing_sign(np.concatenate([a1, b1, a2, b2, [my]])) == (d > 0) - (d < 0)


def _valid_cases(rng):
    out = [H.random_float(rng) for _ in range(60)]
    out += [H.lattice(rng) for _ in range(20)] + [H.grid_holes(rng) for _ in range(20)]
    out += [H.chain(rng, k) for k in (1, 3, 8)] + [H.many_holes(4, 3)]
    out += [(H.mirrored(P), st) for P, st in out[:30]]
    for e in (-140, -75, 121):
        out += [(H.scaled(P, e), st) for P, st in out[60:64]]
    return out


def _check_properties(P, st, small):
    status, tris = oracle_tris(P, st)
    N, nh = len(P), len(st) - 1
    assert status == 0, (P.tolist(), st)
    assert len(tris) == N + 2 * nh - 2
    assert all(E.area2(P, t) >= 0 for t in tris)
    ends = list(st[1:]) + [N]
    rings = [list(range(a, b)) for a, b in zip(st, ends)]
    A = [E.area2(P[r]) for r in rings]
    assert sum(E.area2(P, t) for t in tris) == abs(A[0]) - sum(abs(a) for a in A[1:])
    # every input edge once, in the direction that has the polygon's interior on its left; every other edge (bridges,
    # diagonals) once in each direction
    d = Counter()
    for a, b, c in tris:
        for u, v in ((a, b), (b, c), (c, a)):
            d[(u, v)] += 1
    boundary = set()
    for k, r in enumerate(rings):
        fwd = (A[k] > 0) == (k == 0)
        for i in range(len(r)):
            u, v = r[i], r[(i + 1) % len(r)]
            boundary.add((u, v) if fwd else (v, u))
    assert all(d[e] == 1 for e in boundary)
    for (u, v), k in d.items():
        assert k == 1 and ((u, v) in boundary or d[(v, u)] == 1), (u, v)
    if small:  # triangle interiors pairwise disjoint (exact separating-axis test on the triangles' edges)
        T = [[(Fraction(float(P[i, 0])), Fraction(float(P[i, 1]))) for i in t] for t in tris if E.area2(P, t) > 0]

        def o(a, b, c):
            return (b[0] - a[0]) * (c[1] - a[1]) - (b[1] - a[1]) * (c[0] - a[0])
        for i in range(len(T)):
            for j in range(i + 1, len(T)):
                sep = any(all(o(X[e], X[(e + 1) % 3], q) <= 0 for q in Y) for X, Y in ((T[i], T[j]), (T[j], T[i])) for e in range(3))
                assert sep, (T[i], T[j])


def test_properties_on_valid_polygons():
    rng = np.random.default_rng(12)
    for k, (P, st) in enumerate(_valid_cases(rng)):
        _check_properties(P, st, small=len(P) <= 40 and k % 3 == 0)


def test_no_holes_equals_earclip():
    rng = np.random.default_rng(13)
    polys = E.kill_cases(rng)
    xy, fp = E.pack(polys)
    ref = EO.triangulate_earclip(xy, fp)
    fr = np.arange(len(polys) + 1, dtype=np.uint64)
    got = HO.triangulate_earclip_holes(xy, fp, fr, fp[:-1].copy())
    for k in ("vtx", "bbox", "status", "ntri", "ids"):
        assert np.array_equal(np.asarray(got[k]).view(np.uint8), np.asarray(ref[k]).view(np.uint8)), k


def test_invalid_rings_and_sizes():
    sq = np.array([(0, 0), (10, 0), (10, 10), (0, 10)], np.float32)
    tri = np.array([(2, 2), (2, 4), (4, 3)], np.float32)
    P, st = H.build(sq, [tri])
    xy, fp, fr, rs = H.pack([(P, st)] * 8)
    rs = rs.copy()
    rs[0] += 1                       # polygon 0: first ring does not start at first_point
    rs[3] = rs[2]                    # polygon 1: ring starts not increasing
    rs[5] = rs[4] + 6                # polygon 2: hole of 1 point
    rs[7] = rs[6] + 2                # polygon 3: outer ring of 2 points
    big = np.zeros((4090, 2), np.float32)
    big[:, 0] = np.arange(4090)
    big[:, 1] = (np.arange(4090) % 2) * 0.5
    Pb, stb = H.build(big, [tri, tri + 5, tri + 9])   # N + 2H = 4099 + 6 > 4096
    xy2, fp2, fr2, rs2 = H.pack([(Pb, stb), (np.zeros((2, 2), np.float32), [0]), (np.zeros((0, 2), np.float32), [])])
    nan = P.copy()
    nan[5, 1] = np.nan
    xy3, fp3, fr3, rs3 = H.pack([(nan, st)])
    r = HO.triangulate_earclip_holes(xy, fp, fr, rs)
    assert list(r["status"]) == [1, 1, 1, 1, 0, 0, 0, 0]
    r2 = HO.triangulate_earclip_holes(xy2, fp2, fr2, rs2)
    assert list(r2["status"]) == [32, 1, 1]
    r3 = HO.triangulate_earclip_holes(xy3, fp3, fr3, rs3)
    assert list(r3["status"]) == [2]
    for rr in (r, r2, r3):
        bad = rr["status"] & 35 != 0
        assert (rr["ntri"][bad] == 0).all() and (rr["bbox"][bad].view(np.uint32) == 0).all()
