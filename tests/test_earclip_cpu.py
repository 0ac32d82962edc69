"""CPU tests of ear clipping: the C oracle against the Fraction model, the kill table of the model's wrong variants, and
the properties the header states for simple polygons (no MR_POLY_NO_EAR, n-2 triangles of orientation >= 0 that tile
the polygon exactly)."""
import json
import os
from collections import Counter

import numpy as np
import pytest

from oracle import oracle as O
import _earclip as E
import _earclip_oracle as EO

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def oracle_tris(P):
    xy, fp = E.pack([P])
    r = EO.triangulate_earclip(xy, fp)
    return int(r["status"][0]), [tuple(int(v) for v in r["ids"][3 * t: 3 * t + 3]) for t in range(len(P) - 2)]


@pytest.fixture(scope="module")
def cases():
    return E.kill_cases(np.random.default_rng(20261021))


def test_oracle_equals_model(cases):
    for P in cases:
        assert oracle_tris(P) == E.triangulate(P), P.tolist()


def test_orient_matches_fractions():
    rng = np.random.default_rng(5)
    for _ in range(20000):
        e = int(rng.integers(-149, 120))
        a = rng.standard_normal(2) * 2.0 ** e
        b = rng.standard_normal(2) * 2.0 ** e
        t = rng.random()
        c = a + t * (b - a)
        abc = np.concatenate([a, b, c]).astype(np.float32)
        abc[4 + int(rng.integers(0, 2))] = np.nextafter(abc[5], np.float32(np.inf)) if rng.random() < 0.3 else abc[5]
        assert EO.orient_sign(abc) == E.orient_exact(abc[0:2], abc[2:4], abc[4:6])


def test_kill_table(cases):
    ref = [E.triangulate(P) for P in cases]
    table = Counter()
    for v in E.VARIANTS:
        for P, r in zip(cases, ref):
            if E.triangulate(P, v) != r:
                table[v] += 1
    print("\nkill table (cases on which each wrong variant differs): " + json.dumps({v: table[v] for v in E.VARIANTS}))
    assert all(table[v] > 0 for v in E.VARIANTS), [v for v in E.VARIANTS if not table[v]]


def _check_properties(P):
    st, tris = oracle_tris(P)
    assert st == 0, P.tolist()
    assert len(tris) == len(P) - 2
    assert all(E.area2(P, t) >= 0 for t in tris)
    A = E.area2(P)
    assert sum(E.area2(P, t) for t in tris) == abs(A)
    # every polygon edge once, every diagonal twice in opposite directions (edges oriented like the triangles)
    d = Counter()
    for a, b, c in tris:
        for u, v in ((a, b), (b, c), (c, a)):
            d[(u, v)] += 1
    n = len(P)
    ring = {(i, (i + 1) % n) for i in range(n)} if A > 0 else {((i + 1) % n, i) for i in range(n)}
    for (u, v), k in d.items():
        if (u, v) in ring:
            assert k == 1
        else:
            assert k == 1 and d[(v, u)] == 1, (u, v)
    assert all(d[e] == 1 for e in ring)


def test_simple_random_polygons():
    rng = np.random.default_rng(7)
    for n in list(range(3, 40)) + [64, 100, 200]:
        for _ in range(4):
            P = E.random_simple(rng, n)
            if E.is_simple(P):
                _check_properties(P)
                _check_properties(E.mirror(P))


@pytest.mark.parametrize("family", [O.FAMILY_STAR, O.FAMILY_ELLIPSE, O.FAMILY_ZIPPER])
def test_families(family):
    fp = O.synth_polygon_sizes(0xEA2C, 24, 3, 300)
    xy = O.synth_polygons(0xEA2C, fp, family=family)
    for i in range(len(fp) - 1):
        P = xy[int(fp[i]): int(fp[i + 1])]
        if E.is_simple(P):
            _check_properties(P)
            _check_properties(E.mirror(P))


def test_app_polygons():
    with open(os.path.join(ROOT, "tests", "golden", "app_polygons.json")) as f:
        data = json.load(f)
    for name, p in data.items():
        _check_properties(np.asarray(p, dtype=np.float32).reshape(-1, 2))


def test_spirals_and_grids():
    rng = np.random.default_rng(11)
    for n in (16, 64, 200):
        _check_properties(E.spiral(n))
    for n in (8, 16, 40):
        g = E.grid_polygon(rng, n)
        st, tris = oracle_tris(g)
        assert st == 0 and len(tris) == len(g) - 2 and sum(E.area2(g, t) for t in tris) == E.area2(g)


def test_star_sample_config3_all_ok():
    """Every star of a config-3-sized sample (8..64 points) is MR_POLY_OK; the reference path fails on many."""
    fp = O.synth_polygon_sizes(0x5EED0003, 4000, 8, 64)
    xy = O.synth_polygons(0x5EED0003, fp)
    r = EO.triangulate_earclip(xy, fp)
    assert (r["status"] == 0).all()
    assert np.array_equal(r["ntri"], np.diff(fp.astype(np.int64)) - 2)


def test_self_intersecting_sets_no_ear_sometimes():
    rng = np.random.default_rng(3)
    st = [oracle_tris(E.random_ring(rng, 9))[0] for _ in range(200)]
    assert any(s & E.NO_EAR for s in st)


def test_restated_sink_reproduces_reference_bytes():
    """Fed the reference path's own triangle ids, the oracle's sink writes oracle.polygon_batch's vertex and bbox bytes."""
    fp = O.synth_polygon_sizes(77, 300, 4, 40)
    xy = O.synth_polygons(77, fp, family=O.FAMILY_ZIPPER)
    for layout in (O.GPUVERTEX_DECL, O.GPUVERTEX_ZIGAUTO, (24, ((8, 2), (12, 3))), (8, ((0, 2),))):
        ref = O.polygon_batch(xy, fp, seed=77, layout=layout)
        ok = ref["status"] == 0
        assert ok.sum() > 100
        vtx, bbox = EO.emit_ids(xy, fp, ref["ids"], layout=layout)
        ft = ref["first_tri"]
        s = layout[0]
        for i in np.nonzero(ok)[0]:
            a, b = int(ft[i]) * 3 * s, int(ft[i + 1]) * 3 * s
            assert np.array_equal(vtx[a:b], ref["vtx"][a:b])
            assert np.array_equal(bbox[i].view(np.uint32), ref["bbox"][i].view(np.uint32))


def test_invalid_polygons_match_reference_outputs():
    polys = [np.zeros((0, 2), np.float32), np.ones((1, 2), np.float32), np.ones((2, 2), np.float32),
             np.array([[0, 0], [1, 0], [np.nan, 1]], np.float32), np.array([[0, 0], [1, np.inf], [0, 1]], np.float32),
             np.zeros((4097, 2), np.float32)]
    xy, fp = E.pack(polys)
    r = EO.triangulate_earclip(xy, fp)
    ref = O.polygon_batch(xy, fp, seed=1)
    for k in ("vtx", "bbox", "status", "ntri"):
        assert np.array_equal(np.asarray(r[k]).view(np.uint8), np.asarray(ref[k]).view(np.uint8)), k
