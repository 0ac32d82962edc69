"""CPU tests of the indexed ear-clipping contract (mr_triangulate_earclip_indexed): the expected index buffer built from
the oracles' corner ids replays, through the oracle's sink, into the oracle's vertex bytes and bbox (plain and holes,
invalid polygons, OVERFLOW / UNDERFILL ranges, every index_base); on valid polygons the indexed triangles tile the
polygon minus its holes exactly; mr_polygon_draw_indexed_range; and the argument rejects that need no device."""
import ctypes as C
from collections import Counter

import numpy as np
import pytest

import _earclip as E
import _earclip_holes as H
import _earclip_holes_oracle as HO
import _earclip_indexed as X
import _earclip_oracle as EO


def plain_cases(rng):
    polys = E.kill_cases(rng) + [E.spiral(n) for n in (64, 65, 300)]
    nan = E.random_simple(rng, 8).copy()
    nan[3, 1] = np.nan
    polys += [np.zeros((0, 2), np.float32), np.ones((2, 2), np.float32), nan, E.random_ring(rng, 4097)]
    return polys


def holes_cases(rng):
    polys = H.kill_cases(rng)
    P, st = H.chain(rng, 2)
    P = P.copy()
    P[4, 0] = np.inf
    return polys + [(P, st), (np.zeros((0, 2), np.float32), [0]), (np.ones((2, 2), np.float32), [0])]


def malformed_rings():
    """The malformed ring data of the GPU holes tests: a wrong first start, non-increasing starts, short rings, no rings."""
    sq = np.array([(0, 0), (10, 0), (10, 10), (0, 10)], np.float32)
    tri = np.array([(2, 2), (2, 4), (4, 3)], np.float32)
    xy, fp, fr, rs = H.pack([H.build(sq, [tri, tri + 4])] * 6)
    rs = rs.copy()
    rs[0] += 1
    rs[4] = rs[5]
    rs[8] = rs[7] + 1
    fr = fr.copy()
    fr[5] = fr[4]
    return xy, fp, fr, rs


def index_bases(fp):
    return (int(fp[0]), 0, int(fp[-1]) + 7, (1 << 32) + 3)  # point_base, absolute, past every point, wrapping


@pytest.mark.parametrize("first_tri", ["exact", "ranges"])
def test_replay_plain(first_tri):
    rng = np.random.default_rng(11)
    xy, fp = E.pack(plain_cases(rng))
    ft = None
    if first_tri == "ranges":  # OVERFLOW and UNDERFILL ranges
        cnt = np.maximum(np.diff(fp.astype(np.int64)) - 2, 0) + rng.choice([-3, -1, 0, 1, 4], len(fp) - 1)
        ft = np.concatenate([[0], np.cumsum(np.maximum(cnt, 0))]).astype(np.uint64)
    ref = EO.triangulate_earclip(xy, fp, first_tri=ft)
    if first_tri == "ranges":
        assert (ref["status"] & 8).any() and (ref["status"] & 128).any()
    assert (ref["status"] & (1 | 2 | 32)).any()
    for ib in index_bases(fp):
        idx = X.expected_indices(ref["ids"], fp, ref["first_tri"], ib)
        X.check_replay(ref, idx, xy, fp, ib)


@pytest.mark.parametrize("first_tri", ["exact", "ranges"])
def test_replay_holes(first_tri):
    rng = np.random.default_rng(12)
    xy, fp, fr, rs = H.pack(holes_cases(rng))
    ft = None
    if first_tri == "ranges":
        exact = HO.offsets_rings(fp, fr).astype(np.int64)
        cnt = np.diff(exact) + rng.choice([-3, -1, 0, 1, 4], len(fp) - 1)
        ft = np.concatenate([[0], np.cumsum(np.maximum(cnt, 0))]).astype(np.uint64)
    ref = HO.triangulate_earclip_holes(xy, fp, fr, rs, first_tri=ft)
    assert (ref["status"] & H.BAD_HOLE).any() and (ref["status"] & (1 | 2)).any()
    for ib in index_bases(fp):
        idx = X.expected_indices(ref["ids"], fp, ref["first_tri"], ib)
        X.check_replay(ref, idx, xy, fp, ib)


def test_replay_malformed_rings():
    xy, fp, fr, rs = malformed_rings()
    ref = HO.triangulate_earclip_holes(xy, fp, fr, rs)
    idx = X.expected_indices(ref["ids"], fp, ref["first_tri"], 0)
    X.check_replay(ref, idx, xy, fp, 0)
    ft = ref["first_tri"].astype(np.int64)
    for i in np.nonzero(ref["status"] == 1)[0]:
        assert (idx[3 * ft[i]: 3 * ft[i + 1]] == 0).all()


def test_zeros_of_invalid_polygons_and_tails():
    rng = np.random.default_rng(13)
    xy, fp = E.pack(plain_cases(rng))
    cnt = np.maximum(np.diff(fp.astype(np.int64)) - 2, 0) + 2
    ft = np.concatenate([[0], np.cumsum(cnt)]).astype(np.uint64)
    ref = EO.triangulate_earclip(xy, fp, first_tri=ft)
    idx = X.expected_indices(ref["ids"], fp, ft, 0)
    for i in range(len(fp) - 1):
        r = idx[3 * int(ft[i]): 3 * int(ft[i + 1])]
        assert (r[3 * int(ref["ntri"][i]):] == 0).all()
        if ref["status"][i] & (1 | 2 | 32):
            assert ref["ntri"][i] == 0 and (r == 0).all()
        else:
            assert (r[: 3 * int(ref["ntri"][i])] >= fp[i]).all() and (r[: 3 * int(ref["ntri"][i])] < fp[i + 1]).all()


def _tiles(P, starts, tris):
    """The indexed triangles tile the polygon minus its holes: every triangle has orientation >= 0, the exact areas add
    up, and every directed edge is either a boundary edge in the triangles' (counter-clockwise) sense, used once, or
    cancelled by its reverse."""
    ends = list(starts[1:]) + [len(P)]
    rings = [list(range(a, b)) for a, b in zip(starts, ends)]
    areas = [E.area2(P[r[0]: r[-1] + 1]) for r in rings]
    assert all(E.area2(P, t) >= 0 for t in tris)
    assert sum(E.area2(P, t) for t in tris) == abs(areas[0]) - sum(abs(a) for a in areas[1:])
    edges = Counter()
    for a, b, c in tris:
        edges.update([(a, b), (b, c), (c, a)])
    boundary = Counter()
    for h, (r, a) in enumerate(zip(rings, areas)):
        ccw = (a > 0) == (h == 0)
        for k in range(len(r)):
            u, v = r[k], r[(k + 1) % len(r)]
            boundary[(u, v) if ccw else (v, u)] += 1
    for e, m in edges.items():
        m -= boundary.get(e, 0)
        assert m >= 0 and m == edges.get((e[1], e[0]), 0) - boundary.get((e[1], e[0]), 0), e
    assert all(edges[e] >= m for e, m in boundary.items())


def test_indexed_triangles_tile_the_polygon():
    rng = np.random.default_rng(14)
    polys = [H.random_float(rng) for _ in range(12)] + [H.lattice(rng) for _ in range(6)]
    polys += [(E.random_simple(rng, n), [0]) for n in (5, 9, 14, 30)]
    xy, fp, fr, rs = H.pack(polys)
    ref = HO.triangulate_earclip_holes(xy, fp, fr, rs)
    assert (ref["status"] == 0).all()
    base = 1000
    idx = X.expected_indices(ref["ids"], fp + np.uint64(base), ref["first_tri"], base)  # a batch starting at point 1000
    ft = ref["first_tri"].astype(np.int64)
    for i, (P, st) in enumerate(polys):
        r = idx[3 * ft[i]: 3 * ft[i + 1]].astype(np.int64) - int(fp[i])
        _tiles(P, st, [tuple(r[3 * t: 3 * t + 3]) for t in range(len(r) // 3)])


def test_draw_indexed_range():
    from myrenderer_b200 import _capi
    lib = _capi.load()
    d = _capi.MrDrawIndexedRange()
    assert lib.mr_polygon_draw_indexed_range(10, 15, 4, C.byref(d)) == 0
    assert (d.index_count, d.instance_count, d.first_index, d.base_vertex, d.first_instance) == (15, 1, 18, 0, 0)
    assert lib.mr_polygon_draw_indexed_range(7, 7, 7, C.byref(d)) == 0 and (d.index_count, d.first_index) == (0, 0)
    lim = 0xFFFFFFFF // 3  # the largest count whose threefold fits a u32
    base = 1 << 40
    assert lib.mr_polygon_draw_indexed_range(base + lim, base + 2 * lim, base, C.byref(d)) == 0
    assert (d.index_count, d.first_index) == (3 * lim, 3 * lim)
    bad = [(base, base + lim + 1, base), (base + lim + 1, base + lim + 1, base), (5, 4, 0), (3, 4, 4),
           (0, 0x5555555555555556, 0), (0x5555555555555556, 0x5555555555555556, 0)]  # 3x wraps to 2 in u64
    for args in bad:
        assert lib.mr_polygon_draw_indexed_range(*args, C.byref(d)) == -1, args
    assert lib.mr_polygon_draw_indexed_range(0, 1, 0, None) == -1


def test_null_arguments_are_rejected_without_a_device():
    from myrenderer_b200 import _capi
    lib = _capi.load()
    xy, fp = E.pack([E.random_simple(np.random.default_rng(1), 6)])
    ft = np.array([0, 4], np.uint64)
    idx = np.full(12, 0xA5A5A5A5, np.uint32)
    job = _capi.MrPolygonJob()
    job.xy, job.first_point, job.npoly, job.first_tri = xy.ctypes.data, fp.ctypes.data, 1, ft.ctypes.data
    ix = _capi.MrPolygonIndices(idx.ctypes.data, 0)
    f = lib.mr_triangulate_earclip_indexed
    assert f(None, C.byref(job), None, C.byref(ix)) == -1
    assert f(None, None, None, C.byref(ix)) == -1
    assert f(None, C.byref(job), None, None) == -1
    assert f(None, C.byref(job), None, C.byref(_capi.MrPolygonIndices(None, 0))) == -1
    assert (idx == 0xA5A5A5A5).all()


def test_host_api_rejects_indices_from_the_reference_algorithm():
    import myrenderer_b200 as mr
    xy, fp = E.pack([E.random_simple(np.random.default_rng(2), 6)])
    poly = mr.Polygon(None)
    with pytest.raises(ValueError):
        poly.create_polygons(xy, fp, output="indices")
    with pytest.raises(ValueError):
        poly.create_polygons(xy, fp, output="both", algorithm="reference")
    with pytest.raises(ValueError):
        poly.create_polygons(xy, fp, output="points", algorithm="earclip")
