"""mr_triangulate_earclip_indexed on the GPU against the expectation built from the CPU oracles (tests/_earclip_indexed.py),
byte for byte: indices, and with a vertex buffer every other output, over size-class boundaries plain and with holes,
invalid input and malformed rings, OVERFLOW / UNDERFILL ranges, sub-ranges with sentinel padding, index_base point_base
and 0 (a shard equals its slice of the whole batch), device / pageable / pinned idx_out with and without vtx_out,
rejected calls, against the existing entry points and their tier counts; a 10^5-polygon consistency batch; and the same
cases against the bounds-checked build."""
import ctypes as C
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

import _earclip as E
import _earclip_holes as H
import _earclip_holes_oracle as HO
import _earclip_indexed as X
import _earclip_oracle as EO
import test_earclip_indexed_cpu as T
from oracle import oracle as O

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CHECKED = os.path.join(ROOT, "myrenderer_b200", "lib", "libmyrenderer_b200_checked.so")
SENT = 0xA5
SENT32 = 0xA5A5A5A5


def gpu_indexed(ctx, xy, fp, ft, *, rings=None, point_base=None, tri_base=None, index_base=None, where="device",
                idx_where=None, with_vtx=True, layout=O.GPUVERTEX_DECL, entry="indexed"):
    """One call on the job (xy from row point_base, fp / ft / rings absolute, tri_base <= ft[0]); idx and vtx buffers
    cover triangles [tri_base, ft[-1] + 1), and everything outside [ft[0], ft[-1]) is checked to keep its sentinel.
    entry "plain" calls mr_triangulate_earclip(_holes) on the same job instead."""
    from myrenderer_b200._capi import MrPolygonIndices, MrPolygonJob, MrPolygonRings
    lib = ctx.lib
    npoly = len(fp) - 1
    point_base = int(fp[0]) if point_base is None else point_base
    tri_base = int(ft[0]) if tri_base is None else tri_base
    index_base = point_base if index_base is None else index_base
    idx_where = where if idx_where is None else idx_where
    stride = layout[0]
    span = int(ft[-1]) - tri_base + 1
    arrs = dict(xy=np.ascontiguousarray(xy, np.float32).reshape(-1, 2), fp=np.asarray(fp, np.uint64),
                ft=np.asarray(ft, np.uint64), vtx=np.full(span * 3 * stride, SENT, np.uint8),
                idx=np.full(span * 3, SENT32, np.uint32), bbox=np.full((npoly, 4), np.nan, np.float32),
                status=np.full(npoly, 0xDEADBEEF, np.uint32), ntri=np.full(npoly, 0xDEADBEEF, np.uint32))
    if rings is not None:
        arrs.update(fr=np.asarray(rings[0], np.uint64), rs=np.asarray(rings[1], np.uint64) if len(rings[1]) else np.zeros(1, np.uint64))

    def place(a, w):
        if w == "device":
            return torch.from_numpy(a.view(np.uint8).copy()).cuda()
        if w == "pinned":
            return torch.from_numpy(a.view(np.uint8).copy()).pin_memory()
        return a.copy()

    bufs = {k: place(v, idx_where if k == "idx" else where) for k, v in arrs.items()}

    def ptr(b):
        return b.data_ptr() if isinstance(b, torch.Tensor) else b.ctypes.data

    job = MrPolygonJob()
    job.xy, job.first_point, job.point_base, job.npoly = ptr(bufs["xy"]), ptr(bufs["fp"]), point_base, npoly
    job.layout = O.layout_struct(*layout)
    job.vtx_out = ptr(bufs["vtx"]) if with_vtx else None
    job.first_tri, job.tri_base = ptr(bufs["ft"]), tri_base
    job.bbox_out, job.status_out, job.ntri_out = ptr(bufs["bbox"]), ptr(bufs["status"]), ptr(bufs["ntri"])
    rg = None if rings is None else C.byref(MrPolygonRings(ptr(bufs["fr"]), int(rings[2]), ptr(bufs["rs"])))
    if entry == "plain":
        rc = lib.mr_triangulate_earclip(ctx.handle, C.byref(job)) if rings is None else \
            lib.mr_triangulate_earclip_holes(ctx.handle, C.byref(job), rg)
    else:
        ix = MrPolygonIndices(ptr(bufs["idx"]), index_base)
        rc = lib.mr_triangulate_earclip_indexed(ctx.handle, C.byref(job), rg, C.byref(ix))
    assert rc == 0, lib.mr_last_error(ctx.handle)
    ctx.sync()

    def back(k):
        b = bufs[k]
        a = b.cpu().numpy() if isinstance(b, torch.Tensor) else b
        return a.view(arrs[k].dtype).reshape(arrs[k].shape)

    lo, hi = int(ft[0]) - tri_base, int(ft[-1]) - tri_base
    out = dict(bbox=back("bbox"), status=back("status"), ntri=back("ntri"))
    v = back("vtx")
    if with_vtx:
        assert (v[: lo * 3 * stride] == SENT).all() and (v[hi * 3 * stride:] == SENT).all()
        out["vtx"] = v[lo * 3 * stride: hi * 3 * stride]
    else:
        assert (v == SENT).all()
    i = back("idx")
    if entry != "plain":
        assert (i[: 3 * lo] == SENT32).all() and (i[3 * hi:] == SENT32).all()
        out["idx"] = i[3 * lo: 3 * hi]
    return out


def oracle(xy, fp, ft=None, rings=None, index_base=None, layout=O.GPUVERTEX_DECL):
    """The oracle's outputs of a job whose xy starts at fp[0], plus the expected idx."""
    if rings is None:
        ref = EO.triangulate_earclip(xy, fp, first_tri=ft, layout=layout)
    else:
        ref = HO.triangulate_earclip_holes(xy, fp, rings[0], rings[1], first_tri=ft, ring_base=int(rings[2]), layout=layout)
    ref["idx"] = X.expected_indices(ref["ids"], fp, ref["first_tri"], int(fp[0]) if index_base is None else index_base)
    return ref


def compare(got, ref):
    assert np.array_equal(got["idx"], ref["idx"]), "indices differ"
    if "vtx" in got:
        assert np.array_equal(got["vtx"], ref["vtx"]), "vertex bytes differ"
    assert np.array_equal(got["status"], ref["status"]), (got["status"], ref["status"])
    assert np.array_equal(got["ntri"], ref["ntri"])
    assert np.array_equal(got["bbox"].view(np.uint32), ref["bbox"].view(np.uint32)), "bbox bits differ"


def check(ctx, xy, fp, *, rings=None, ft=None, **kw):
    ref = oracle(xy, fp, ft, rings, layout=kw.get("layout", O.GPUVERTEX_DECL))
    for with_vtx in (True, False):
        compare(gpu_indexed(ctx, xy, fp, ref["first_tri"], rings=rings, with_vtx=with_vtx, **kw), ref)
    return ref


def rings_of(fr, rs):
    return (fr, rs, 0)


def test_size_class_boundaries_plain(ctx):
    polys = [E.spiral(n) if n >= 8 else E.random_simple(np.random.default_rng(n), n) for n in
             (3, 4, 63, 64, 65, 255, 256, 257, 1023, 1024, 1025, 4095, 4096)]
    polys.append(E.random_ring(np.random.default_rng(3), 4097))
    xy, fp = E.pack(polys)
    ref = check(ctx, xy, fp)
    assert (ref["status"][:-1] == 0).all() and ref["status"][-1] == 32


def test_merged_size_class_boundaries(ctx):
    import test_gpu_earclip_holes as G
    rng = np.random.default_rng(31)
    polys = [G.sized(rng, L) for L in G.BOUNDARY]
    polys += [(H.mirrored(P), st) for P, st in polys]
    xy, fp, fr, rs = H.pack(polys)
    ref = check(ctx, xy, fp, rings=rings_of(fr, rs))
    valid = np.array([3 <= len(P) + 2 * (len(st) - 1) <= 4096 for P, st in polys])
    assert (ref["status"][valid] == 0).all() and (ref["status"][~valid] == 32).all()


def test_invalid_input_plain_and_holes(ctx):
    rng = np.random.default_rng(20261022)
    xy, fp = E.pack(T.plain_cases(rng))
    check(ctx, xy, fp)
    xy, fp, fr, rs = H.pack(T.holes_cases(rng))
    ref = check(ctx, xy, fp, rings=rings_of(fr, rs))
    assert (ref["status"] & H.BAD_HOLE).any() and (ref["status"] & 2).any()


def test_malformed_rings(ctx):
    xy, fp, fr, rs = T.malformed_rings()
    ref = check(ctx, xy, fp, rings=rings_of(fr, rs))
    assert (ref["status"][[0, 1, 2, 4]] == 1).all()


@pytest.mark.parametrize("holes", [False, True])
def test_overflow_underfill_ranges(ctx, holes):
    rng = np.random.default_rng(8)
    if holes:
        xy, fp, fr, rs = H.pack([H.random_float(rng) for _ in range(20)] + [H.lattice(rng) for _ in range(10)])
        exact, rings = HO.offsets_rings(fp, fr).astype(np.int64), rings_of(fr, rs)
    else:
        xy, fp = E.pack([E.random_simple(rng, int(n)) for n in rng.integers(3, 40, 30)] + [E.spiral(300)])
        exact, rings = O.polygon_offsets(fp).astype(np.int64), None
    cnt = np.maximum(np.diff(exact) + rng.choice([-3, -1, 0, 1, 4], len(fp) - 1), 0)
    ft = np.concatenate([[0], np.cumsum(cnt)]).astype(np.uint64)
    ref = check(ctx, xy, fp, rings=rings, ft=ft)
    assert (ref["status"] & 8).any() and (ref["status"] & 128).any()


@pytest.mark.parametrize("holes", [False, True])
def test_subranges_and_shards(ctx, holes):
    """Sentinel padding around every range, point_base / tri_base / ring_base below the job's first entries; a shard's
    call with index_base 0 equals its slice of the whole batch's, and with index_base = point_base that slice shifted."""
    rng = np.random.default_rng(9)
    if holes:
        polys = [H.random_float(rng) for _ in range(8)] + [H.lattice(rng) for _ in range(4)] + H.invalid_cases(rng)[:4]
        xy, fp, fr, rs = H.pack(polys)
        ft = HO.offsets_rings(fp, fr)
    else:
        polys = [E.random_simple(rng, int(n)) for n in rng.integers(3, 70, 20)] + [np.ones((2, 2), np.float32)]
        xy, fp = E.pack(polys)
        fr = rs = None
        ft = O.polygon_offsets(fp)
    npoly = len(fp) - 1
    # the batch itself starts at point 100, triangle 50 and ring 10, so that no index is 0 and every shard has room for
    # padding in front
    fp, ft = fp + np.uint64(100), ft + np.uint64(50)
    wrings = None if fr is None else (fr + np.uint64(10), rs + np.uint64(100), 10)
    whole = gpu_indexed(ctx, xy, fp, ft, rings=wrings, index_base=0)
    compare(whole, oracle(xy, fp, ft, wrings, index_base=0))
    for a, b in ((0, 5), (5, 13), (13, npoly), (7, 8)):
        pp, tp = 11, 6  # padding rows and triangles in front of the shard's own entries
        pb, tb = int(fp[a]) - pp, int(ft[a]) - tp
        sxy = np.concatenate([np.full((pp, 2), np.nan, np.float32), xy[int(fp[a]) - 100: int(fp[b]) - 100]])
        sfp, sft = fp[a: b + 1].copy(), ft[a: b + 1].copy()
        srings = None
        if fr is not None:
            fra = wrings[0]
            srs = np.concatenate([np.full(3, 0xFFFFFFFFFFFF, np.uint64), wrings[1][int(fr[a]): int(fr[b])]])
            srings = (fra[a: b + 1].copy(), srs, int(fra[a]) - 3)
        for ib in (0, pb):
            for with_vtx in (True, False):
                got = gpu_indexed(ctx, sxy, sfp, sft, rings=srings, point_base=pb, tri_base=tb, index_base=ib,
                                  with_vtx=with_vtx)
                lo, hi = 3 * int(ft[a] - ft[0]), 3 * int(ft[b] - ft[0])
                want = whole["idx"][lo:hi].astype(np.int64) - ib
                want = np.where(whole["idx"][lo:hi] == 0, 0, want & 0xFFFFFFFF).astype(np.uint32)
                assert np.array_equal(got["idx"], want), (a, b, ib)
                for k in ("status", "ntri"):
                    assert np.array_equal(got[k], whole[k][a:b])
                assert np.array_equal(got["bbox"].view(np.uint32), whole["bbox"][a:b].view(np.uint32))
                if with_vtx:
                    assert np.array_equal(got["vtx"], whole["vtx"][int(ft[a] - ft[0]) * 96: int(ft[b] - ft[0]) * 96])


@pytest.mark.parametrize("where", ["device", "pageable", "pinned"])
@pytest.mark.parametrize("holes", [False, True])
def test_pointer_kinds(ctx, where, holes):
    rng = np.random.default_rng(5)
    if holes:
        xy, fp, fr, rs = H.pack([H.random_float(rng) for _ in range(6)] + H.kill_cases(rng)[40:70])
        rings = rings_of(fr, rs)
    else:
        xy, fp = E.pack(E.kill_cases(rng)[:80])
        rings = None
    check(ctx, xy, fp, rings=rings, where=where)  # every buffer of that kind, vtx_out NULL and not
    ref = oracle(xy, fp, rings=rings)
    for other in ("device", "pageable", "pinned"):  # idx_out alone of that kind
        compare(gpu_indexed(ctx, xy, fp, ref["first_tri"], rings=rings, where=other, idx_where=where, with_vtx=False), ref)


@pytest.mark.parametrize("layout", ["zigauto", "nocolour"])
def test_layouts(ctx, layout):
    L = {"zigauto": O.GPUVERTEX_ZIGAUTO, "nocolour": (8, ((0, 2),))}[layout]
    rng = np.random.default_rng(6)
    xy, fp, fr, rs = H.pack([H.random_float(rng) for _ in range(6)])
    check(ctx, xy, fp, rings=rings_of(fr, rs), layout=L)


@pytest.mark.parametrize("holes", [False, True])
def test_equals_existing_entry_points_and_keeps_tier_counts(ctx, holes):
    """With vtx_out every output but idx_out is byte-identical to mr_triangulate_earclip(_holes) on the same job, and the
    reference path's tier counts stay as they were."""
    rng = np.random.default_rng(7)
    seed = 0x5EED0003
    sfp = O.synth_polygon_sizes(seed, 2048, 8, 1024, 1)
    sxy = O.synth_polygons(seed, sfp)
    import myrenderer_b200 as mr
    mr.Polygon(ctx).create_polygons(sxy, sfp, seed=seed)
    counts = (C.c_uint32 * 8)()
    assert ctx.lib.mr_triangulate_tier_counts(ctx.handle, counts) == 0
    before = list(counts)
    if holes:
        xy, fp, fr, rs = H.pack(H.kill_cases(rng))
        rings = rings_of(fr, rs)
        ft = HO.offsets_rings(fp, fr)
    else:
        xy, fp = E.pack(E.kill_cases(rng))
        rings, ft = None, O.polygon_offsets(fp)
    a = gpu_indexed(ctx, xy, fp, ft, rings=rings, entry="plain")
    b = gpu_indexed(ctx, xy, fp, ft, rings=rings)
    for k in ("vtx", "status", "ntri"):
        assert np.array_equal(a[k], b[k]), k
    assert np.array_equal(a["bbox"].view(np.uint32), b["bbox"].view(np.uint32))
    assert ctx.lib.mr_triangulate_tier_counts(ctx.handle, counts) == 0
    assert list(counts) == before


def test_rejected_calls_write_nothing(ctx):
    from myrenderer_b200._capi import MrPolygonIndices, MrPolygonJob, MrPolygonRings
    P, st = H.chain(np.random.default_rng(1), 2)
    xy, fp, fr, rs = H.pack([(P, st)])
    ft = HO.offsets_rings(fp, fr)
    n = int(ft[-1])
    vtx = np.full(n * 96, SENT, np.uint8)
    idx = np.full(3 * n + 1, SENT32, np.uint32)
    status = np.full(1, 0xDEADBEEF, np.uint32)
    job = MrPolygonJob()
    job.xy, job.first_point, job.npoly = xy.ctypes.data, fp.ctypes.data, 1
    job.layout = O.layout_struct(*O.GPUVERTEX_DECL)
    job.vtx_out, job.first_tri, job.status_out = vtx.ctypes.data, ft.ctypes.data, status.ctypes.data
    rg = MrPolygonRings(fr.ctypes.data, 0, rs.ctypes.data)
    f, h = ctx.lib.mr_triangulate_earclip_indexed, ctx.handle
    ix = MrPolygonIndices(idx.ctypes.data, 0)
    assert f(h, C.byref(job), C.byref(rg), None) == -1
    assert f(h, C.byref(job), C.byref(rg), C.byref(MrPolygonIndices(None, 0))) == -1
    assert f(h, C.byref(job), C.byref(rg), C.byref(MrPolygonIndices(idx.ctypes.data + 2, 0))) == -1
    assert f(h, C.byref(job), C.byref(MrPolygonRings(None, 0, rs.ctypes.data)), C.byref(ix)) == -1
    job.layout.stride = 6
    assert f(h, C.byref(job), C.byref(rg), C.byref(ix)) == -1
    job.vtx_out = vtx.ctypes.data + 2
    job.layout = O.layout_struct(*O.GPUVERTEX_DECL)
    assert f(h, C.byref(job), C.byref(rg), C.byref(ix)) == -1
    job.vtx_out = None
    job.first_tri = None
    assert f(h, C.byref(job), C.byref(rg), C.byref(ix)) == -1
    assert (vtx == SENT).all() and (idx == SENT32).all() and status[0] == 0xDEADBEEF
    job.first_tri = ft.ctypes.data
    job.layout.stride = 6  # not read without vtx_out
    assert f(h, C.byref(job), C.byref(rg), C.byref(ix)) == 0
    assert status[0] != 0xDEADBEEF and idx[-1] == SENT32 and (vtx == SENT).all() and (idx[:-1] != SENT32).any()


def _consistent(batch, xy, layout_stride=32):
    """xy[idx] equals the positions in the vertex buffer, triangle for triangle."""
    idx = batch.index_buffer.view(torch.int32).to(torch.int64) & 0xFFFFFFFF
    pts = torch.from_numpy(np.ascontiguousarray(xy, np.float32).reshape(-1, 2)).cuda()
    gathered = pts[idx - batch.index_base]
    pos = batch.vertex_buffer.view(torch.float32).view(-1, layout_stride // 4)[:, :2]
    assert torch.equal(gathered.view(torch.int32), pos.contiguous().view(torch.int32))


def test_consistency_batches_100k(ctx):
    """10^5 star polygons of 8..64 points, and the 0-4-hole workload of bench_earclip_holes.py: all OK, xy[idx] equals
    the positions of vtx_out, draw_indexed_range describes each polygon's range."""
    import myrenderer_b200 as mr
    sys.path.insert(0, os.path.join(ROOT, "scripts"))
    import bench_earclip_holes as BH
    seed = 0x5EED0008
    fp = O.synth_polygon_sizes(seed, 100_000, 8, 64)
    xy = O.synth_polygons(seed, fp)
    poly = mr.Polygon(ctx)
    batch = poly.create_polygons(xy, fp, algorithm="earclip", output="both")
    ctx.sync()
    assert (batch.status.cpu().numpy() == 0).all()
    _consistent(batch, xy)
    only = poly.create_polygons(xy, fp, algorithm="earclip", output="indices")
    assert only.vertex_buffer is None and torch.equal(only.index_buffer.view(torch.int32), batch.index_buffer.view(torch.int32))
    d = batch.draw_indexed_range(77)
    assert (d.index_count, d.first_index, d.instance_count) == (3 * int(fp[78] - fp[77] - 2), 3 * int(batch.first_tri[77]), 1)
    hxy, hfp, hfr, hrs, _, _ = BH.make(np, np.random.default_rng(BH.SEED), 100_000, 8, 64, 0, 4)
    hb = poly.create_polygons(hxy, hfp, algorithm="earclip", rings=(hfr, hrs), output="both")
    ctx.sync()
    assert (hb.status.cpu().numpy() == 0).all()
    _consistent(hb, hxy)


def test_cases_under_the_checked_build():
    if not os.path.exists(CHECKED):
        pytest.skip("checked library not built (make -C myrenderer_b200/csrc checked)")
    env = dict(os.environ, MR_B200_LIB=CHECKED, MR_EARCLIP_INDEXED_CHECKED="1")
    r = subprocess.run([sys.executable, "-m", "pytest", os.path.abspath(__file__), "-x", "-q", "-k",
                        "boundaries or invalid or malformed or overflow or subranges or pointer_kinds or loaded"],
                       capture_output=True, text=True, timeout=1700, cwd=ROOT, env=env)
    tail = r.stdout[-3000:] + r.stderr[-2000:]
    assert r.returncode == 0, tail
    assert "MR_CHECKED" not in r.stdout + r.stderr, tail
    assert " passed" in r.stdout, tail


def test_checked_build_is_loaded_when_asked():
    if os.environ.get("MR_EARCLIP_INDEXED_CHECKED") != "1":
        pytest.skip("runs inside test_cases_under_the_checked_build")
    import myrenderer_b200 as m
    assert m.load().mr_build_flags() == 1
