"""mr_triangulate_earclip_holes on the GPU against the CPU oracle (tests/earclip_oracle), byte for byte: vertex bytes,
bbox bits, status and ntri, over merged sizes at every class boundary, the kill set, invalid and non-finite input,
layouts, pointer kinds and sub-ranges; H = 0 batches against mr_triangulate_earclip; the crossing predicate against the
oracle; a 10^5-polygon property batch; and the same cases against the bounds-checked build."""
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
import _earclip_oracle as EO
from oracle import oracle as O

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CHECKED = os.path.join(ROOT, "myrenderer_b200", "lib", "libmyrenderer_b200_checked.so")
LAYOUTS = {"decl": O.GPUVERTEX_DECL, "zigauto": O.GPUVERTEX_ZIGAUTO, "stride24": (24, ((8, 2), (12, 3))), "nocolour": (8, ((0, 2),))}
SENT = 0xA5


def gpu_holes(ctx, xy, fp, fr, rs, *, layout=O.GPUVERTEX_DECL, where="device", optional=True, base_pad=(0, 0, 0)):
    """One mr_triangulate_earclip_holes call; base_pad = (points, triangles, rings) of sentinel padding in front of the
    caller's arrays (point_base / tri_base / ring_base sub-range), checked to stay untouched."""
    from myrenderer_b200._capi import MrPolygonJob, MrPolygonRings
    lib = ctx.lib
    npoly = len(fp) - 1
    ft = HO.offsets_rings(fp, fr)
    pp, tp, rp = base_pad
    fp_c = fp + np.uint64(pp)
    ft_c = ft + np.uint64(tp)
    fr_c = fr + np.uint64(rp)
    rs_c = np.concatenate([np.full(rp, 0xFFFFFFFFFFFF, np.uint64), rs + np.uint64(pp)]) if len(rs) + rp else np.zeros(1, np.uint64)
    xy_c = np.concatenate([np.full((pp, 2), np.nan, np.float32), np.asarray(xy, np.float32).reshape(-1, 2)])
    stride = layout[0]
    total = int(ft[-1])
    vtx = np.full((total + tp + 1) * 3 * stride, SENT, np.uint8)
    bbox = np.full((npoly, 4), np.nan, np.float32)
    status = np.full(npoly, 0xDEADBEEF, np.uint32)
    ntri = np.full(npoly, 0xDEADBEEF, np.uint32)

    def place(a):
        if where == "device":
            return torch.from_numpy(a.view(np.uint8).copy()).cuda()
        if where == "pinned":
            return torch.from_numpy(a.view(np.uint8).copy()).pin_memory()
        return a

    bufs = {k: place(v) for k, v in dict(xy=xy_c, fp=fp_c, ft=ft_c, fr=fr_c, rs=rs_c, vtx=vtx, bbox=bbox, status=status,
                                         ntri=ntri).items()}

    def ptr(b):
        return b.data_ptr() if isinstance(b, torch.Tensor) else b.ctypes.data

    job = MrPolygonJob()
    job.xy, job.first_point, job.point_base, job.npoly = ptr(bufs["xy"]), ptr(bufs["fp"]), 0, npoly
    job.offset_prime, job.seed, job.poly_index0 = None, 0, 0
    job.layout = O.layout_struct(*layout)
    job.vtx_out, job.first_tri, job.tri_base = ptr(bufs["vtx"]), ptr(bufs["ft"]), 0
    job.bbox_out = ptr(bufs["bbox"]) if optional else None
    job.status_out = ptr(bufs["status"]) if optional else None
    job.ntri_out = ptr(bufs["ntri"]) if optional else None
    rg = MrPolygonRings(ptr(bufs["fr"]), 0, ptr(bufs["rs"]))
    rc = lib.mr_triangulate_earclip_holes(ctx.handle, C.byref(job), C.byref(rg))
    assert rc == 0, lib.mr_last_error(ctx.handle)
    ctx.sync()

    def back(k, like):
        b = bufs[k]
        a = b.cpu().numpy() if isinstance(b, torch.Tensor) else b
        return a.view(like.dtype).reshape(like.shape)

    v = back("vtx", vtx)
    assert (v[: tp * 3 * stride] == SENT).all() and (v[(total + tp) * 3 * stride:] == SENT).all()
    out = dict(vtx=v[tp * 3 * stride: (total + tp) * 3 * stride])
    if optional:
        out.update(bbox=back("bbox", bbox), status=back("status", status), ntri=back("ntri", ntri))
    return out


def compare(got, ref):
    assert np.array_equal(got["vtx"], ref["vtx"]), "vertex bytes differ"
    if "status" in got:
        assert np.array_equal(got["status"], ref["status"]), (got["status"], ref["status"])
        assert np.array_equal(got["ntri"], ref["ntri"])
        assert np.array_equal(got["bbox"].view(np.uint32), ref["bbox"].view(np.uint32)), "bbox bits differ"


def check(ctx, polys, **kw):
    xy, fp, fr, rs = H.pack(polys)
    ref = HO.triangulate_earclip_holes(xy, fp, fr, rs, layout=kw.get("layout", O.GPUVERTEX_DECL))
    got = gpu_holes(ctx, xy, fp, fr, rs, **kw)
    compare(got, ref)
    return ref


def sized(rng, L):
    """A valid polygon of merged size L: a star outer ring of L - 5*h points and h triangle holes around its centre."""
    h = min(3, max(0, (L - 3) // 8))
    n = L - 5 * h
    outer = H.star(rng, (100, 100), 60, 90, n)
    holes = [np.array([(100 + 12 * k, 95), (106 + 12 * k, 100), (100 + 12 * k, 105)], np.float32)[::-1].copy() for k in range(h)]
    holes = [q if not k % 2 else q[::-1].copy() for k, q in enumerate(holes)]
    return H.build(outer, holes)


BOUNDARY = sorted({m + d for m in (64, 256, 1024, 4096) for d in (-1, 0, 1)} | {3, 4, 5, 4097})


def test_merged_size_class_boundaries(ctx):
    rng = np.random.default_rng(31)
    polys = [sized(rng, L) for L in BOUNDARY]
    polys += [(H.mirrored(P), st) for P, st in polys]
    ref = check(ctx, polys)
    valid = np.array([3 <= len(P) + 2 * (len(st) - 1) <= 4096 for P, st in polys])
    assert (ref["status"][valid] == 0).all() and (ref["status"][~valid] == 32).all()


def test_kill_set_and_invalid(ctx):
    rng = np.random.default_rng(20261022)
    polys = H.kill_cases(rng)
    for axis in (0, 1):
        for pos in (0, 5, 9):
            P, st = H.chain(rng, 2)
            P = P.copy()
            P[pos, axis] = (np.nan, np.inf, -np.inf)[pos % 3]
            polys.append((P, st))
    polys += [(np.zeros((0, 2), np.float32), [0]), (np.ones((2, 2), np.float32), [0]), H.many_holes(20, 20)]
    ref = check(ctx, polys)
    assert (ref["status"] & H.BAD_HOLE).any() and (ref["status"] & 2).any()


def test_no_holes_equals_earclip(ctx):
    rng = np.random.default_rng(4)
    polys = E.kill_cases(rng) + [E.spiral(n) for n in (64, 65, 300)]
    xy, fp = E.pack(polys)
    fr = np.arange(len(polys) + 1, dtype=np.uint64)
    got = gpu_holes(ctx, xy, fp, fr, fp[:-1].copy())
    ref = EO.triangulate_earclip(xy, fp)
    compare(got, ref)


def test_malformed_rings(ctx):
    sq = np.array([(0, 0), (10, 0), (10, 10), (0, 10)], np.float32)
    tri = np.array([(2, 2), (2, 4), (4, 3)], np.float32)
    P, st = H.build(sq, [tri, tri + 4])
    xy, fp, fr, rs = H.pack([(P, st)] * 6)
    rs = rs.copy()
    rs[0] += 1
    rs[4] = rs[5]
    rs[8] = rs[7] + 1
    fr = fr.copy()
    fr[5] = fr[4]  # polygon 4 without rings; polygon 5 takes its three and its own
    ref = HO.triangulate_earclip_holes(xy, fp, fr, rs)
    got = gpu_holes(ctx, xy, fp, fr, rs)
    compare(got, ref)
    assert (ref["status"][[0, 1, 2, 4]] == 1).all()


@pytest.mark.parametrize("layout", list(LAYOUTS))
@pytest.mark.parametrize("where", ["device", "pageable", "pinned"])
def test_layouts_and_pointers(ctx, layout, where):
    rng = np.random.default_rng(5)
    polys = [H.random_float(rng) for _ in range(6)] + H.kill_cases(rng)[40:70]
    check(ctx, polys, layout=LAYOUTS[layout], where=where)


@pytest.mark.parametrize("where", ["device", "pageable"])
def test_null_optional_outputs_and_subranges(ctx, where):
    rng = np.random.default_rng(6)
    polys = [H.lattice(rng) for _ in range(4)] + [H.chain(rng, 5)]
    xy, fp, fr, rs = H.pack(polys)
    ref = HO.triangulate_earclip_holes(xy, fp, fr, rs)
    compare(dict(vtx=gpu_holes(ctx, xy, fp, fr, rs, where=where, optional=False)["vtx"]), ref)
    compare(gpu_holes(ctx, xy, fp, fr, rs, where=where, base_pad=(13, 7, 5)), ref)


def test_rejected_call_writes_nothing(ctx):
    from myrenderer_b200._capi import MrPolygonJob, MrPolygonRings
    P, st = H.chain(np.random.default_rng(1), 2)
    xy, fp, fr, rs = H.pack([(P, st)])
    ft = HO.offsets_rings(fp, fr)
    vtx = np.full(int(ft[-1]) * 96, SENT, np.uint8)
    status = np.full(1, 0xDEADBEEF, np.uint32)
    job = MrPolygonJob()
    job.xy, job.first_point, job.npoly = xy.ctypes.data, fp.ctypes.data, 1
    job.layout = O.layout_struct(*O.GPUVERTEX_DECL)
    job.vtx_out, job.first_tri, job.status_out = vtx.ctypes.data, ft.ctypes.data, status.ctypes.data
    assert ctx.lib.mr_triangulate_earclip_holes(ctx.handle, C.byref(job), None) == -1
    assert ctx.lib.mr_triangulate_earclip_holes(ctx.handle, C.byref(job), C.byref(MrPolygonRings(None, 0, rs.ctypes.data))) == -1
    job.layout.stride = 6
    assert ctx.lib.mr_triangulate_earclip_holes(ctx.handle, C.byref(job), C.byref(MrPolygonRings(fr.ctypes.data, 0, rs.ctypes.data))) == -1
    assert (vtx == SENT).all() and status[0] == 0xDEADBEEF


def test_offsets_rings(ctx):
    rng = np.random.default_rng(2)
    fp = np.cumsum(np.concatenate([[0], rng.integers(0, 40, 5000)])).astype(np.uint64)
    fr = np.cumsum(np.concatenate([[3], rng.integers(0, 12, 5000)])).astype(np.uint64)
    out = np.zeros_like(fp)
    assert ctx.lib.mr_polygon_offsets_rings(ctx.handle, fp.ctypes.data, fr.ctypes.data, 5000, out.ctypes.data) == 0
    assert np.array_equal(out, HO.offsets_rings(fp, fr))
    from myrenderer_b200.host import polygon_offsets_rings_host
    assert np.array_equal(out, polygon_offsets_rings_host(fp, fr))


def test_crossing_predicate_against_oracle(ctx):
    import test_earclip_holes_cpu as T
    qs = T._quads(np.random.default_rng(41), 100_000)
    got = np.zeros(len(qs), np.int8)
    assert ctx.lib.mr_selftest_crossing(ctx.handle, qs.ctypes.data, len(qs), got.ctypes.data) == 0
    ref = np.array([HO.crossing_sign(q) for q in qs], np.int8)
    assert np.array_equal(got, ref)


def test_property_batch_100k(ctx):
    """10^5 star polygons with 0-4 triangle holes around the centre: all OK, N + 2H - 2 triangles, every triangle of
    orientation >= 0 (f64), areas add up to outer minus holes; a sample bit-exact against the oracle."""
    import myrenderer_b200 as mr
    rng = np.random.default_rng(77)
    polys = []
    base = [sized(rng, L) for L in (20, 40, 64, 100)]
    for i in range(100_000):
        P, st = base[i % 4]
        k = int(rng.integers(0, len(st)))
        polys.append((P[: st[k]] if k else P, st[:k] if k else st) if k else (P, st))
    xy, fp, fr, rs = H.pack(polys)
    batch = mr.Polygon(ctx).create_polygons(xy, fp, algorithm="earclip", rings=(fr, rs))
    ctx.sync()
    st = batch.status.cpu().numpy().view(np.uint32)
    assert (st == 0).all(), np.unique(st, return_counts=True)
    n = np.diff(fp.astype(np.int64))
    h = np.diff(fr.astype(np.int64)) - 1
    assert np.array_equal(batch.ntri.cpu().numpy(), (n + 2 * h - 2).astype(np.int32))
    tri = batch.vertex_buffer.view(torch.float32).view(-1, 8)[:, :2].double().view(-1, 3, 2)
    a2 = (tri[:, 1, 0] - tri[:, 0, 0]) * (tri[:, 2, 1] - tri[:, 0, 1]) - (tri[:, 1, 1] - tri[:, 0, 1]) * (tri[:, 2, 0] - tri[:, 0, 0])
    assert (a2 >= -1e-9).all()
    ft = torch.from_numpy(batch.first_tri.astype(np.int64)).cuda()
    seg = torch.repeat_interleave(torch.arange(len(polys), device="cuda"), ft[1:] - ft[:-1])
    tri_sum = torch.zeros(len(polys), dtype=torch.float64, device="cuda").index_add_(0, seg, a2).cpu().numpy()
    for i in range(0, len(polys), 97):
        P, s = polys[i]
        ends = list(s[1:]) + [len(P)]
        a = [abs(float(E.area2(P[u:v]))) for u, v in zip(s, ends)]
        assert abs(tri_sum[i] - (a[0] - sum(a[1:]))) < 1e-9 * a[0]
    idx = np.arange(0, len(polys), 331)
    sxy, sfp, sfr, srs = H.pack([polys[i] for i in idx])
    ref = HO.triangulate_earclip_holes(sxy, sfp, sfr, srs)
    sft = ref["first_tri"]
    for k, i in enumerate(idx):
        got = batch.vertex_buffer[int(batch.first_tri[i]) * 96: int(batch.first_tri[i + 1]) * 96].cpu().numpy()
        assert np.array_equal(got, ref["vtx"][int(sft[k]) * 96: int(sft[k + 1]) * 96])


def test_create_polygon_with_holes(ctx):
    import myrenderer_b200 as mr
    outer = np.array([(0, 0), (10, 0), (10, 10), (0, 10)], np.float32)
    holes = [np.array([(2, 2), (2, 4), (4, 4), (4, 2)], np.float32), np.array([(6, 6), (8, 6), (7, 8)], np.float32)]
    poly = mr.Polygon(ctx)
    one = poly.create_polygon(outer, holes=holes, algorithm="earclip")
    assert one.status == 0 and one.ntri == 11 + 4 - 2
    P, st = H.build(outer, holes)
    xy, fp, fr, rs = H.pack([(P, st)])
    ref = HO.triangulate_earclip_holes(xy, fp, fr, rs)
    assert np.array_equal(one.vertex_buffer.vertex_buffer.numpy(), ref["vtx"])
    with pytest.raises(ValueError):
        poly.create_polygon(outer, holes=holes)
    with pytest.raises(ValueError):
        poly.create_polygons(xy, fp, rings=(fr, rs))


def test_cases_under_the_checked_build():
    if not os.path.exists(CHECKED):
        pytest.skip("checked library not built (make -C myrenderer_b200/csrc checked)")
    env = dict(os.environ, MR_B200_LIB=CHECKED, MR_EARCLIP_HOLES_CHECKED="1")
    r = subprocess.run([sys.executable, "-m", "pytest", os.path.abspath(__file__), "-x", "-q", "-k",
                        "boundaries or kill_set or no_holes or malformed or layouts or subranges"],
                       capture_output=True, text=True, timeout=1700, cwd=ROOT, env=env)
    tail = r.stdout[-3000:] + r.stderr[-2000:]
    assert r.returncode == 0, tail
    assert "MR_CHECKED" not in r.stdout + r.stderr, tail
    assert " passed" in r.stdout, tail


def test_checked_build_is_loaded_when_asked():
    if os.environ.get("MR_EARCLIP_HOLES_CHECKED") != "1":
        pytest.skip("runs inside test_cases_under_the_checked_build")
    import myrenderer_b200 as m
    assert m.load().mr_build_flags() == 1
