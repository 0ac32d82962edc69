"""mr_triangulate_earclip on the GPU against the CPU oracle (tests/earclip_oracle), byte for byte: vertex bytes, bbox
bits, status and ntri, over sizes at every class boundary, the kill set, invalid input, layouts, pointer kinds and
sub-ranges; the exact orientation predicate against fractions; the full-size star batch; and the same cases against the
bounds-checked build."""
import ctypes as C
import os
import subprocess
import sys
from fractions import Fraction

import numpy as np
import pytest
import torch

import _earclip as E
import _earclip_oracle as EO
from oracle import oracle as O

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CHECKED = os.path.join(ROOT, "myrenderer_b200", "lib", "libmyrenderer_b200_checked.so")
LAYOUTS = {"decl": O.GPUVERTEX_DECL, "zigauto": O.GPUVERTEX_ZIGAUTO, "stride24": (24, ((8, 2), (12, 3))), "nocolour": (8, ((0, 2),))}
SENT = 0xA5


def gpu_earclip(ctx, xy, fp, *, layout=O.GPUVERTEX_DECL, where="device", optional=True, base_pad=(0, 0)):
    """One mr_triangulate_earclip call; returns dict like the oracle.  base_pad = (points, triangles) of sentinel padding
    in front of the caller's arrays (point_base / tri_base sub-range), checked to stay untouched."""
    from myrenderer_b200._capi import MrPolygonJob
    lib = ctx.lib
    fp = np.ascontiguousarray(fp, dtype=np.uint64)
    npoly = len(fp) - 1
    ft = O.polygon_offsets(fp)
    pp, tp = base_pad
    fp_c = fp + np.uint64(pp) if pp else fp
    ft_c = ft + np.uint64(tp)
    xy_c = np.concatenate([np.full((pp, 2), np.nan, np.float32), np.asarray(xy, np.float32).reshape(-1, 2)])
    stride = layout[0]
    total = int(ft[-1])
    vtx = np.full((total + tp + 1) * 3 * stride, SENT, np.uint8)  # one triangle of sentinel past the end
    bbox = np.full((npoly, 4), np.nan, np.float32)
    status = np.full(npoly, 0xDEADBEEF, np.uint32)
    ntri = np.full(npoly, 0xDEADBEEF, np.uint32)

    def place(a):
        if where == "device":
            return torch.from_numpy(a.view(np.uint8).copy()).cuda()
        if where == "pinned":
            t = torch.from_numpy(a.view(np.uint8).copy()).pin_memory()
            return t
        return a

    bufs = {k: place(v) for k, v in dict(xy=xy_c, fp=fp_c, ft=ft_c, vtx=vtx, bbox=bbox, status=status, ntri=ntri).items()}

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
    rc = lib.mr_triangulate_earclip(ctx.handle, C.byref(job))
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
    xy, fp = E.pack(polys)
    ref = EO.triangulate_earclip(xy, fp, layout=kw.get("layout", O.GPUVERTEX_DECL))
    got = gpu_earclip(ctx, xy, fp, **kw)
    if not kw.get("optional", True):
        got = dict(vtx=got["vtx"])
    compare(got, ref)
    return ref


def family_polys(n_list, family, seed):
    fp = np.zeros(len(n_list) + 1, np.uint64)
    fp[1:] = np.cumsum(n_list)
    xy = O.synth_polygons(seed, fp, family=family)
    return [xy[int(fp[i]): int(fp[i + 1])] for i in range(len(n_list))]


BOUNDARY_SIZES = sorted({m + d for m in (64, 256, 1024, 4096) for d in (-1, 0, 1)} | {3, 4, 5, 4097})


@pytest.mark.parametrize("family", [O.FAMILY_STAR, O.FAMILY_ELLIPSE, O.FAMILY_ZIPPER])
def test_class_boundaries_families(ctx, family):
    polys = family_polys(BOUNDARY_SIZES, family, 0xB0 + family)
    polys += [E.mirror(p) for p in polys]
    ref = check(ctx, polys)
    valid = np.array([3 <= len(p) <= 4096 for p in polys])
    assert (ref["status"][valid] == 0).all() and (ref["status"][~valid] == 32).all()


def test_kill_set_and_invalid(ctx):
    rng = np.random.default_rng(20261021)
    polys = E.kill_cases(rng)
    polys += [E.random_ring(rng, n) for n in (5, 9, 17, 33, 70, 300) for _ in range(3)]
    polys += [E.spiral(n) for n in (64, 65, 257, 1000)] + [E.grid_polygon(rng, n) for n in (30, 200)]
    for e in (-140, -75, 121):
        polys += [E.scaled(p, e) for p in family_polys([10, 70, 300], O.FAMILY_STAR, 9)]
    for axis in (0, 1):
        for pos in (0, 3, 6):
            for bad in (np.nan, np.inf, -np.inf):
                p = family_polys([7], O.FAMILY_ZIPPER, pos)[0].copy()
                p[pos, axis] = bad
                polys.append(p)
    polys += [np.zeros((0, 2), np.float32), np.ones((1, 2), np.float32), np.ones((2, 2), np.float32)]
    ref = check(ctx, polys)
    assert (ref["status"] & E.NO_EAR).any(), "self-intersecting rings set MR_POLY_NO_EAR"


@pytest.mark.parametrize("layout", list(LAYOUTS))
@pytest.mark.parametrize("where", ["device", "pageable", "pinned"])
def test_layouts_and_pointers(ctx, layout, where):
    rng = np.random.default_rng(4)
    polys = family_polys([3, 8, 40, 64, 65, 200], O.FAMILY_STAR, 17) + E.kill_cases(rng)[:40]
    check(ctx, polys, layout=LAYOUTS[layout], where=where)


@pytest.mark.parametrize("where", ["device", "pageable"])
def test_null_optional_outputs_and_subranges(ctx, where):
    polys = family_polys([5, 30, 100, 700], O.FAMILY_ZIPPER, 23)
    check(ctx, polys, where=where, optional=False)
    check(ctx, polys, where=where, base_pad=(13, 7))


def test_interleaved_with_reference_keeps_tier_counts(ctx):
    import myrenderer_b200 as mr
    fp = O.synth_polygon_sizes(0x5EED0003, 3000, 8, 300)
    xy = O.synth_polygons(0x5EED0003, fp)
    poly = mr.Polygon(ctx)
    ref_a = poly.create_polygons(xy, fp, seed=3)
    ctx.sync()
    counts = (C.c_uint32 * 8)()
    assert ctx.lib.mr_triangulate_tier_counts(ctx.handle, counts) == 0
    before = list(counts)
    ear = poly.create_polygons(xy, fp, algorithm="earclip")
    ctx.sync()
    assert ctx.lib.mr_triangulate_tier_counts(ctx.handle, counts) == 0
    assert list(counts) == before
    ref_b = poly.create_polygons(xy, fp, seed=3)
    ctx.sync()
    o = O.polygon_batch(xy, fp, seed=3)
    for r in (ref_a, ref_b):
        assert np.array_equal(r.vertex_buffer.cpu().numpy(), o["vtx"])
    e = EO.triangulate_earclip(xy, fp)
    assert np.array_equal(ear.vertex_buffer.cpu().numpy(), e["vtx"])
    assert np.array_equal(ear.status.cpu().numpy().view(np.uint32), e["status"])
    with pytest.raises(ValueError):
        poly.create_polygons(xy, fp, algorithm="earclip", offset_prime=np.zeros(2 * (len(fp) - 1), np.uint32))
    one = poly.create_polygon(xy[: int(fp[1])], algorithm="earclip")
    assert one.status == 0 and one.ntri == int(fp[1]) - 2


def _adversarial_triples(rng, count):
    out = np.empty((count, 6), np.float32)
    e = rng.integers(-149, 126, count)
    a = rng.standard_normal((count, 2)) * np.exp2(e)[:, None]
    b = rng.standard_normal((count, 2)) * np.exp2(np.clip(e + rng.integers(-40, 40, count), -149, 125))[:, None]
    t = rng.random(count)[:, None]
    with np.errstate(all="ignore"):
        c = a + t * (b - a)
        out[:, 0:2], out[:, 2:4], out[:, 4:6] = a, b, c
        steps = rng.integers(-3, 4, count)
        for k in range(1, 4):
            sel = np.abs(steps) >= k
            out[sel, 5] = np.nextafter(out[sel, 5], np.where(steps[sel] > 0, np.inf, -np.inf).astype(np.float32))
    z = rng.random(out.shape) < 0.03
    out[z] = np.where(rng.random(int(z.sum())) < 0.5, np.float32(0.0), np.float32(-0.0))
    sub = rng.random(out.shape) < 0.03
    out[sub] = (rng.integers(-(1 << 23), 1 << 23, int(sub.sum())) * 2.0 ** -149).astype(np.float32)
    out[~np.isfinite(out)] = np.float32(1.0)
    return out


def test_orient_predicate_against_fractions(ctx):
    rng = np.random.default_rng(99)
    abc = _adversarial_triples(rng, 1_000_000)
    got = np.zeros(len(abc), np.int8)
    assert ctx.lib.mr_selftest_orient(ctx.handle, abc.ctypes.data, len(abc), got.ctypes.data) == 0
    # every triple against the C oracle's exact expansion; a sample of 20000 against fractions
    ref = np.array([EO.orient_sign(t) for t in abc[:200_000]], np.int8)
    assert np.array_equal(got[:200_000], ref)
    for i in rng.choice(len(abc), 20_000, replace=False):
        t = abc[i]
        d = (Fraction(float(t[2])) - Fraction(float(t[0]))) * (Fraction(float(t[5])) - Fraction(float(t[1]))) - \
            (Fraction(float(t[3])) - Fraction(float(t[1]))) * (Fraction(float(t[4])) - Fraction(float(t[0])))
        assert got[i] == (d > 0) - (d < 0), t
    assert (got == 0).sum() > 1000 and (got > 0).sum() > 1000 and (got < 0).sum() > 1000


def test_full_size_star_batch(ctx):
    import myrenderer_b200 as mr
    seed = 0x5EED0005
    fp = O.synth_polygon_sizes(seed, 1_000_000, 8, 1024, dist=1)
    fp_d = torch.from_numpy(fp.view(np.int64)).cuda()
    xy_d = torch.empty((int(fp[-1]), 2), dtype=torch.float32, device="cuda")
    assert ctx.lib.mr_synth_polygons(ctx.handle, seed, 0, fp_d.data_ptr(), len(fp) - 1, xy_d.data_ptr()) == 0
    batch = mr.Polygon(ctx).create_polygons(xy_d, fp, algorithm="earclip")
    ctx.sync()
    st = batch.status.cpu().numpy().view(np.uint32)
    assert (st == 0).all(), np.unique(st, return_counts=True)
    assert np.array_equal(batch.ntri.cpu().numpy(), (np.diff(fp.astype(np.int64)) - 2).astype(np.int32))
    # areas: the triangles of each polygon sum to its shoelace area (f64 sums, relative 1e-9)
    vb = batch.vertex_buffer.view(torch.float32).view(-1, 8)[:, :2].double()
    tri = vb.view(-1, 3, 2)
    a2 = (tri[:, 1, 0] - tri[:, 0, 0]) * (tri[:, 2, 1] - tri[:, 0, 1]) - (tri[:, 1, 1] - tri[:, 0, 1]) * (tri[:, 2, 0] - tri[:, 0, 0])
    assert (a2 >= -1e-9).all()
    ft = torch.from_numpy(O.polygon_offsets(fp).astype(np.int64)).cuda()
    seg = torch.repeat_interleave(torch.arange(len(fp) - 1, device="cuda"), ft[1:] - ft[:-1])
    tri_sum = torch.zeros(len(fp) - 1, dtype=torch.float64, device="cuda").index_add_(0, seg, a2)
    P = xy_d.double()
    pseg = torch.repeat_interleave(torch.arange(len(fp) - 1, device="cuda"), fp_d[1:] - fp_d[:-1])
    nxt = torch.arange(len(P), device="cuda") + 1
    nxt[fp_d[1:] - 1] = fp_d[:-1]
    cross = P[:, 0] * P[nxt, 1] - P[nxt, 0] * P[:, 1]
    poly_sum = torch.zeros(len(fp) - 1, dtype=torch.float64, device="cuda").index_add_(0, pseg, cross)
    assert torch.allclose(tri_sum, poly_sum, rtol=1e-9, atol=1e-6)
    # a sample bit-exact against the oracle
    idx = np.random.default_rng(1).choice(len(fp) - 1, 300, replace=False)
    xy_h = xy_d.cpu().numpy()
    polys = [xy_h[int(fp[i]): int(fp[i + 1])] for i in idx]
    sx, sfp = E.pack(polys)
    ref = EO.triangulate_earclip(sx, sfp)
    ft_h = O.polygon_offsets(fp)
    sft = ref["first_tri"]
    for k, i in enumerate(idx):
        got = batch.vertex_buffer[int(ft_h[i]) * 96: int(ft_h[i + 1]) * 96].cpu().numpy()
        assert np.array_equal(got, ref["vtx"][int(sft[k]) * 96: int(sft[k + 1]) * 96])
        assert np.array_equal(batch.bbox[i].cpu().numpy().view(np.uint32), ref["bbox"][k].view(np.uint32))


def test_worst_case_spiral_4096(ctx):
    ref = check(ctx, [E.spiral(4096), E.mirror(E.spiral(4096))])
    assert (ref["status"] == 0).all()


def test_cases_under_the_checked_build():
    if not os.path.exists(CHECKED):
        pytest.skip("checked library not built (make -C myrenderer_b200/csrc checked)")
    env = dict(os.environ, MR_B200_LIB=CHECKED, MR_EARCLIP_CHECKED="1")
    r = subprocess.run([sys.executable, "-m", "pytest", os.path.abspath(__file__), "-x", "-q", "-k",
                        "boundaries or kill_set or layouts or subranges or spiral"],
                       capture_output=True, text=True, timeout=1700, cwd=ROOT, env=env)
    tail = r.stdout[-3000:] + r.stderr[-2000:]
    assert r.returncode == 0, tail
    assert "MR_CHECKED" not in r.stdout + r.stderr, tail
    assert " passed" in r.stdout, tail


def test_checked_build_is_loaded_when_asked():
    if os.environ.get("MR_EARCLIP_CHECKED") != "1":
        pytest.skip("runs inside test_cases_under_the_checked_build")
    import myrenderer_b200 as m
    assert m.load().mr_build_flags() == 1
