"""Where a caller's buffers live does not change what an entry point computes.  Every entry point that takes host or
device pointers is called with its buffers all on the device, all in pageable host memory, all in pinned host memory,
with inputs on the host and outputs on the device, and the reverse; each output must equal the all-device call's byte
for byte, including the bytes a call must leave alone.  Also: the cull's optional outputs left NULL, the host xy_out that
mr_synth_polygons_family rejects, and a rejected mr_triangulate_earclip_holes call with host inputs, which must write
nothing and leave the context usable."""
import ctypes as C

import numpy as np
import pytest
import torch

from oracle import oracle as O
from test_terrain_cull_cpu import camera_matrix

pytestmark = pytest.mark.gpu

# (inputs, outputs)
PLACEMENTS = [("device", "device"), ("pageable", "pageable"), ("pinned", "pinned"), ("pageable", "device"),
              ("device", "pageable")]
SENT = 0xA5


@pytest.fixture(scope="module")
def sctx():
    """A context of this module's own, so that no other test's scratch or stream state is involved."""
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    import myrenderer_b200 as mr

    c = mr.Context(0)
    yield c
    c.close()


class Buf:
    """A copy of a numpy array in device, pageable-host or pinned-host memory."""

    def __init__(self, ctx, a, where, pinned):
        a = np.ascontiguousarray(a)
        self.like, self.where, self.nbytes = a, where, max(a.nbytes, 1)
        raw = a.view(np.uint8).reshape(-1)
        if where == "device":
            self.t = torch.from_numpy(raw.copy()).cuda()
            self.ptr = self.t.data_ptr()
        elif where == "pageable":  # 64-byte aligned, like any allocator's large blocks
            self.t = np.zeros(self.nbytes + 64, np.uint8)
            off = (-self.t.ctypes.data) % 64
            self.t = self.t[off: off + self.nbytes]
            self.t[: raw.size] = raw
            self.ptr = self.t.ctypes.data
        else:
            p = C.c_void_p()
            ctx.check(ctx.lib.mr_pinned_alloc(ctx.handle, self.nbytes, C.byref(p)), "mr_pinned_alloc")
            pinned.append(p.value)
            self.ptr = p.value
            C.memmove(self.ptr, raw.ctypes.data, raw.size)

    def get(self):
        if self.where == "device":
            raw = self.t.cpu().numpy()
        elif self.where == "pageable":
            raw = self.t.copy()
        else:
            raw = np.frombuffer(C.string_at(self.ptr, self.nbytes), np.uint8).copy()
        return raw[: self.like.nbytes].view(self.like.dtype).reshape(self.like.shape)


@pytest.fixture
def place(sctx):
    """place(array, where) -> Buf.  Pinned buffers come from mr_pinned_alloc and are freed after the test."""
    pinned = []
    yield lambda a, where: Buf(sctx, a, where, pinned)
    sctx.sync()
    for p in pinned:
        sctx.lib.mr_pinned_free(sctx.handle, p)


def sentinel(shape, dtype):
    return np.full(int(np.prod(shape)) * np.dtype(dtype).itemsize, SENT, np.uint8).view(dtype).reshape(shape)


# ---- one call per entry point: (ctx, place, where_in, where_out) -> {output name: array} --------------------------------
def _first_point(seed, npoly, nmin, nmax, pad=0):
    """Polygon offsets with sizes nmin..nmax (and a few invalid ones), starting at `pad`."""
    rng = np.random.default_rng(seed)
    sizes = rng.integers(nmin, nmax + 1, npoly)
    sizes[::37] = rng.integers(0, 3, len(sizes[::37]))
    return np.concatenate([[0], np.cumsum(sizes)]).astype(np.uint64) + np.uint64(pad)


def run_heightmap_normalize(ctx, place, wi, wo):
    h = np.random.default_rng(1).integers(0, 65536, 100_003, dtype=np.uint16)
    i, o = place(h, wi), place(sentinel(h.size, np.float32), wo)
    ctx.check(ctx.lib.mr_heightmap_normalize(ctx.handle, i.ptr, h.size, o.ptr), "normalize")
    ctx.sync()
    return {"out": o.get()}


def run_polygon_offsets(ctx, place, wi, wo):
    fp = _first_point(2, 5000, 3, 300)
    i, o = place(fp, wi), place(sentinel(fp.size, np.uint64), wo)
    ctx.check(ctx.lib.mr_polygon_offsets(ctx.handle, i.ptr, len(fp) - 1, o.ptr), "offsets")
    ctx.sync()
    return {"first_tri": o.get()}


def _rings(seed, fp):
    """first_ring of polygons with 1..3 rings each."""
    counts = np.random.default_rng(seed).integers(1, 4, len(fp) - 1)
    return np.concatenate([[0], np.cumsum(counts)]).astype(np.uint64)


def run_polygon_offsets_rings(ctx, place, wi, wo):
    fp = _first_point(3, 5000, 3, 300)
    fr = _rings(3, fp)
    a, b, o = place(fp, wi), place(fr, wi), place(sentinel(fp.size, np.uint64), wo)
    ctx.check(ctx.lib.mr_polygon_offsets_rings(ctx.handle, a.ptr, b.ptr, len(fp) - 1, o.ptr), "offsets_rings")
    ctx.sync()
    return {"first_tri": o.get()}


def _selftest(name, per, seed):
    def run(ctx, place, wi, wo):
        rng = np.random.default_rng(seed)
        q = (rng.integers(-8, 9, (20_011, per)) * rng.choice([1.0, 0.5, 1e-3, 3e5], (20_011, per))).astype(np.float32)
        i, o = place(q, wi), place(sentinel(len(q), np.int8), wo)
        ctx.check(getattr(ctx.lib, name)(ctx.handle, i.ptr, len(q), o.ptr), name)
        ctx.sync()
        return {"sign": o.get()}
    return run


def run_unirand_seed_batch(ctx, place, wi, wo):
    fp = _first_point(4, 3000, 3, 500)
    i, o = place(fp, wi), place(sentinel(2 * (len(fp) - 1), np.uint32), wo)
    ctx.check(ctx.lib.mr_unirand_seed_batch(ctx.handle, i.ptr, len(fp) - 1, 0xABCDEF, 7, o.ptr), "seed")
    ctx.sync()
    return {"offset_prime": o.get()}


def run_synth_heightmap_u16(ctx, place, wi, wo):
    n, row0, rows = 513, 17, 300
    o = place(sentinel(rows * n, np.uint16), wo)
    ctx.check(ctx.lib.mr_synth_heightmap_u16(ctx.handle, 0x5EED0004, n, row0, rows, o.ptr), "synth heightmap")
    ctx.sync()
    return {"height": o.get()}


def run_synth_polygons_family(ctx, place, wi, wo):
    fp = _first_point(5, 2000, 3, 200)
    i, o = place(fp, wi), place(sentinel(2 * int(fp[-1]), np.float32), wo)
    ctx.check(ctx.lib.mr_synth_polygons_family(ctx.handle, O.FAMILY_ZIPPER, 0x5EED0005, 3, i.ptr, len(fp) - 1, o.ptr), "synth")
    ctx.sync()
    return {"xy": o.get()}


TILE_N, TILE_R, TILE_C = 301, 16, 20


def _heightmap(n):
    return np.random.default_rng(n).integers(0, 65536, n * n, dtype=np.uint16)


def run_terrain_tile_bounds(ctx, place, wi, wo):
    tr, tc = C.c_uint32(), C.c_uint32()
    ctx.check(ctx.lib.mr_terrain_tile_count(TILE_N, TILE_R, TILE_C, C.byref(tr), C.byref(tc)), "tile count")
    h = place(_heightmap(TILE_N), wi)
    o = place(sentinel((tr.value * tc.value, 8), np.float32), wo)
    ctx.check(ctx.lib.mr_terrain_tile_bounds(ctx.handle, h.ptr, 0, TILE_N, TILE_R, TILE_C, None, o.ptr), "tile bounds")
    ctx.sync()
    return {"bbox": o.get()}


def _tile_boxes(ctx, place):
    return run_terrain_tile_bounds(ctx, place, "device", "device")["bbox"]


CULL_OUTPUTS = ("visible", "ids", "idx", "counts")


def _cull(name, ctx, place, wi, wo, given=CULL_OUTPUTS):
    boxes = _tile_boxes(ctx, place)
    ntiles = len(boxes)
    b = place(boxes, wi)
    spec = {"visible": (ntiles, np.uint32), "ids": (ntiles, np.uint32), "idx": (6 * (TILE_N - 1) ** 2, np.uint32),
            "counts": (2, np.uint64)}
    outs = {k: place(sentinel(*spec[k]), wo) if k in given else None for k in CULL_OUTPUTS}
    m = np.ascontiguousarray(camera_matrix((20.0, 30.0, -25.0), (5.0, 0.0, 5.0)), np.float32).reshape(16)
    rc = getattr(ctx.lib, name)(ctx.handle, b.ptr, TILE_N, TILE_R, TILE_C, m.ctypes.data,
                                *(None if outs[k] is None else outs[k].ptr for k in CULL_OUTPUTS))
    ctx.check(rc, name)
    ctx.sync()
    return {k: o.get() for k, o in outs.items() if o is not None}


def _cull_prefixes(got, counts):
    """The bytes a cull defines: every visible flag, the filled prefixes of ids and idx, the counts."""
    out = dict(got)
    if "ids" in out:
        out["ids"] = out["ids"][: int(counts[0])]
    if "idx" in out:
        out["idx"] = out["idx"][: int(counts[1])]
    return out


def run_terrain_cull(ctx, place, wi, wo):
    got = _cull("mr_terrain_cull", ctx, place, wi, wo)
    return _cull_prefixes(got, got["counts"])


def run_terrain_cull_frustum(ctx, place, wi, wo):
    got = _cull("mr_terrain_cull_frustum", ctx, place, wi, wo)
    return _cull_prefixes(got, got["counts"])


def run_terrain_build(ctx, place, wi, wo):
    """A band of rows and a band of quad rows, into full-size buffers whose other bytes must stay untouched."""
    from myrenderer_b200._capi import MrTerrainJob
    n = 300
    h = place(_heightmap(n), wi)
    vtx = place(sentinel(n * n * 32, np.uint8), wo)
    idx = place(sentinel(6 * (n - 1) ** 2, np.uint32), wo)
    j = MrTerrainJob()
    j.n, j.height_fmt, j.height, j.height_row0, j.height_rows = n, 0, h.ptr, 0, n
    j.row_begin, j.row_end, j.vtx_out, j.vtx_row0 = 37, 211, vtx.ptr, 0
    j.qrow_begin, j.qrow_end, j.idx_out, j.idx_qrow0 = 40, 200, idx.ptr, 0
    j.layout = O.layout_struct(*O.TERRAINVERTEX)
    ctx.check(ctx.lib.mr_terrain_params_default(C.byref(j.params)), "params")
    ctx.check(ctx.lib.mr_terrain_build(ctx.handle, C.byref(j)), "terrain build")
    ctx.sync()
    return {"vtx": vtx.get(), "idx": idx.get()}


def _polygon_job(ctx, place, wi, wo, fp, xy, ft, *, offset_prime=None, pads=(0, 0)):
    """An mr_polygon_job over caller buffers; the job's first point and first triangle lie `pads` past the bases, so
    the vertex bytes in front of its range must stay untouched."""
    from myrenderer_b200._capi import MrPolygonJob
    npoly = len(fp) - 1
    ntri_total = int(ft[-1])
    bufs = {"xy": place(xy, wi), "fp": place(fp, wi), "ft": place(ft, wi),
            "vtx": place(sentinel(ntri_total * 3 * 32, np.uint8), wo),
            "bbox": place(sentinel((npoly, 4), np.float32), wo), "status": place(sentinel(npoly, np.uint32), wo),
            "ntri": place(sentinel(npoly, np.uint32), wo)}
    if offset_prime is not None:
        bufs["op"] = place(offset_prime, wi)
    j = MrPolygonJob()
    j.xy, j.first_point, j.point_base, j.npoly = bufs["xy"].ptr, bufs["fp"].ptr, 0, npoly
    j.offset_prime = bufs["op"].ptr if offset_prime is not None else None
    j.seed, j.poly_index0 = 11, 0
    j.layout = O.layout_struct(*O.GPUVERTEX_DECL)
    j.vtx_out, j.first_tri, j.tri_base = bufs["vtx"].ptr, bufs["ft"].ptr, 0
    j.bbox_out, j.status_out, j.ntri_out = bufs["bbox"].ptr, bufs["status"].ptr, bufs["ntri"].ptr
    return j, bufs


def _polygons(seed, npoly, pads):
    fp = _first_point(seed, npoly, 3, 150, pad=pads[0])
    xy = np.concatenate([np.full((pads[0], 2), np.nan, np.float32), O.synth_polygons(seed, fp - fp[0])]).astype(np.float32)
    ft = O.polygon_offsets(fp - fp[0]) + np.uint64(pads[1])
    return fp, xy, ft


OUT_KEYS = ("vtx", "bbox", "status", "ntri")


def run_triangulate_batch(ctx, place, wi, wo):
    fp, xy, ft = _polygons(6, 400, (5, 3))
    op = np.zeros(2 * (len(fp) - 1), np.uint32)
    ctx.check(ctx.lib.mr_unirand_seed_batch(ctx.handle, fp.ctypes.data, len(fp) - 1, 11, 0, op.ctypes.data), "seed")
    j, bufs = _polygon_job(ctx, place, wi, wo, fp, xy, ft, offset_prime=op)
    ctx.check(ctx.lib.mr_triangulate_batch(ctx.handle, C.byref(j)), "triangulate")
    ctx.sync()
    return {k: bufs[k].get() for k in OUT_KEYS}


def run_triangulate_earclip(ctx, place, wi, wo):
    fp, xy, ft = _polygons(7, 400, (4, 6))
    j, bufs = _polygon_job(ctx, place, wi, wo, fp, xy, ft)
    ctx.check(ctx.lib.mr_triangulate_earclip(ctx.handle, C.byref(j)), "earclip")
    ctx.sync()
    return {k: bufs[k].get() for k in OUT_KEYS}


def _holed_polygons(npoly, ring_pad=0):
    """Regular outer rings with 0..2 square holes: (first_point, xy, first_ring, ring_start, first_tri)."""
    rng = np.random.default_rng(8)
    pts, fr, rs, fp = [], [0], [], [0]
    for i in range(npoly):
        n = int(rng.integers(8, 120))
        holes = int(rng.integers(0, 3))
        a = 2 * np.pi * np.arange(n) / n
        ring_pts = [np.stack([30.0 * i + 10 * np.cos(a), 10 * np.sin(a)], 1)]
        for k in range(holes):  # clockwise squares inside the counter-clockwise outer ring
            cx = 30.0 * i + (4.0 if k == 0 else -4.0)
            ring_pts.append(np.array([[cx - 1, -1], [cx - 1, 1], [cx + 1, 1], [cx + 1, -1]]))
        start = fp[-1]
        for r in ring_pts:
            rs.append(start)
            start += len(r)
        pts += ring_pts
        fp.append(start)
        fr.append(len(rs))
    fp, fr = np.array(fp, np.uint64), np.array(fr, np.uint64) + np.uint64(ring_pad)
    rs = np.concatenate([np.zeros(ring_pad, np.uint64), np.array(rs, np.uint64)])
    hole_counts = np.diff(fr) - 1
    ft = np.concatenate([[0], np.cumsum(np.diff(fp).astype(np.int64) + 2 * hole_counts.astype(np.int64) - 2)]).astype(np.uint64)
    return fp, np.concatenate(pts).astype(np.float32), fr, rs, ft


def _holes_call(ctx, place, wi, wo, ring_base=0):
    from myrenderer_b200._capi import MrPolygonRings
    fp, xy, fr, rs, ft = _holed_polygons(300, ring_pad=2)
    j, bufs = _polygon_job(ctx, place, wi, wo, fp, xy, ft)
    bufs["fr"], bufs["rs"] = place(fr, wi), place(rs, wi)
    rc = ctx.lib.mr_triangulate_earclip_holes(ctx.handle, C.byref(j), C.byref(MrPolygonRings(bufs["fr"].ptr, ring_base,
                                                                                             bufs["rs"].ptr)))
    ctx.sync()
    return rc, bufs


def run_triangulate_earclip_holes(ctx, place, wi, wo):
    rc, bufs = _holes_call(ctx, place, wi, wo)
    ctx.check(rc, "earclip holes")
    return {k: bufs[k].get() for k in OUT_KEYS}


ENTRY_POINTS = {
    "heightmap_normalize": run_heightmap_normalize,
    "polygon_offsets": run_polygon_offsets,
    "polygon_offsets_rings": run_polygon_offsets_rings,
    "selftest_orient": _selftest("mr_selftest_orient", 6, 9),
    "selftest_crossing": _selftest("mr_selftest_crossing", 9, 10),
    "unirand_seed_batch": run_unirand_seed_batch,
    "synth_heightmap_u16": run_synth_heightmap_u16,
    "synth_polygons_family": run_synth_polygons_family,
    "terrain_tile_bounds": run_terrain_tile_bounds,
    "terrain_cull": run_terrain_cull,
    "terrain_cull_frustum": run_terrain_cull_frustum,
    "terrain_build": run_terrain_build,
    "triangulate_batch": run_triangulate_batch,
    "triangulate_earclip": run_triangulate_earclip,
    "triangulate_earclip_holes": run_triangulate_earclip_holes,
}


def assert_same_bytes(got, ref):
    assert got.keys() == ref.keys()
    for k in ref:
        assert got[k].shape == ref[k].shape, k
        assert got[k].tobytes() == ref[k].tobytes(), f"{k} differs from the all-device call"


# (a host xy_out with a device first_point is rejected: test_synth_polygons_rejects_host_xy_with_device_first_point)
CASES = [(e, p) for e in ENTRY_POINTS for p in PLACEMENTS[1:] if (e, p) != ("synth_polygons_family", ("device", "pageable"))]


@pytest.mark.parametrize("entry,placement", CASES, ids=[f"{e}-{p[0]}-{p[1]}" for e, p in CASES])
def test_placements_match_the_all_device_call(sctx, place, entry, placement):
    run = ENTRY_POINTS[entry]
    ref = run(sctx, place, "device", "device")
    if entry == "synth_heightmap_u16":  # no inputs: only the output's placement matters
        assert (ref["height"].view(np.uint8) != SENT).any()
    got = run(sctx, place, *placement)
    assert_same_bytes(got, ref)


@pytest.mark.parametrize("where", ["device", "pageable", "pinned"])
@pytest.mark.parametrize("name", ["mr_terrain_cull", "mr_terrain_cull_frustum"])
def test_cull_null_outputs(sctx, place, name, where):
    full = _cull(name, sctx, place, "device", "device")
    assert 0 < full["counts"][0] < len(full["visible"]), "the camera sees some tiles and misses others"
    for drop in [(k,) for k in CULL_OUTPUTS] + [CULL_OUTPUTS]:
        given = tuple(k for k in CULL_OUTPUTS if k not in drop)
        got = _cull(name, sctx, place, where, where, given)
        assert_same_bytes(_cull_prefixes(got, full["counts"]), _cull_prefixes({k: full[k] for k in given}, full["counts"]))


@pytest.mark.parametrize("where", ["pageable", "pinned"])
def test_synth_polygons_rejects_host_xy_with_device_first_point(sctx, place, where):
    fp = _first_point(5, 200, 3, 50)
    i, o = place(fp, "device"), place(sentinel(2 * int(fp[-1]), np.float32), where)
    rc = sctx.lib.mr_synth_polygons_family(sctx.handle, O.FAMILY_STAR, 1, 0, i.ptr, len(fp) - 1, o.ptr)
    assert rc == -1  # MR_E_BADARG
    sctx.sync()
    assert (o.get().view(np.uint8) == SENT).all()


@pytest.mark.parametrize("where", ["pageable", "pinned"])
def test_bad_ring_base_with_host_inputs_writes_nothing(sctx, place, where):
    """ring_base past first_ring[npoly] with every buffer in host memory: rejected before anything is produced, and the
    next call on the context, all on the device, is unaffected."""
    fp, _, fr, _, _ = _holed_polygons(300, ring_pad=2)
    rc, bufs = _holes_call(sctx, place, where, where, ring_base=int(fr[-1]) + 1)
    assert rc == -1  # MR_E_BADARG
    for k in OUT_KEYS:
        assert (bufs[k].get().view(np.uint8) == SENT).all(), f"{k} was written"
    got = run_triangulate_earclip_holes(sctx, place, "device", "device")
    ref = run_triangulate_earclip_holes(sctx, place, "device", "device")
    assert_same_bytes(got, ref)
    assert (got["status"] == 0).all() and (got["ntri"] == np.diff(_holed_polygons(300)[4])).all()
