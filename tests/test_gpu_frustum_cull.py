"""mr_terrain_cull_frustum on the GPU against the CPU oracle, bit for bit: visibility flags, visible ids, the compacted
index buffer and the counts.  Ragged tilings of a hash-noise terrain under the cameras of tests/_frustum.py, the float-edge
boxes of tests/_frustum.py across more than one 1024-tile chunk of the scan, device / pageable / pinned / NULL outputs, the
GPU's own tile boxes fed back in, rejected calls, and two wiring checks at the size limit with the synthetic boxes of
tests/_terrain_limits.py."""
import ctypes as C
import gc

import numpy as np
import pytest

import _frustum as F
import _frustum_oracle as FO
import _terrain_limits as L
from test_terrain_cull_cpu import camera_matrix

pytestmark = pytest.mark.gpu

MR_E_BADARG = -1
OUTPUTS = ("visible", "ids", "idx", "counts")
MODES = ("device", "pageable", "pinned", None)


def _torch():
    import torch

    return torch


def _ntiles(n, tr, tc):
    return ((n - 1 + tr - 1) // tr) * ((n - 1 + tc - 1) // tc)


class _Buf:
    """One argument buffer in device, pageable host or pinned host memory, filled with a sentinel."""

    def __init__(self, mode, count, dtype, fill):
        torch = _torch()
        tdt = {np.uint32: torch.int32, np.uint64: torch.int64, np.float32: torch.float32}[dtype]
        self.dtype = dtype
        if isinstance(fill, np.ndarray):
            t = torch.from_numpy(fill.view({np.uint32: np.int32, np.uint64: np.int64}.get(dtype, dtype)).copy())
        else:
            t = torch.full((count,), fill, dtype=tdt)
        if mode == "device":
            t = t.cuda()
        elif mode == "pinned":
            t = t.pin_memory()
        self.t = t

    @property
    def ptr(self):
        return self.t.data_ptr()

    def numpy(self):
        return self.t.cpu().numpy().view(self.dtype)


def _gpu_cull(ctx, boxes, n, tr, tc, m, modes, bbox_mode="device", gpu_boxes=None):
    """Run the cull with each output in the memory of modes[name] (None: NULL).  Returns {name: numpy array or None}."""
    ntiles = _ntiles(n, tr, tc)
    words = 6 * (n - 1) * (n - 1)
    if gpu_boxes is not None:
        bptr = gpu_boxes.data_ptr()
    else:
        bb = _Buf(bbox_mode, 0, np.float32, np.ascontiguousarray(boxes, dtype=np.float32).reshape(-1))
        bptr = bb.ptr
    spec = {"visible": (ntiles, np.uint32, -1), "ids": (ntiles, np.uint32, -1), "idx": (words, np.uint32, -1),
            "counts": (2, np.uint64, -1)}
    bufs = {k: None if modes[k] is None else _Buf(modes[k], *spec[k]) for k in OUTPUTS}
    m = np.ascontiguousarray(m, dtype=np.float32)
    rc = ctx.lib.mr_terrain_cull_frustum(ctx.handle, bptr, n, tr, tc, m.ctypes.data,
                                         *(None if bufs[k] is None else bufs[k].ptr for k in OUTPUTS))
    ctx.check(rc, "mr_terrain_cull_frustum")
    ctx.sync()
    return {k: None if b is None else b.numpy() for k, b in bufs.items()}


def _compare(got, ref, what):
    cnt = got["counts"] if got["counts"] is not None else ref["counts"]
    if got["counts"] is not None:
        assert got["counts"].tolist() == ref["counts"].tolist(), what
    if got["visible"] is not None:
        v = got["visible"]
        assert np.array_equal(v, ref["visible"]), (what, np.nonzero(v != ref["visible"])[0][:8])
    if got["ids"] is not None:
        assert np.array_equal(got["ids"][: int(cnt[0])], ref["ids"]), what
        assert (got["ids"][int(cnt[0]):] == 0xFFFFFFFF).all(), what
    if got["idx"] is not None:
        assert np.array_equal(got["idx"][: int(cnt[1])], ref["idx"]), what
        assert (got["idx"][int(cnt[1]):] == 0xFFFFFFFF).all(), what


def _check(ctx, oracle, boxes, n, tr, tc, m, what, gpu_boxes=None, host=True):
    ref = FO.terrain_cull_frustum(boxes, n, tr, tc, m)
    for mode in ("device", "pageable") if host else ("device",):
        got = _gpu_cull(ctx, boxes, n, tr, tc, m, dict.fromkeys(OUTPUTS, mode), bbox_mode=mode,
                        gpu_boxes=gpu_boxes if mode == "device" else None)
        _compare(got, ref, (what, mode))
    return ref


# ---- cameras and tilings --------------------------------------------------------------------------------------------------
TILINGS = ((16, 16), (7, 13), (32, 5), (300, 300), (1, 1), (256, 3))
WIDE = (4.0, 2.0, 40.0)  # terrain params: -514..510 in x and z, so that each camera sees a part of it
VIEWS = [("reference", camera_matrix())] + [(nm, F.camera_by_name(nm)) for nm, *_ in F.CAMERAS]


@pytest.fixture(scope="module")
def noise_terrain(oracle):
    n = 257
    return n, oracle.synth_heightmap_u16(0x5EED0001, n)


@pytest.mark.parametrize("tiling", TILINGS)
def test_tilings_and_cameras(ctx, oracle, noise_terrain, tiling):
    """A 257^2 hash-noise terrain, at the default scale (wholly in view of every camera) and scaled up around the origin
    (partly in view): ragged tilings, from 65,536 one-quad tiles (64 chunks of the scan) to one tile, under the reference
    camera and the four cameras of the benchmark."""
    n, h = noise_terrain
    tr, tc = tiling
    kept = 0
    for params in ((0.2, 0.1, 5.0), (1.5, 0.75, 20.0), WIDE):
        boxes = oracle.terrain_tile_bounds(h, n, tr, tc, params)
        for name, m in VIEWS:
            ref = _check(ctx, oracle, boxes, n, tr, tc, m, (tiling, params, name))
            kept += int(0 < ref["counts"][0] < len(boxes))
    assert kept > 0 or tiling == (300, 300)


# ---- float edges ----------------------------------------------------------------------------------------------------------
def test_float_edge_cases(ctx, oracle):
    """Every generated box of tests/_frustum.py in a terrain of 40 x 29 = 1160 tiles (two chunks of the scan, ragged last
    tile row and column); each matrix's boxes are cycled through the tiles."""
    n, tr, tc = 200, 5, 7
    ntiles = _ntiles(n, tr, tc)
    assert ntiles > 1024
    flips = 0
    for kind, m, boxes in F.frustum_cases():
        order = np.arange(-(-len(boxes) // ntiles) * ntiles) % len(boxes)
        for k, chunk in enumerate(order.reshape(-1, ntiles)):
            ref = _check(ctx, oracle, boxes[chunk], n, tr, tc, m, (kind, k), host=False)
            assert np.array_equal(ref["visible"].astype(bool), F.frustum_visible(m, boxes[chunk]))
            flips += int(0 < ref["visible"].sum() < ntiles)
    assert flips > 0


# ---- memory kinds -----------------------------------------------------------------------------------------------------------
def test_pointer_kinds_and_null_outputs(ctx, oracle, noise_terrain):
    """Each output in device, pageable and pinned memory and NULL, the others on the device; then all of them pageable, and
    all pinned; the boxes from each kind of memory."""
    n, h = noise_terrain
    tr, tc = 9, 11
    boxes = oracle.terrain_tile_bounds(h, n, tr, tc, WIDE)
    m = camera_matrix()
    ref = FO.terrain_cull_frustum(boxes, n, tr, tc, m)
    assert 0 < int(ref["counts"][0]) < len(boxes)
    for out in OUTPUTS:
        for mode in MODES:
            modes = dict.fromkeys(OUTPUTS, "device")
            modes[out] = mode
            _compare(_gpu_cull(ctx, boxes, n, tr, tc, m, modes), ref, (out, mode))
    for mode in ("device", "pageable", "pinned"):
        _compare(_gpu_cull(ctx, boxes, n, tr, tc, m, dict.fromkeys(OUTPUTS, mode), bbox_mode=mode), ref, ("all", mode))
    _compare(_gpu_cull(ctx, boxes, n, tr, tc, m, dict.fromkeys(OUTPUTS)), ref, "all NULL")


# ---- the GPU's own boxes --------------------------------------------------------------------------------------------------
def test_gpu_tile_boxes_fed_back(ctx, oracle):
    """mr_terrain_tile_bounds on the device, its boxes culled where they lie: boxes, then cull, equal the oracle's."""
    torch = _torch()
    n = 1025
    h = oracle.synth_heightmap_u16(0x5EED0002, n)
    hd = torch.from_numpy(h.view(np.int16).reshape(-1)).cuda()
    params = (C.c_float * 3)(0.2, 0.1, 5.0)
    for tr, tc in ((32, 32), (64, 17), (600, 600)):
        bd = torch.empty(_ntiles(n, tr, tc) * 8, dtype=torch.float32, device="cuda")
        ctx.check(ctx.lib.mr_terrain_tile_bounds(ctx.handle, hd.data_ptr(), 0, n, tr, tc, params, bd.data_ptr()), "tiles")
        ctx.sync()
        boxes = oracle.terrain_tile_bounds(h, n, tr, tc)
        assert np.array_equal(bd.cpu().numpy().reshape(-1, 8).view(np.uint32), boxes.view(np.uint32))
        for name, m in VIEWS:
            _check(ctx, oracle, boxes, n, tr, tc, m, (tr, tc, name), gpu_boxes=bd, host=False)


# ---- rejected calls ---------------------------------------------------------------------------------------------------------
def test_invalid_calls_write_nothing(ctx):
    """Bad n or tile size, a misaligned idx_out, NULL view_proj or bbox: MR_E_BADARG, every output left as it was."""
    torch = _torch()
    n, tr, tc = 65, 8, 8
    ntiles = _ntiles(n, tr, tc)
    boxes = torch.from_numpy(L.cull_boxes(np.ones(ntiles, dtype=bool)).reshape(-1)).cuda()
    m = L.IDENTITY.copy()
    vis = torch.full((ntiles,), 7, dtype=torch.int32, device="cuda")
    ids = torch.full((ntiles,), 7, dtype=torch.int32, device="cuda")
    idx = torch.full((6 * (n - 1) ** 2 + 2,), 7, dtype=torch.int32, device="cuda")
    cnt = torch.full((2,), 7, dtype=torch.int64, device="cuda")
    f = ctx.lib.mr_terrain_cull_frustum
    mp = m.ctypes.data
    calls = {
        "n = 1": (boxes.data_ptr(), 1, tr, tc, mp, idx.data_ptr()),
        "n = 65536": (boxes.data_ptr(), 65536, tr, tc, mp, idx.data_ptr()),
        "tile_rows = 0": (boxes.data_ptr(), n, 0, tc, mp, idx.data_ptr()),
        "tile_cols = 0": (boxes.data_ptr(), n, tr, 0, mp, idx.data_ptr()),
        "idx_out + 4 bytes": (boxes.data_ptr(), n, tr, tc, mp, idx.data_ptr() + 4),
        "NULL view_proj": (boxes.data_ptr(), n, tr, tc, None, idx.data_ptr()),
        "NULL bbox": (None, n, tr, tc, mp, idx.data_ptr()),
    }
    for what, (b, nn, a, c, mm, ip) in calls.items():
        rc = f(ctx.handle, b, nn, a, c, mm, vis.data_ptr(), ids.data_ptr(), ip, cnt.data_ptr())
        assert rc == MR_E_BADARG, what
        ctx.sync()
        for t in (vis, ids, idx, cnt):
            assert bool((t == 7).all()), what
    # the same call with valid arguments succeeds
    ctx.check(f(ctx.handle, boxes.data_ptr(), n, tr, tc, mp, vis.data_ptr(), ids.data_ptr(), idx.data_ptr(), cnt.data_ptr()),
              "cull")
    ctx.sync()
    assert cnt.cpu().tolist() == [ntiles, 6 * (n - 1) ** 2]


# ---- wiring at the size limit -----------------------------------------------------------------------------------------------
def test_size_limit_2_20_tiles(ctx, oracle):
    """n = 65535 in 64 x 64 tiles: 2^20 tiles whose visibility under the identity is set by boxes inside and outside the
    clip volume; flags, ids and counts equal the oracle's (device and host outputs), and with a few visible tiles the
    compacted index buffer does too."""
    torch = _torch()
    n, (tr, tc) = L.N_MAX, L.CULL_TILE
    ntiles = _ntiles(n, tr, tc)
    assert ntiles == 1 << 20
    rng = np.random.default_rng(0x5EED0F23)
    for p in (0.5, 2e-4):
        vis = rng.random(ntiles) < p
        vis[-1] = True  # the ragged last tile
        boxes = L.cull_boxes(vis)
        want_idx = p < 0.01
        ref = FO.terrain_cull_frustum(boxes, n, tr, tc, L.IDENTITY, want_idx=want_idx, idx_capacity=1 << 24)
        assert np.array_equal(ref["visible"], vis.astype(np.uint32))
        for mode in ("device", "pageable"):
            modes = {"visible": mode, "ids": mode, "counts": mode, "idx": None}
            got = _gpu_cull(ctx, boxes, n, tr, tc, L.IDENTITY, modes, bbox_mode=mode)
            _compare(got, ref, (p, mode))
        if want_idx:
            words = int(ref["counts"][1])
            idx = torch.full((words + 64,), -1, dtype=torch.int32, device="cuda")
            bd = torch.from_numpy(boxes.reshape(-1)).cuda()
            cnt = torch.zeros(2, dtype=torch.int64, device="cuda")
            ctx.check(ctx.lib.mr_terrain_cull_frustum(ctx.handle, bd.data_ptr(), n, tr, tc, L.IDENTITY.ctypes.data, None, None,
                                                       idx.data_ptr(), cnt.data_ptr()), "cull")
            ctx.sync()
            assert cnt.cpu().tolist() == ref["counts"].tolist()
            assert np.array_equal(idx[:words].cpu().numpy().view(np.uint32), ref["idx"])
            assert bool((idx[words:] == -1).all())


def test_one_tile_of_more_than_65535_chunks(ctx):
    """n = 8193 with one 8192 x 8192-quad tile (65,536 chunks of 1024 quads): the compacted buffer is mr_terrain_build's
    whole index buffer."""
    import myrenderer_b200 as mr

    torch = _torch()
    n, t = 8193, 8192
    words = 6 * (n - 1) ** 2
    full = torch.empty(words, dtype=torch.int32, device="cuda")
    T = mr.Terrain(ctx)
    T.build(T.job(torch.zeros(1, dtype=torch.int16, device="cuda"), n, rows=(0, 0), height_rows=0, idx_out=full))
    idx = torch.full((words + 64,), -1, dtype=torch.int32, device="cuda")
    bd = torch.from_numpy(L.cull_boxes([True]).reshape(-1)).cuda()
    cnt = torch.zeros(2, dtype=torch.int64, device="cuda")
    vis = torch.zeros(1, dtype=torch.int32, device="cuda")
    ctx.check(ctx.lib.mr_terrain_cull_frustum(ctx.handle, bd.data_ptr(), n, t, t, L.IDENTITY.ctypes.data, vis.data_ptr(), None,
                                               idx.data_ptr(), cnt.data_ptr()), "cull")
    ctx.sync()
    assert cnt.cpu().tolist() == [1, words] and vis.cpu().tolist() == [1]
    assert torch.equal(idx[:words], full) and bool((idx[words:] == -1).all())
    del full, idx
    gc.collect()
    torch.cuda.empty_cache()
