"""The terrain kernels at float edges, against the CPU oracle: the cull on boxes within a few ulps of its thresholds and
with +-inf / NaN components, the mesh and the tile boxes of heightmaps holding NaN, +-inf, +-0, subnormals and +-FLT_MAX,
and special height scales.  Outputs are compared bit for bit, except that any two NaNs are equal (the header leaves a
NaN's sign and payload unspecified).  The cases come from tests/_float_edges.py; tests/test_float_edges_cpu.py checks
that they tell plausible wrong kernels apart."""
import ctypes as C

import numpy as np
import pytest

import _float_edges as E

pytestmark = pytest.mark.gpu

FAST32 = (32, ((0, 3), (16, 3)))    # terrain_vertices_k<*, true>: one 32-byte store per vertex
GENERIC = (48, ((4, 3), (28, 3)))   # terrain_vertices_k<*, false>
SPECIAL_HS = (0.0, -0.0, 1e-40, E.FLT_MAX, np.inf)  # 1e-40 makes y subnormal


def _torch():
    import torch

    return torch


def _dev(x):
    torch = _torch()
    v = x.view(np.int16) if x.dtype == np.uint16 else x.view(np.int32) if x.dtype == np.uint32 else x
    return torch.from_numpy(np.ascontiguousarray(v)).cuda()


def _params(p):
    return (C.c_float * 3)(*p)


# ---- cull -----------------------------------------------------------------------------------------------------------------
def _gpu_cull(ctx, boxes, n, tr, tc, m, host):
    torch = _torch()
    ntiles = ((n - 1 + tr - 1) // tr) * ((n - 1 + tc - 1) // tc)
    m = np.ascontiguousarray(m, dtype=np.float32)
    if host:
        b = np.ascontiguousarray(boxes, dtype=np.float32)
        vis, ids = np.zeros(ntiles, np.uint32), np.zeros(ntiles, np.uint32)
        idx = np.full(6 * (n - 1) * (n - 1), 0xFFFFFFFF, np.uint32)
        cnt = np.zeros(2, np.uint64)
        ptr = lambda a: a.ctypes.data
    else:
        b = boxes if isinstance(boxes, torch.Tensor) else _dev(np.ascontiguousarray(boxes, dtype=np.float32).reshape(-1))
        vis = torch.empty(ntiles, dtype=torch.int32, device="cuda")
        ids = torch.empty(ntiles, dtype=torch.int32, device="cuda")
        idx = torch.full((6 * (n - 1) * (n - 1),), -1, dtype=torch.int32, device="cuda")
        cnt = torch.zeros(2, dtype=torch.int64, device="cuda")
        ptr = lambda a: a.data_ptr()
    ctx.check(ctx.lib.mr_terrain_cull(ctx.handle, ptr(b), n, tr, tc, m.ctypes.data, ptr(vis), ptr(ids), ptr(idx), ptr(cnt)), "cull")
    ctx.sync()
    if host:
        return vis, ids, idx, cnt
    return tuple(a.cpu().numpy().view(np.uint64 if a.dtype == torch.int64 else np.uint32) for a in (vis, ids, idx, cnt))


def _check_cull(ctx, oracle, boxes, n, tr, tc, m, what, gpu_boxes=None):
    """GPU cull of `boxes` (or of the device tensor gpu_boxes holding them) against the oracle, device and host pointers."""
    ref = oracle.terrain_cull(boxes, n, tr, tc, m)
    for host in (False, True):
        vis, ids, idx, cnt = _gpu_cull(ctx, boxes if host or gpu_boxes is None else gpu_boxes, n, tr, tc, m, host)
        where = (what, "host" if host else "device")
        assert cnt.tolist() == ref["counts"].tolist(), where
        assert np.array_equal(vis, ref["visible"]), (where, np.nonzero(vis != ref["visible"])[0][:8])
        assert np.array_equal(ids[: int(cnt[0])], ref["ids"]), where
        assert np.array_equal(idx[: int(cnt[1])], ref["idx"]) and (idx[int(cnt[1]):] == 0xFFFFFFFF).all(), where
    return ref


def test_cull_near_thresholds_and_nonfinite_boxes(ctx, oracle):
    """Every generated box in a terrain of 40 x 29 = 1160 tiles: the scan of terrain_cull_k runs two chunks of 1024, and
    the last tile row and column are ragged (199 quads = 39 * 5 + 4 = 28 * 7 + 3)."""
    n, tr, tc = 200, 5, 7
    tiles_r, tiles_c = oracle.tile_count(n, tr, tc)
    ntiles = tiles_r * tiles_c
    assert ntiles > 1024 and (n - 1) % tr and (n - 1) % tc
    flips = 0
    for kind, m, boxes in E.cull_cases():
        order = np.arange(-(-len(boxes) // ntiles) * ntiles) % len(boxes)
        for k, chunk in enumerate(order.reshape(-1, ntiles)):
            ref = _check_cull(ctx, oracle, boxes[chunk], n, tr, tc, m, (kind, k))
            flips += int(0 < ref["visible"].sum() < ntiles)
    assert flips > 0


# ---- mesh -----------------------------------------------------------------------------------------------------------------
def _gpu_build(ctx, h, n, layout, params, rows=None):
    """Device build of rows [rows) (all by default) from a band-local height buffer (the band plus its halo), written to a
    band-local vertex buffer; the quad rows of the same band to a band-local index buffer."""
    import myrenderer_b200 as mr

    torch = _torch()
    r0, r1 = rows or (0, n)
    q0, q1 = r0, min(r1, n - 1)
    lo, hi = max(r0 - 1, 0), min(r1 + 1, n)
    stride = layout[0]
    vtx = torch.full(((r1 - r0) * n * stride,), 0x5A, dtype=torch.uint8, device="cuda")
    idx = torch.full((max((q1 - q0) * 6 * (n - 1), 2),), -1, dtype=torch.int32, device="cuda")
    T = mr.Terrain(ctx, mr.VertexLayout(layout[0], layout[1]), params)
    hd = _dev(np.ascontiguousarray(h[lo:hi]))
    T.build(T.job(hd, n, rows=(r0, r1), qrows=(q0, q1), height_row0=lo, height_rows=hi - lo, vtx_out=vtx, vtx_row0=r0,
                  idx_out=idx, idx_qrow0=q0))
    ctx.sync()
    return vtx.cpu().numpy(), idx.cpu().numpy().view(np.uint32)[: (q1 - q0) * 6 * (n - 1)], (r0, r1), (q0, q1)


def _check_build(ctx, oracle, h, n, layout, params, rows=None, nan_log=None):
    gv, gi, rows, qrows = _gpu_build(ctx, h, n, layout, params, rows)
    ov, oi = oracle.terrain_build(h, n, layout=layout, params=params, rows=rows, qrows=qrows, nthreads=0)
    mask = E.vertex_float_mask(gv.size, layout)
    what = (h.dtype.name, layout, params, rows)
    assert E.float_mismatch(gv, ov, mask) is None, (what, E.float_mismatch(gv, ov, mask))
    assert np.array_equal(gi, oi), what
    if nan_log is not None:
        nan_log.update(E.nan_words(gv, mask))


def test_build_special_heightmap(ctx, oracle):
    """FAST32 and a generic layout; grid_step 0.2 (constant-divisor quotients) and 0.3 (IEEE division); the whole mesh and
    a row band built from its band-local heights with a one-row halo."""
    n = 600
    h = E.special_heightmap(np.random.default_rng(11), n, ((8, 24), (16, 520)))
    nans = set()
    for layout in (FAST32, GENERIC):
        for gs in (0.2, 0.3):
            for rows in (None, (137, 291)):
                _check_build(ctx, oracle, h, n, layout, (gs, 0.1, 5.0), rows, nans)
    print("NaN words written by the vertex kernel:", " ".join("0x%08x" % w for w in sorted(nans)))
    assert nans  # the map does produce NaN outputs (see test_float_edges_cpu)


def _u16_map(n):
    from oracle import oracle as O

    h = O.synth_heightmap_u16(0x5EED0E01, n)
    h[0, :] = 0          # height 1
    h[2, :] = 65535      # height +0
    h[5, 3::7] = 65535
    return h


def _f32_map(n):
    return E.special_heightmap(np.random.default_rng(n), n, ((8, 24), (16, 600)))


def test_special_height_scales_build(ctx, oracle):
    """height_scale 0, -0, 1e-40, FLT_MAX and +inf on u16 and f32 maps, through both layouts (four vertex kernels)."""
    n = 301
    for h in (_u16_map(n), _f32_map(n)):
        for hs in SPECIAL_HS:
            for layout in (FAST32, GENERIC):
                _check_build(ctx, oracle, h, n, layout, (0.2, 0.1, hs))


# (n, tile_rows, tile_cols) -> kernel for u16 maps; f32 maps take the generic strip kernel for tile_cols <= 512
TILE_CASES_U16 = ((301, 8, 24),    # terrain_tile_bounds_strip_k<true, false>: n odd
                  (302, 8, 10),    # terrain_tile_bounds_strip_k<true, true> (PAIR): n and tile_cols even, n % 8 != 0
                  (304, 8, 16),    # terrain_tile_bounds_wide_k: n and the strip width multiples of 8
                  (700, 8, 600))   # terrain_tile_bounds_k<true>: tile_cols > 512
TILE_CASES_F32 = ((301, 8, 24), (700, 16, 600))


def _gpu_tile_bounds(ctx, hd, fmt, n, tr, tc, params):
    torch = _torch()
    tiles_r, tiles_c = (n - 1 + tr - 1) // tr, (n - 1 + tc - 1) // tc
    bd = torch.full((tiles_r * tiles_c * 8,), -1, dtype=torch.int32, device="cuda").view(torch.float32)
    ctx.check(ctx.lib.mr_terrain_tile_bounds(ctx.handle, hd.data_ptr(), fmt, n, tr, tc, _params(params), bd.data_ptr()), "tile bounds")
    ctx.sync()
    return bd


def _check_tile_bounds(ctx, oracle, h, n, tr, tc, params):
    bd = _gpu_tile_bounds(ctx, _dev(h), 0 if h.dtype == np.uint16 else 1, n, tr, tc, params)
    got = bd.cpu().numpy().reshape(-1, 8)
    want = oracle.terrain_tile_bounds(h, n, tr, tc, params)
    assert E.float_mismatch(got, want) is None, ((h.dtype.name, n, tr, tc, params), E.float_mismatch(got, want))
    return bd, got


def test_special_height_scales_tile_bounds(ctx, oracle):
    for hs in SPECIAL_HS:
        for n, tr, tc in TILE_CASES_U16:
            _check_tile_bounds(ctx, oracle, _u16_map(n), n, tr, tc, (0.2, 0.1, hs))
        for n, tr, tc in TILE_CASES_F32:
            _check_tile_bounds(ctx, oracle, _f32_map(n), n, tr, tc, (0.2, 0.1, hs))


def test_tile_bounds_of_special_heightmap_then_cull(ctx, oracle):
    """Boxes of a map with NaN tiles and +-inf heights, through the strip kernel (tile_cols <= 512) and the generic one
    (tile_cols > 512); then the GPU's own boxes -- y bounds of -inf, +inf and NaN among them -- go to the cull, so that the
    +-inf skip rule is reached from real data."""
    from test_terrain_cull_cpu import camera_matrix

    n = 600
    tiles = ((8, 24), (16, 520))
    h = E.special_heightmap(np.random.default_rng(12), n, tiles)
    rng = np.random.default_rng(13)
    mats = [camera_matrix(), camera_matrix((5.0, 60.0, 5.0), (40.0, 0.0, 40.0))] + [rng.normal(size=16).astype(np.float32) for _ in range(3)]
    nonfinite, nans = 0, set()
    for tr, tc in tiles:
        for hs in (5.0, -5.0, 0.0):
            bd, got = _check_tile_bounds(ctx, oracle, h, n, tr, tc, (0.2, 0.1, hs))
            nonfinite += int((~np.isfinite(got[:, [1, 5]])).any(1).sum())
            nans.update(E.nan_words(got))
            for k, m in enumerate(mats):
                _check_cull(ctx, oracle, got, n, tr, tc, m, (tr, tc, hs, k), gpu_boxes=bd)
    print("NaN words written by the tile-box kernels:", " ".join("0x%08x" % w for w in sorted(nans)))
    assert nonfinite > 0 and nans
