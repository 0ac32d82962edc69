"""The terrain kernels at the size limit of the header, n = 65535: every quad of the index buffer at seven sizes up to the
limit, vertex bands read from whole resident maps at texel offsets past 2^31 and 2^32, a normalisation of more than 2^32
texels, the tile boxes of 65535^2 and 65528^2 maps, and culls with index counts past 2^32 and tiles of more than
65535 chunks.  Sizes, rows, shapes and the tile-box restatement come from tests/_terrain_limits.py, which
tests/test_terrain_limits_cpu.py checks.  Each large buffer is freed by the test that allocated it; the peak is about
30 GB."""
import gc
import sys
import traceback

import numpy as np
import pytest

import _terrain_limits as L

pytestmark = pytest.mark.gpu

FAST32 = (32, ((0, 3), (16, 3)))   # terrain_vertices_k<*, true>: one 32-byte store per vertex
GENERIC = (48, ((4, 3), (28, 3)))  # terrain_vertices_k<*, false>
PARAMS = ((0.2, 0.1, 5.0), (0.3, 0.1, 5.0))  # grid_step 0.2: reciprocal-and-correct quotients; 0.3: IEEE division
CHUNK_WORDS = 1 << 28  # about 1 GB of indices per call / comparison


def _torch():
    import torch

    return torch


@pytest.fixture(autouse=True)
def _release_gpu_memory():
    """A failing test's traceback keeps its frames, and with them tens of GB of tensors: clear them."""
    yield
    tb = getattr(sys, "last_traceback", None)
    if tb is not None:
        traceback.clear_frames(tb)
    gc.collect()
    _torch().cuda.empty_cache()


def _terrain(ctx, layout=FAST32, params=PARAMS[0]):
    import myrenderer_b200 as mr

    return mr.Terrain(ctx, layout=mr.VertexLayout(*layout), params=params)


def _synth_u16(ctx, n, seed=L.SEED):
    torch = _torch()
    h = torch.empty(n * n, dtype=torch.int16, device="cuda")
    ctx.check(ctx.lib.mr_synth_heightmap_u16(ctx.handle, seed, n, 0, n, h.data_ptr()), "synth")
    return h


def _normalize(ctx, h):
    torch = _torch()
    f = torch.empty(h.numel(), dtype=torch.float32, device="cuda")
    ctx.check(ctx.lib.mr_heightmap_normalize(ctx.handle, h.data_ptr(), h.numel(), f.data_ptr()), "normalize")
    return f


def _offsets(n):
    torch = _torch()
    return torch.tensor([n, 0, n + 1, n + 1, 0, 1], dtype=torch.int64, device="cuda")


def _as_u32(x):
    """int32 tensor -> int64 holding its words as unsigned values."""
    return x.to(_torch().int64) & 0xFFFFFFFF


def _check_rows_of_quads(got, n, r_lo, r_hi, c_lo, c_hi, what):
    """got (int32, device) holds the quads of rows [r_lo, r_hi) x columns [c_lo, c_hi), row-major, six words each:
    compare with i00 = r n + c in int64, in chunks of rows."""
    torch = _torch()
    qc = c_hi - c_lo
    step = max(1, CHUNK_WORDS // (6 * qc))
    off, c = _offsets(n), torch.arange(c_lo, c_hi, dtype=torch.int64, device="cuda")
    for a in range(r_lo, r_hi, step):
        b = min(a + step, r_hi)
        r = torch.arange(a, b, dtype=torch.int64, device="cuda")
        want = (r[:, None] * n + c[None, :])[:, :, None] + off
        g = _as_u32(got[(a - r_lo) * qc * 6:(b - r_lo) * qc * 6]).view(b - a, qc, 6)
        bad = (g != want).any(2).nonzero()
        assert bad.numel() == 0, (what, "first wrong quad (row, col)", (a + int(bad[0, 0]), c_lo + int(bad[0, 1])))


# ---- (a) every quad of the index buffer -----------------------------------------------------------------------------------
@pytest.mark.parametrize("n", L.SIZES)
def test_index_buffer_every_quad(ctx, n):
    """All (n-1)^2 quads, about 1 GB of indices per mr_terrain_build call (qrows = one chunk, idx_qrow0 = its first row,
    no vertices, so no map), each compared on the device with the closed form q = Q // (n-1), i00 = Q + q, read as
    unsigned.  idx_out alternates between 16-byte alignment and 8 mod 16 to cover the head and tail stores."""
    torch = _torch()
    d = n - 1
    rows = max(1, CHUNK_WORDS // (6 * d))
    buf = torch.empty(rows * 6 * d + 2, dtype=torch.int32, device="cuda")
    assert buf.data_ptr() % 16 == 0
    dummy = torch.zeros(1, dtype=torch.int16, device="cuda")
    T = _terrain(ctx)
    off = _offsets(n)
    for i, q0 in enumerate(range(0, d, rows)):
        q1 = min(q0 + rows, d)
        buf.fill_(-1)
        out = buf[2 * (i & 1):2 * (i & 1) + (q1 - q0) * 6 * d]
        T.build(T.job(dummy, n, rows=(0, 0), qrows=(q0, q1), height_rows=0, idx_out=out, idx_qrow0=q0))
        Q = torch.arange(q0 * d, q1 * d, dtype=torch.int64, device="cuda")
        want = (Q + Q // d)[:, None] + off
        bad = (_as_u32(out).view(-1, 6) != want).any(1).nonzero()
        assert bad.numel() == 0, (n, "first wrong quad", q0 * d + int(bad[0, 0]))
        del Q, want
    ctx.sync()
    del buf, dummy
    torch.cuda.empty_cache()


def test_index_buffer_one_launch_whole_range(ctx):
    """n = 16417 in one call: one launch whose quad counter runs over all 2.7e8 quads."""
    torch = _torch()
    n = 16417
    idx = torch.full((6 * (n - 1) ** 2,), -1, dtype=torch.int32, device="cuda")
    T = _terrain(ctx)
    T.build(T.job(torch.zeros(1, dtype=torch.int16, device="cuda"), n, rows=(0, 0), height_rows=0, idx_out=idx))
    _check_rows_of_quads(idx, n, 0, n - 1, 0, n - 1, "n = 16417, one launch")
    del idx
    torch.cuda.empty_cache()


# ---- (b) vertex bands of whole resident maps ------------------------------------------------------------------------------
@pytest.mark.parametrize("n,fmt", [(65535, "u16"), (65535, "f32"), (46341, "u16")])
def test_vertex_bands_whole_map(ctx, oracle, n, fmt):
    """The whole map on the device (8.6 GB u16 or 17 GB f32 at 65535) and height_row0 = 0, so that the kernel forms texel
    offsets past 2^31 texels and 2^32 bytes; band-local vtx_out.  Against the oracle on the band plus its halo."""
    torch = _torch()
    h = _synth_u16(ctx, n)
    if fmt == "f32":
        f = _normalize(ctx, h)
        del h
        h = f
        del f
    for r0, r1 in L.bands(n):
        lo, hi = max(r0 - 1, 0), min(r1 + 1, n)
        band = oracle.synth_heightmap_u16(L.SEED, n, lo, hi - lo)
        if fmt == "f32":
            band = oracle.heightmap_normalize(band)
        for layout in (FAST32, GENERIC):
            for params in PARAMS:
                T = _terrain(ctx, layout, params)
                vtx = torch.full(((r1 - r0) * n * layout[0],), 0xA5, dtype=torch.uint8, device="cuda")
                T.build(T.job(h, n, rows=(r0, r1), qrows=(0, 0), height_row0=0, height_rows=n, vtx_out=vtx, vtx_row0=r0))
                want, _ = oracle.terrain_build(band, n, layout=layout, params=params, rows=(r0, r1), qrows=(0, 0),
                                               height_row0=lo, want_idx=False, nthreads=0)
                got = vtx.cpu().numpy()
                if not np.array_equal(got, want):
                    v = np.nonzero((got != want).reshape(-1, layout[0]).any(1))[0]
                    pytest.fail(f"n={n} {fmt} rows {r0}..{r1} layout {layout[0]} params {params}: {v.size} vertices "
                                f"differ, first (row, col) {(r0 + int(v[0]) // n, int(v[0]) % n)}")
    del h, vtx
    torch.cuda.empty_cache()


# ---- (c) normalisation past 2^32 texels -----------------------------------------------------------------------------------
def test_heightmap_normalize_count_past_2_32(ctx, oracle):
    """2^32 + 4097 texels (8.6 GB in, 17 GB out): the output equals a gather from the 65536-entry table everywhere, the
    4097 texels past 2^32 included."""
    torch = _torch()
    count = (1 << 32) + 4097
    inp = torch.empty(65537 * 65536, dtype=torch.int16, device="cuda")
    ctx.check(ctx.lib.mr_synth_heightmap_u16(ctx.handle, L.SEED, 65536, 0, 65537, inp.data_ptr()), "synth")
    out = torch.full((count,), float("nan"), dtype=torch.float32, device="cuda")
    ctx.check(ctx.lib.mr_heightmap_normalize(ctx.handle, inp.data_ptr(), count, out.data_ptr()), "normalize")
    table = torch.from_numpy(L.u16_height_table(oracle).view(np.int32)).cuda()
    for a in range(0, count, CHUNK_WORDS):
        b = min(a + CHUNK_WORDS, count)
        want = table[inp[a:b].to(torch.int64) & 0xFFFF]
        bad = (out[a:b].view(torch.int32) != want).nonzero()
        assert bad.numel() == 0, ("first wrong texel", a + int(bad[0, 0]))
    assert count > 1 << 32 and int(out[-1].view(torch.int32)) == int(table[int(inp[count - 1]) & 0xFFFF])
    del inp, out, want
    torch.cuda.empty_cache()


# ---- (d) tile boxes at the limit ------------------------------------------------------------------------------------------
@pytest.mark.parametrize("n", L.TILE_SIZES)
def test_tile_bounds_at_the_limit(ctx, oracle, n):
    """Every shape of L.TILE_SHAPES on a u16 and an f32 map of n^2 texels against the restatement, bit for bit; the
    shapes reach the wide, PAIR strip, u16 strip, f32 strip and per-tile kernels between them."""
    torch = _torch()
    import ctypes as C

    table = L.u16_height_table(oracle)
    params = PARAMS[0]
    h = _synth_u16(ctx, n)
    for fmt in ("u16", "f32"):
        m = h if fmt == "u16" else _normalize(ctx, h)
        for tr, tc in L.TILE_SHAPES:
            tiles = int(np.prod(L.tile_count(n, tr, tc)))
            bd = torch.full((tiles * 8,), float("nan"), dtype=torch.float32, device="cuda")
            ctx.check(ctx.lib.mr_terrain_tile_bounds(ctx.handle, m.data_ptr(), 0 if fmt == "u16" else 1, n, tr, tc,
                                                     (C.c_float * 3)(*params), bd.data_ptr()), "tile bounds")
            want = L.tile_boxes(m, n, tr, tc, params, table=table)
            got = bd.cpu().numpy().reshape(-1, 8)
            bad = np.nonzero((got.view(np.uint32) != want.view(np.uint32)).any(1))[0]
            assert bad.size == 0, (n, fmt, (tr, tc), L.tile_bounds_kernel(n, tr, tc, fmt == "u16"), "tiles", bad[:8])
            del bd
        del m
        torch.cuda.empty_cache()
    del h
    torch.cuda.empty_cache()


# ---- (e) cull at the limit ------------------------------------------------------------------------------------------------
def _cull(ctx, boxes, n, tr, tc, *, host, want_idx_words=None, sentinel=64):
    """mr_terrain_cull of `boxes` under the identity.  host: visible / ids / counts (and the boxes) in host memory.  The
    index buffer, when asked for, is always on the device: a host idx_out stages 24 (n-1)^2 bytes of device memory."""
    torch = _torch()
    ntiles = boxes.shape[0]
    m = L.IDENTITY.copy()
    if host:
        b = np.ascontiguousarray(boxes)
        vis, ids, cnt = np.zeros(ntiles, np.uint32), np.zeros(ntiles, np.uint32), np.zeros(2, np.uint64)
        ptr = lambda a: a.ctypes.data
    else:
        b = torch.from_numpy(np.ascontiguousarray(boxes).reshape(-1)).cuda()
        vis = torch.full((ntiles,), -1, dtype=torch.int32, device="cuda")
        ids = torch.full((ntiles,), -1, dtype=torch.int32, device="cuda")
        cnt = torch.zeros(2, dtype=torch.int64, device="cuda")
        ptr = lambda a: a.data_ptr()
    idx = None
    if want_idx_words is not None:
        idx = torch.full((want_idx_words + sentinel,), -1, dtype=torch.int32, device="cuda")
    ctx.check(ctx.lib.mr_terrain_cull(ctx.handle, ptr(b), n, tr, tc, m.ctypes.data, ptr(vis), ptr(ids),
                                      None if idx is None else idx.data_ptr(), ptr(cnt)), "cull")
    ctx.sync()
    if not host:
        vis, ids, cnt = (a.cpu().numpy().view(np.uint64 if a.dtype == torch.int64 else np.uint32) for a in (vis, ids, cnt))
    return vis, ids, cnt, idx


def test_cull_all_tiles_visible_index_count_past_2_32(ctx):
    """n = 65535, 64 x 64 tiles, all 2^20 visible, no index buffer: counts[1] = 6 * 65534^2, past 2^32."""
    n, (tr, tc) = L.N_MAX, L.CULL_TILE
    ntiles = int(np.prod(L.tile_count(n, tr, tc)))
    boxes = L.cull_boxes(np.ones(ntiles, dtype=bool))
    for host in (False, True):
        vis, ids, cnt, _ = _cull(ctx, boxes, n, tr, tc, host=host)
        assert cnt.tolist() == [ntiles, 6 * (n - 1) ** 2], host
        assert (vis == 1).all() and np.array_equal(ids, np.arange(ntiles, dtype=np.uint32)), host


def test_cull_last_tile_row_and_column(ctx, oracle):
    """n = 65535, 64 x 64 tiles, only those of the last tile row and column visible: the compacted buffer holds values up
    to n^2 - 1 = 2^32 - 2n - 2 and equals the oracle's; device and host pointers for visible / ids / counts."""
    torch = _torch()
    n, (tr, tc) = L.N_MAX, L.CULL_TILE
    tiles_r, tiles_c = L.tile_count(n, tr, tc)
    vis_want = np.zeros((tiles_r, tiles_c), dtype=bool)
    vis_want[-1, :] = vis_want[:, -1] = True
    boxes = L.cull_boxes(vis_want.reshape(-1))
    ref = oracle.terrain_cull(boxes, n, tr, tc, L.IDENTITY, idx_capacity=1 << 28)
    words = int(ref["counts"][1])
    assert int(ref["idx"].max()) == n * n - 1
    want = torch.from_numpy(ref["idx"].view(np.int32)).cuda()
    for host in (False, True):
        vis, ids, cnt, idx = _cull(ctx, boxes, n, tr, tc, host=host, want_idx_words=words)
        assert cnt.tolist() == ref["counts"].tolist(), host
        assert np.array_equal(vis, ref["visible"]) and np.array_equal(ids[: int(cnt[0])], ref["ids"]), host
        assert torch.equal(idx[:words], want), host
        assert bool((idx[words:] == -1).all()), host
        del idx
    del want
    torch.cuda.empty_cache()


@pytest.mark.parametrize("n,t", L.CULL_SINGLE)
def test_cull_single_tile_whole_terrain(ctx, n, t):
    """One tile covering the terrain (tile size n - 1, or 65535: larger than the terrain) holds more than 65535 chunks of
    1024 quads.  The call succeeds, and its compacted buffer equals mr_terrain_build's index buffer (6.4 GB at 16384)."""
    torch = _torch()
    words = 6 * (n - 1) ** 2
    full = torch.empty(words, dtype=torch.int32, device="cuda")
    T = _terrain(ctx)
    T.build(T.job(torch.zeros(1, dtype=torch.int16, device="cuda"), n, rows=(0, 0), height_rows=0, idx_out=full))
    vis, ids, cnt, idx = _cull(ctx, L.cull_boxes([True]), n, t, t, host=False, want_idx_words=words)
    assert cnt.tolist() == [1, words] and vis.tolist() == [1] and ids.tolist() == [0]
    assert torch.equal(idx[:words], full)
    assert bool((idx[words:] == -1).all())
    del full, idx
    torch.cuda.empty_cache()


@pytest.mark.parametrize("shape", L.CULL_CHUNK_SHAPES)
def test_cull_chunks_around_the_old_launch_limit(ctx, shape):
    """n = 65535 with tiles of 65534 x 1024 quads (65534 chunks) and 65534 x 1025 (65598 chunks: more than one CTA row
    per chunk can count): the first tile, the last full one and the ragged last are visible; each tile's quads are
    compared with the closed form on the device."""
    torch = _torch()
    n, (tr, tc) = L.N_MAX, shape
    _, tiles_c = L.tile_count(n, tr, tc)
    vis_want = np.zeros(tiles_c, dtype=bool)
    vis_want[list(L.cull_chunk_visible(tiles_c))] = True
    cols = [(k * tc, min(k * tc + tc, n - 1)) for k in L.cull_chunk_visible(tiles_c)]
    words = sum(6 * (n - 1) * (c1 - c0) for c0, c1 in cols)
    vis, ids, cnt, idx = _cull(ctx, L.cull_boxes(vis_want), n, tr, tc, host=False, want_idx_words=words)
    assert cnt.tolist() == [3, words] and np.array_equal(vis, vis_want.astype(np.uint32))
    assert ids.tolist()[:3] == list(L.cull_chunk_visible(tiles_c))
    first = 0
    for c0, c1 in cols:
        size = 6 * (n - 1) * (c1 - c0)
        _check_rows_of_quads(idx[first:first + size], n, 0, n - 1, c0, c1, (shape, (c0, c1)))
        first += size
    assert bool((idx[words:] == -1).all())
    del idx
    torch.cuda.empty_cache()
