"""The terrain kernels at their size limit, n = 65535: the sizes, rows and tile shapes that tests/test_gpu_terrain_limits.py
runs, and the references it compares with.  tests/test_terrain_limits_cpu.py checks these lists and references on the CPU.

- The quad-row division of terrain_indices_k, q = (Q * div_magic) >> 48, and the condition under which a multiply-shift
  is exact for every quad of an n x n terrain.
- The choice of tile-bounds kernel made by mr_terrain_tile_bounds_impl.
- A torch restatement of the tile boxes for a map held on the device.  The C oracle walks the whole map on one thread,
  which takes seconds per tiling at 65535^2, so it only validates this restatement, on small maps.
"""
import numpy as np

N_MAX = 65535
SEED = 0x5EED0065

# Every size runs the whole index buffer; the first two also run the vertex bands, the tile boxes and the cull.
SIZES = (
    65535,  # the limit; odd: the u16 strip kernel, the per-tile kernel and the f32 strip kernel
    65528,  # a multiple of 8: terrain_tile_bounds_wide_k and the PAIR strip kernel
    52187,  # the first n at which a 47-bit multiply-shift gives some quad the wrong row
    46341,  # the first n with n^2 > 2^31: texel and vertex indices past the int32 range
    32801,  # the first n at which a 45-bit multiply-shift fails
    16417,  # the first n at which a 42-bit multiply-shift fails
    8193,   # the first n whose single-tile cull has more than 65535 chunks of 1024 quads
)
# Sizes the rest of the suite builds whole (test_gpu_parity.py, scripts/fuzz_terrain.py, test_gpu_fullsize.py).
OLD_SIZES = tuple(range(1, 1601)) + (4096, 16384)

VERTEX_SIZES = (65535, 46341)  # maps resident on the device with height_row0 = 0
TILE_SIZES = (65535, 65528)
# (tile_rows, tile_cols) at TILE_SIZES, u16 and f32 maps.  None divides n - 1, so every last tile row and column is ragged.
TILE_SHAPES = (
    (64, 64),     # n = 65528: wide; n = 65535: u16 strip; f32: f32 strip
    (100, 10),    # n = 65528: PAIR strip (51 tiles of 10 columns per strip: 510 is no multiple of 8)
    (65535, 256), # taller than the terrain: one tile row, 65534 rows walked per strip
    (700, 600),   # tile_cols > 512: one CTA per tile
)
# The same shapes on small maps for the CPU check of the restatement, and shapes only a small map can afford.
CPU_TILE_SIZES = (1999, 2000)
CPU_TILE_SHAPES = TILE_SHAPES + ((1, 1), (7, 3), (3000, 3000), (1999, 1), (2, 5000))

TB_COLS = 512  # columns per strip of the tile-bounds strip kernels (terrain.cu)
TI_QUADS = 1024  # quads per chunk of terrain_indices_k and terrain_cull_indices_k
OLD_CULL_CHUNK_LIMIT = 65535  # the cull used to launch one CTA row per chunk and refuse more


def bands(n):
    """Row bands [r0, r1) of the vertex tests: the first rows, rows 16383..16386 and 32767..32770 (where texel offsets
    cross 2^32 bytes of f32 and 2^31 texels), and the last 9 rows.  No height is a multiple of the 8 rows of a vertex
    tile, so each band ends in a ragged tile."""
    out = [(0, 5), (16383, 16387), (32767, 32771), (n - 9, n)]
    return [b for b in out if b[1] <= n and b[0] >= 0]


# ---- the quad-row division of terrain_indices_k -------------------------------------------------------------------------
def div_magic(n, k=48):
    """floor(2^k / (n-1)) + 1, as terrain.cu computes it for k = 48."""
    return (1 << k) // (n - 1) + 1


def shift_is_exact(n, k=48):
    """(Q * m) >> k == Q // d for every quad Q < d^2 (d = n - 1, m = div_magic) exactly when d (m d - 2^k) < m, i.e.
    (d^2 - 1)(m d - 2^k) < 2^k: the error term Q (m d - 2^k) / (d 2^k) of the last quad of the last row must not
    reach the 1/d left by its remainder d - 1."""
    d, m = n - 1, div_magic(n, k)
    return d * (m * d - (1 << k)) < m


def first_wrong_quad(n, k):
    """The first quad Q whose row (Q * m) >> k is wrong, or None.  Only quads at the end of a row (remainder d - 1) fail
    first: the smallest such Q with Q (m d - 2^k) >= 2^k."""
    d = n - 1
    e = div_magic(n, k) * d - (1 << k)
    qmin = -(-(1 << k) // e)
    q = max(0, -(-(qmin - (d - 1)) // d))
    Q = q * d + d - 1
    return Q if Q < d * d else None


def quad_row_shift(Q, n, k=48):
    """(Q * m) >> k in 64-bit unsigned arithmetic (numpy uint64 or Python ints), as the kernel does."""
    if isinstance(Q, np.ndarray):
        return (Q.astype(np.uint64) * np.uint64(div_magic(n, k))) >> np.uint64(k)
    return ((Q * div_magic(n, k)) & 0xFFFFFFFFFFFFFFFF) >> k


def quad_row_float(Q, n):
    """(uint32_t)((float)Q / (float)(n - 1)): a float division instead of the multiply-shift."""
    q = np.asarray(Q, dtype=np.uint64).astype(np.float64).astype(np.float32) / np.float32(n - 1)
    return q.astype(np.uint64)


def row_boundary_quads(n):
    """The last quad of every row and the first of the next: where a division that rounds the wrong way fails first."""
    d = n - 1
    q = np.arange(1, d, dtype=np.uint64) * np.uint64(d)
    return np.concatenate([q - np.uint64(1), q, np.array([d * d - 1], dtype=np.uint64)])


# ---- tile-bounds kernel choice (mr_terrain_tile_bounds_impl) --------------------------------------------------------------
def tile_count(n, tile_rows, tile_cols):
    return (n - 1 + tile_rows - 1) // tile_rows, (n - 1 + tile_cols - 1) // tile_cols


def tile_bounds_kernel(n, tile_rows, tile_cols, u16, base_align=256):
    """Which kernel mr_terrain_tile_bounds runs, for a map at an address aligned to base_align bytes (torch allocations
    are aligned to at least 256)."""
    tiles_r, _ = tile_count(n, tile_rows, tile_cols)
    if tile_cols <= TB_COLS and tiles_r <= 65535:
        per = max(1, TB_COLS // tile_cols)
        pair = u16 and n % 2 == 0 and tile_cols % 2 == 0 and base_align % 4 == 0
        wide = u16 and n % 8 == 0 and (per * tile_cols) % 8 == 0 and base_align % 16 == 0
        if wide:
            return "wide"
        if pair:
            return "pair_strip"
        return "u16_strip" if u16 else "f32_strip"
    return "per_tile"


TILE_KERNELS = ("wide", "pair_strip", "u16_strip", "f32_strip", "per_tile")


# ---- tile boxes -------------------------------------------------------------------------------------------------------------
def u16_height_table(oracle):
    """height(v) = 1 - v / 65535 for all 65536 texels, from the oracle."""
    return oracle.heightmap_normalize(np.arange(65536, dtype=np.uint16))


def tile_extremes(h, n, tile_rows, tile_cols, rows_per_step=2048):
    """Per-tile minimum and maximum texel over the inclusive vertex ranges r0..r1, c0..c1 (boundary rows and columns are
    shared by neighbouring tiles).  h: torch tensor of n*n texels, int16 holding raw u16 values (compared unsigned) or
    float32 without NaN, on any device.  Returns (lo, hi) of shape [tiles], int32 texels or float32 heights."""
    import torch

    u16 = h.dtype == torch.int16
    H = h.view(n, n)
    tiles_r, tiles_c = tile_count(n, tile_rows, tile_cols)
    dt = torch.int32 if u16 else torch.float32
    big, small = (65535, 0) if u16 else (float("inf"), float("-inf"))
    cmin = torch.empty((tiles_r, n), dtype=dt, device=h.device)
    cmax = torch.empty((tiles_r, n), dtype=dt, device=h.device)
    for tr in range(tiles_r):  # rows: per tile row, the column-wise extremes of rows r0..r1
        r0 = tr * tile_rows
        r1 = min(r0 + tile_rows, n - 1)
        lo = hi = None
        for a in range(r0, r1 + 1, rows_per_step):
            x = H[a:min(a + rows_per_step, r1 + 1)]
            if u16:
                x = x.to(torch.int32) & 0xFFFF
            m0, m1 = x.amin(0), x.amax(0)
            lo = m0 if lo is None else torch.minimum(lo, m0)
            hi = m1 if hi is None else torch.maximum(hi, m1)
        cmin[tr], cmax[tr] = lo, hi
    # columns: tile tc takes columns [c0, min(c0 + tile_cols, n - 1)) as a block, plus its right boundary column c1
    width = tiles_c * tile_cols
    c1 = torch.clamp(torch.arange(1, tiles_c + 1, device=h.device) * tile_cols, max=n - 1)
    out = []
    for cm, pad, red, comb in ((cmin, big, torch.amin, torch.minimum), (cmax, small, torch.amax, torch.maximum)):
        blk = torch.full((tiles_r, width), pad, dtype=dt, device=h.device)
        blk[:, : n - 1] = cm[:, : n - 1]
        blk = red(blk.view(tiles_r, tiles_c, tile_cols), 2)
        out.append(comb(blk, cm[:, c1]).reshape(-1))
    return out[0], out[1]


def tile_boxes(h, n, tile_rows, tile_cols, params=(0.2, 0.1, 5.0), table=None):
    """[tiles, 8] float32 boxes as mr_terrain_tile_bounds writes them, restated: the texel extremes of tile_extremes, for
    a u16 map converted through `table` (u16_height_table: the smallest height is the height of the largest texel),
    then the box formula of write_tile_box (terrain.cu) in float32, every operation rounded on its own."""
    import torch

    lo, hi = tile_extremes(h, n, tile_rows, tile_cols)
    if h.dtype == torch.int16:
        lo, hi = table[hi.cpu().numpy()], table[lo.cpu().numpy()]
    else:
        lo, hi = lo.cpu().numpy(), hi.cpu().numpy()
    return box_formula(n, tile_rows, tile_cols, lo, hi, params)


def box_formula(n, tile_rows, tile_cols, lo, hi, params):
    """write_tile_box for every tile, from the height extremes lo, hi ([tiles] float32)."""
    f = np.float32
    gs, osc, hs = (f(p) for p in params)
    tiles_r, tiles_c = tile_count(n, tile_rows, tile_cols)
    r0 = np.arange(tiles_r, dtype=np.int64) * tile_rows
    c0 = np.arange(tiles_c, dtype=np.int64) * tile_cols
    r1, c1 = np.minimum(r0 + tile_rows, n - 1), np.minimum(c0 + tile_cols, n - 1)
    org = f(osc * f(n))
    pos = lambda v: (gs * v.astype(np.float32)) - org
    xa, xb, za, zb = pos(r0), pos(r1), pos(c0), pos(c1)
    xa, xb = np.repeat(xa, tiles_c), np.repeat(xb, tiles_c)
    za, zb = np.tile(za, tiles_r), np.tile(zb, tiles_r)
    ya, yb = hs * lo.astype(np.float32), hs * hi.astype(np.float32)
    y0, y1 = np.where(yb < ya, yb, ya), np.where(yb > ya, yb, ya)
    y0, y1 = np.where(y0 == 0, f(0), y0), np.where(y1 == 0, f(0), y1)
    one = np.ones_like(y0)
    return np.stack([np.where(xb < xa, xb, xa), y0, np.where(zb < za, zb, za), one,
                     np.where(xb > xa, xb, xa), y1, np.where(zb > za, zb, za), one], axis=1).astype(np.float32)


# ---- boxes for the cull ---------------------------------------------------------------------------------------------------
IDENTITY = np.eye(4, dtype=np.float32).reshape(16)
VISIBLE_BOX = np.array([0, 0, 0, 0, 1, 1, 1, 1], dtype=np.float32)     # q1 = p1 > 0 under the identity
HIDDEN_BOX = np.array([2, 2, 2, 2, -1, -1, -1, -1], dtype=np.float32)  # q1 <= 0 and q0 >= 1


CULL_TILE = (64, 64)  # at N_MAX: 1024 x 1024 tiles, all visible, then those of the last tile row and column
CULL_SINGLE = ((8193, 8192), (8193, 65535), (16384, 16383), (16384, 65535))  # (n, tile size): one tile, the whole terrain
CULL_CHUNK_SHAPES = ((65534, 1024), (65534, 1025))  # at N_MAX: 65534 and 65598 chunks in a full tile


def cull_chunk_visible(tiles_c):
    """Visible tiles of the CULL_CHUNK_SHAPES runs (one tile row): the first, the last full one and the ragged last."""
    return (0, tiles_c - 2, tiles_c - 1)


def cull_boxes(visible):
    """[tiles, 8] boxes whose visibility under IDENTITY is `visible` ([tiles] bool) by construction."""
    visible = np.asarray(visible, dtype=bool)
    return np.where(visible[:, None], VISIBLE_BOX[None, :], HIDDEN_BOX[None, :]).astype(np.float32)
