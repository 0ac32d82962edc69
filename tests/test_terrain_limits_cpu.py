"""The size-limit lists and references of tests/_terrain_limits.py, checked without a GPU: the multiply-shift of
terrain_indices_k is exact for every quad of every n <= 65535 and weaker shifts are caught by the GPU sizes, the bands
and sizes cross every integer threshold of terrain.cu, the tile shapes reach every tile-bounds kernel, and the torch
restatement of the tile boxes equals the C oracle bit for bit."""
import numpy as np
import pytest

import _terrain_limits as L

MUTANT_SHIFTS = tuple(range(41, 48))
# the failure table of the 41..47-bit shifts: first n with a wrong quad row, and the first wrong row at n = 65535
SHIFT_TABLE = {41: (13081, 528), 42: (16417, 1092), 43: (20711, 2340), 44: (26141, 5461), 45: (32801, 16385),
               46: (41336, 16385), 47: (52187, 32772)}


# ---- the multiply-shift ---------------------------------------------------------------------------------------------------
def test_multiply_shift_is_exact_up_to_the_limit():
    """For every n in 2..65535 the 48-bit shift gives every quad its row, and the 64-bit product cannot wrap."""
    margins = []
    for n in range(2, L.N_MAX + 1):
        d, m = n - 1, L.div_magic(n)
        assert L.shift_is_exact(n), n
        assert (d * d - 1) * m < 1 << 64, n
        margins.append(m - d * (m * d - (1 << 48)))
    assert int(np.argmin(margins)) + 2 == L.N_MAX  # the thinnest margin is at the limit


def test_condition_matches_direct_evaluation_small_d():
    """For every n up to 301 and every shift 20..48, the condition holds exactly when every quad Q < d^2 gets Q // d,
    and first_wrong_quad names the first quad that does not."""
    for n in range(2, 302):
        d = n - 1
        Q = np.arange(d * d, dtype=np.uint64)
        want = Q // np.uint64(d)
        for k in range(20, 49):
            wrong = np.nonzero(L.quad_row_shift(Q, n, k) != want)[0]
            assert L.shift_is_exact(n, k) == (wrong.size == 0), (n, k)
            assert L.first_wrong_quad(n, k) == (int(wrong[0]) if wrong.size else None), (n, k)


@pytest.mark.parametrize("k", MUTANT_SHIFTS)
def test_first_wrong_quad_matches_direct_evaluation(k):
    """At the predicted first failing quad of each weaker shift, at the first failing n and at n = 65535, direct evaluation
    is wrong; one quad earlier, and at the end of every earlier row (the only quads that can fail first), it is right."""
    first_n, row_at_limit = SHIFT_TABLE[k]
    assert next(n for n in range(2, L.N_MAX + 1) if not L.shift_is_exact(n, k)) == first_n
    assert all(L.first_wrong_quad(n, k) is None for n in range(2, first_n))
    for n in (first_n, L.N_MAX):
        d = n - 1
        Q = L.first_wrong_quad(n, k)
        assert Q is not None and Q % d == d - 1
        assert L.quad_row_shift(Q, n, k) != Q // d
        assert L.quad_row_shift(Q - 1, n, k) == (Q - 1) // d
        ends = np.arange(Q // d, dtype=np.uint64) * np.uint64(d) + np.uint64(d - 1)
        assert np.array_equal(L.quad_row_shift(ends, n, k), ends // np.uint64(d))
    assert L.first_wrong_quad(L.N_MAX, k) // (L.N_MAX - 1) == row_at_limit


def _witness(n, mutant):
    """A quad of an n x n terrain that the mutant gives the wrong row, or None."""
    if mutant == "float":
        Q = L.row_boundary_quads(n)
        bad = np.nonzero(L.quad_row_float(Q, n) != Q // np.uint64(n - 1))[0]
        return int(Q[bad[0]]) if bad.size else None
    return L.first_wrong_quad(n, mutant)


def test_kill_table():
    """Every weaker multiply-shift, and a float division, gives some quad the wrong row at some size of the GPU list; the
    sizes the rest of the suite builds whole (1..1600, 4096, 16384) catch none of the shifts but 40 bits."""
    mutants = (40,) + MUTANT_SHIFTS + ("float",)
    old = [n for n in L.OLD_SIZES if n >= 2]
    print("\nfirst wrong quad row per quad-row mutant and size ('-': every quad right)")
    print("%-7s" % "mutant" + "".join("%8d" % n for n in L.SIZES) + "  old sizes")
    for mu in mutants:
        row = []
        for n in L.SIZES:
            w = _witness(n, mu)
            row.append("%8s" % ("-" if w is None else w // (n - 1)))
        old_kill = next((n for n in old if _witness(n, mu) is not None), None)
        print("%-7s" % (mu if mu == "float" else "k=%d" % mu) + "".join(row) + "  %s" % (old_kill or "-"))
        if mu != 40:
            assert any(_witness(n, mu) is not None for n in L.SIZES), mu
        if mu in MUTANT_SHIFTS:
            assert old_kill is None, (mu, old_kill)
    assert any(_witness(n, 40) is not None for n in old)


# ---- coverage of the thresholds -------------------------------------------------------------------------------------------
def _band_rows(n):
    """Texel rows a vertex band reads (the band plus its halo)."""
    return [(max(r0 - 1, 0), min(r1 + 1, n)) for r0, r1 in L.bands(n)]


def _crossed(n, rows, bound):
    """Some band holds a texel below `bound` (an element index) and one at or above it."""
    return any(lo * n < bound <= hi * n - 1 for lo, hi in rows)


def test_sizes_and_bands_cross_every_threshold():
    assert L.SIZES[0] == L.N_MAX and all(n <= L.N_MAX for n in L.SIZES)
    for n in L.VERTEX_SIZES:
        for r0, r1 in L.bands(n):
            assert (r1 - r0) % 8, (n, r0, r1)  # the last vertex tile of the band is ragged
    rows = _band_rows(L.N_MAX)
    assert _crossed(L.N_MAX, rows, 1 << 30)  # f32 texel byte offset 2^32
    assert _crossed(L.N_MAX, rows, 1 << 31)  # texel element index 2^31, u16 byte offset 2^32
    assert _crossed(46341, _band_rows(46341), 1 << 31)  # ... in the last row, at column 41708
    assert 46341 in L.VERTEX_SIZES and 46340 ** 2 < 1 << 31 < 46341 ** 2
    # index values >= 2^31: the whole index buffer of every size, among them n >= 46341
    assert any(n * n - 1 >= 1 << 31 for n in L.SIZES)
    # i00 = (r0+lr)*n + c0 + lc of the cull kernel near 2^32: the culls at the limit write the last tile, whose last
    # index n^2 - 1 is 2n + 2 short of 2^32
    n = L.N_MAX
    tiles_r, tiles_c = L.tile_count(n, *L.CULL_TILE)
    assert (1 << 32) - (n * n - 1) == 2 * n + 2
    tr, tc = L.CULL_CHUNK_SHAPES[0]
    assert L.cull_chunk_visible(L.tile_count(n, tr, tc)[1])[-1] == L.tile_count(n, tr, tc)[1] - 1
    # a total cull index count past 2^32 (64-bit scan): all tiles of the limit visible
    assert 6 * (n - 1) ** 2 > 1 << 32 and tiles_r * tiles_c == 1 << 20
    # chunks of 1024 quads in one full tile: one shape at the old launch limit, one past it; the single-tile culls past it
    chunks = [-(-min(tr, n - 1) * min(tc, n - 1) // L.TI_QUADS) for tr, tc in L.CULL_CHUNK_SHAPES]
    assert chunks[0] <= L.OLD_CULL_CHUNK_LIMIT < chunks[1]
    for m, t in L.CULL_SINGLE:
        assert L.tile_count(m, t, t) == (1, 1) and -(-(m - 1) ** 2 // L.TI_QUADS) > L.OLD_CULL_CHUNK_LIMIT
    assert -(-8191 ** 2 // L.TI_QUADS) <= L.OLD_CULL_CHUNK_LIMIT  # 8193 is the first size past it


def test_tile_shapes_reach_every_kernel():
    reached = {}
    for n in L.TILE_SIZES:
        for tr, tc in L.TILE_SHAPES:
            for u16 in (True, False):
                reached.setdefault(L.tile_bounds_kernel(n, tr, tc, u16), []).append((n, tr, tc, u16))
                tiles_r, tiles_c = L.tile_count(n, tr, tc)
                assert (n - 1) % tr and (n - 1) % tc, (n, tr, tc)  # ragged last tile row and column
    print("\n" + "\n".join("%-11s %s" % (k, v) for k, v in sorted(reached.items())))
    assert set(reached) == set(L.TILE_KERNELS)
    assert any(tr > n - 1 for n in L.TILE_SIZES for tr, _ in L.TILE_SHAPES)  # a tile taller than the terrain
    # the scaled-down shapes of the CPU check reach them too, and hold tiles larger than the terrain in both directions
    small = {L.tile_bounds_kernel(n, tr, tc, u16) for n in L.CPU_TILE_SIZES for tr, tc in L.CPU_TILE_SHAPES
             for u16 in (True, False)}
    assert small == set(L.TILE_KERNELS)
    assert any(tr > n - 1 and tc > n - 1 for n in L.CPU_TILE_SIZES for tr, tc in L.CPU_TILE_SHAPES)


# ---- the tile-box restatement ---------------------------------------------------------------------------------------------
def _maps(oracle, n):
    """A u16 noise map with both extreme texels, and f32 maps: its heights, and heights with signed zeros and values
    outside [0, 1]."""
    h = oracle.synth_heightmap_u16(L.SEED, n)
    h[0, 0], h[n - 1, n - 1], h[n // 2, 3] = 0, 65535, 65535
    f = oracle.heightmap_normalize(h)
    g = f.copy()
    g[::7, ::5] = -0.0
    g[3::11, ::3] = 0.0
    g[::13, 1::4] *= np.float32(-3e5)
    return h, (f, g)


@pytest.mark.parametrize("n", L.CPU_TILE_SIZES)
def test_tile_box_restatement_equals_oracle(oracle, n):
    import torch

    h, fmaps = _maps(oracle, n)
    table = L.u16_height_table(oracle)
    ht = torch.from_numpy(h.view(np.int16).reshape(-1))
    for tr, tc in L.CPU_TILE_SHAPES:
        for params in ((0.2, 0.1, 5.0), (0.3, 0.5, -2.0)):
            want = oracle.terrain_tile_bounds(h, n, tr, tc, params)
            got = L.tile_boxes(ht, n, tr, tc, params, table=table)
            assert np.array_equal(got.view(np.uint32), want.view(np.uint32)), ("u16", n, tr, tc, params)
            for f in fmaps:
                want = oracle.terrain_tile_bounds(f, n, tr, tc, params)
                got = L.tile_boxes(torch.from_numpy(f.reshape(-1)), n, tr, tc, params)
                assert np.array_equal(got.view(np.uint32), want.view(np.uint32)), ("f32", n, tr, tc, params)


def test_cull_boxes_and_oracle_idx_capacity(oracle):
    """The constructed boxes are visible exactly where asked, and the oracle's exact-size index buffer equals the full one."""
    n, tr, tc = 300, 64, 37
    tiles = int(np.prod(L.tile_count(n, tr, tc)))
    vis = np.zeros(tiles, dtype=bool)
    vis[[0, 5, tiles - 1]] = True
    boxes = L.cull_boxes(vis)
    full = oracle.terrain_cull(boxes, n, tr, tc, L.IDENTITY)
    small = oracle.terrain_cull(boxes, n, tr, tc, L.IDENTITY, idx_capacity=int(full["counts"][1]))
    assert np.array_equal(full["visible"], vis.astype(np.uint32))
    assert np.array_equal(full["idx"], small["idx"]) and np.array_equal(full["counts"], small["counts"])
    with pytest.raises(ValueError):
        oracle.terrain_cull(boxes, n, tr, tc, L.IDENTITY, idx_capacity=int(full["counts"][1]) - 1)
