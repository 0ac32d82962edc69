"""CPU checks of the float-edge cases of tests/_float_edges.py: the numpy model of the cull's visibility test is the
oracle's, the generated boxes tell every plausible wrong implementation apart from it, and the special heightmap drives
the oracle's mesh and tile boxes to subnormal, infinite and NaN outputs.  These keep tests/test_gpu_float_edges.py able
to fail."""
import numpy as np
import pytest

import _float_edges as E

PARAMS = (0.2, 0.1, 5.0)


@pytest.fixture(scope="module")
def cases():
    return E.cull_cases()


def test_contract_model_is_the_oracle(oracle, cases):
    total = 0
    for kind, m, boxes in cases:
        want = E.oracle_should_render(oracle, m, boxes)
        got = E.should_render(m, boxes)
        assert np.array_equal(got, want), (kind, np.nonzero(got != want)[0][:10])
        for b in boxes[:: max(1, len(boxes) // 40)]:  # and box by box through the single-box entry point
            assert oracle.scene_node_should_render(m, b[:4], b[4:]) == bool(E.should_render(m, b)[0])
        total += len(boxes)
    assert total > 1000


def test_every_mutant_is_told_apart(cases):
    told = {mu: 0 for mu in E.MUTANTS}
    for _, m, boxes in cases:
        want = E.should_render(m, boxes)
        for mu in E.MUTANTS:
            told[mu] += int((E.should_render(m, boxes, mu) != want).sum())
    msg = ", ".join("%s: %d" % kv for kv in told.items())
    assert all(told[mu] >= 3 for mu in E.MUTANTS if mu not in E.EQUIVALENT_MUTANTS), msg
    assert all(told[mu] == 0 for mu in E.EQUIVALENT_MUTANTS), msg


def test_cases_cover_every_matrix_kind_and_nonfinite_slot(cases):
    assert {k for k, _, _ in cases} == {"camera", "normal", "subnormal", "huge", "zeros"}
    for _, _, boxes in cases:
        for s in range(8):
            col = boxes[:, s]
            assert np.isnan(col).any() and (col == np.inf).any() and (col == -np.inf).any()
    negz = sum(int((np.isfinite(b).all(1) & (b.view(np.uint32) == 0x80000000).any(1)).sum()) for _, _, b in cases)
    assert negz >= 10, negz  # finite boxes with -0 components that tell some mutant apart


def test_fma_model_rounds_once():
    a = np.float32(1 + 2.0 ** -12)
    b = np.array([1 + 2.0 ** -12], dtype=np.float32)
    c = np.array([-1.0], dtype=np.float32)
    # a*b + c = 2^-11 + 2^-24 exactly; the separately rounded form loses the 2^-24
    assert E._fma(a, b, c)[0] == np.float32(2.0 ** -11 + 2.0 ** -24)
    assert np.float32(a * b[0]) + c[0] == np.float32(2.0 ** -11)
    # the tie that f64-then-f32 rounds wrongly: 1 + 2^-24 + 2^-60 must round up
    from fractions import Fraction
    assert E.round_f32(Fraction(1) + Fraction(1, 2 ** 24) + Fraction(1, 2 ** 60)) == np.nextafter(np.float32(1), np.float32(2))
    assert np.float32(np.float64(1) + 2.0 ** -24 + 2.0 ** -60) == np.float32(1)
    assert E.round_f32(Fraction(2) ** -150 * 3) == E.f32_from_bits(2)  # subnormal, tie to even
    assert E.round_f32(Fraction(2) ** 128) == np.inf


def _special_outputs(oracle, n, tiles, seed):
    h = E.special_heightmap(np.random.default_rng(seed), n, tiles)
    vtx, _ = oracle.terrain_build(h, n, params=PARAMS, want_idx=False)
    boxes = {hs: np.concatenate([oracle.terrain_tile_bounds(h, n, tr, tc, PARAMS[:2] + (hs,)).reshape(-1) for tr, tc in tiles])
             for hs in (5.0, 0.0)}
    return h, vtx.view(np.float32), boxes


def _kinds(x):
    x = np.asarray(x, dtype=np.float32).reshape(-1)
    return {"subnormal": bool(((x != 0) & (np.abs(x) < E.MIN_NORMAL)).any()), "inf": bool(np.isinf(x).any()),
            "nan": bool(np.isnan(x).any())}


def test_special_heightmap_reaches_the_edges(oracle):
    """The mesh and the tile boxes of the map the GPU test uses hold subnormal, infinite and NaN outputs, and some box has
    a -inf y bound (a tile of NaNs only, or one holding -inf)."""
    n, tiles = 600, ((8, 24), (16, 520))
    h, vtx, boxes = _special_outputs(oracle, n, tiles, 1)
    w = h.view(np.uint32)
    assert {int(v) for v in E.NAN_WORDS} <= set(np.unique(w).tolist())
    pos = vtx.reshape(n * n, 8)[:, :3]
    nrm = vtx.reshape(n * n, 8)[:, 4:7]
    assert _kinds(pos) == {"subnormal": True, "inf": True, "nan": True}, _kinds(pos)
    assert _kinds(nrm) == {"subnormal": True, "inf": False, "nan": True}, _kinds(nrm)  # a unit normal is never infinite
    got = {k: _kinds(boxes[5.0])[k] or _kinds(boxes[0.0])[k] for k in ("subnormal", "inf", "nan")}
    assert got == {"subnormal": True, "inf": True, "nan": True}, got
    y0 = np.concatenate([b.reshape(-1, 8)[:, 1] for b in boxes.values()])
    assert (y0 == -np.inf).any()
    # differences reach both sides of the guarded range of the constant-divisor quotient: |5 * d| in [2^-63, 2^64)
    with np.errstate(all="ignore"):
        d = np.abs(np.float32(5.0) * (h[:, 2:] - h[:, :-2]))
    fin = d[np.isfinite(d)]
    for edge in (2.0 ** -63, 2.0 ** 64):
        assert ((fin < edge) & (fin > edge / 2)).any() and ((fin >= edge) & (fin < edge * 2)).any(), edge


def test_special_heightmap_tiles(oracle):
    """The all-NaN tile gives the box y range (-inf, +inf) at height_scale 5, and NaN at height_scale 0 (0 * inf)."""
    n, tr, tc = 200, 8, 24
    h = E.special_heightmap(np.random.default_rng(2), n, ((tr, tc),))
    b5 = oracle.terrain_tile_bounds(h, n, tr, tc, PARAMS)
    b0 = oracle.terrain_tile_bounds(h, n, tr, tc, PARAMS[:2] + (0.0,))
    tiles_r, tiles_c = oracle.tile_count(n, tr, tc)
    allnan = np.array([np.isnan(h[a * tr: a * tr + tr + 1, b * tc: b * tc + tc + 1]).all()
                       for a in range(tiles_r) for b in range(tiles_c)])
    assert allnan.any()
    assert (b5[allnan][:, 1] == -np.inf).all() and (b5[allnan][:, 5] == np.inf).all()
    assert np.isnan(b0[allnan][:, [1, 5]]).all()


def test_float_mismatch_comparator():
    a = np.array([0x7FC00000, 0x3F800000, 0], dtype=np.uint32)
    b = np.array([0x7FFFFFFF, 0x3F800000, 0], dtype=np.uint32)
    mask = np.array([True, True, False])
    assert E.float_mismatch(a, b, mask) is None
    assert E.float_mismatch(a, b, ~mask) is not None  # NaNs outside the float words must match exactly
    c = b.copy()
    c[0] = 0x7F800000  # NaN against a number (inf)
    assert E.float_mismatch(a, c, mask) is not None
    c = b.copy()
    c[1] = 0x3F800001
    assert "word 1" in E.float_mismatch(a, c, mask)
    c = a.copy()
    c[2] = 0x7FC00000  # a NaN in a padding word
    assert E.float_mismatch(c, a, mask) is not None
    assert E.vertex_float_mask(64, (32, ((0, 3), (16, 3)))).tolist() == [True] * 3 + [False] + [True] * 3 + [False] + \
        [True] * 3 + [False] + [True] * 3 + [False]
