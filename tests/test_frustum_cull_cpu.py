"""CPU tests of the six-plane frustum test of mr_terrain_cull_frustum, on the oracle: the numpy model of tests/_frustum.py
equals it on every generated case, every wrong variant of the model is caught, the test is conservative in exact
arithmetic, and on a hash-noise terrain it keeps every tile with a vertex on screen, where the reference's test does not."""
import numpy as np
import pytest

import _frustum as F
import _frustum_oracle as FO
import _terrain_limits as L
from test_terrain_cull_cpu import camera_matrix


@pytest.fixture(scope="module")
def cases():
    return F.frustum_cases()


def test_model_equals_oracle_on_every_case(oracle, cases):
    total = 0
    for kind, m, boxes in cases:
        want = F.frustum_visible(m, boxes)
        got = F.oracle_visible(m, boxes)
        assert np.array_equal(got, want), (kind, np.nonzero(got != want)[0][:8])
        total += len(boxes)
        assert 0 < want.sum() < len(want), kind
    assert total > 4000
    # the per-box entry point agrees with the cull
    kind, m, boxes = cases[0]
    for b in boxes[:64]:
        assert FO.frustum_visible(m, b[:4], b[4:]) == bool(F.frustum_visible(m, b)[0])


def test_kill_table(cases):
    """Every mutant is told apart from the contract by some generated box, unless it is listed as equivalent (then no box
    tells it apart)."""
    table = {mu: {} for mu in F.MUTANTS}
    for kind, m, boxes in cases:
        want = F.frustum_visible(m, boxes)
        for mu in F.MUTANTS:
            k = int((F.frustum_visible(m, boxes, mu) != want).sum())
            if k:
                table[mu][kind] = table[mu].get(kind, 0) + k
    print("\nfrustum cull kill table (mutant: boxes that catch it, by matrix kind)")
    for mu in F.MUTANTS:
        caught = sum(table[mu].values())
        print(f"  {mu:10s} {'caught' if caught else 'equivalent':10s} {caught:5d}  {table[mu]}")
        if mu in F.EQUIVALENT_MUTANTS:
            assert caught == 0, mu
        else:
            assert caught > 0, mu


def test_selection_mutants_need_nonfinite_boxes_at_signed_zero_coefficients():
    """With every coordinate finite, a +-0 coefficient times either corner is a zero, so the choice made at a zero
    coefficient shows only through an infinite or NaN corner coordinate (0 * inf = NaN)."""
    m = np.eye(4, dtype=np.float32).reshape(16).copy()
    m[12] = np.float32(-0.0)  # R0 = (1, 0, 0, -0): the left plane gets d = 1 + -0, the x plane coefficient stays 1
    R = F.rows(m)
    R[2] = np.float32([0.0, -0.0, 1.0, 0.0])  # the near plane R2 has b = -0
    m = np.ascontiguousarray(R.T.reshape(16))
    # lo.y = 0.5 (finite), hi.y = +inf.  At the near plane's b = -0 the contract picks hi (s = NaN: kept), the sign-bit
    # mutant picks lo (s = the z term alone, 1 * hi.z = -1: culled).
    box = np.array([[-0.5, 0.5, -2, 1, 0.5, np.inf, -1, 1]], dtype=np.float32)
    assert F.frustum_visible(m, box)[0] and not F.frustum_visible(m, box, "sign_bit")[0]
    finite = np.array([[-0.5, 0.5, -2, 1, 0.5, 7, -1, 1]], dtype=np.float32)
    assert F.frustum_visible(m, finite, "sign_bit")[0] == F.frustum_visible(m, finite)[0]


def _random_camera(rng):
    eye = rng.uniform(-300, 300, 3)
    eye[1] = rng.uniform(1, 200)
    tgt = rng.uniform(-100, 100, 3)
    tgt[1] = rng.uniform(-5, 20)
    return F.camera(tuple(eye), tuple(tgt), far=float(rng.uniform(100, 3000)), aspect=float(rng.uniform(0.5, 2.5)),
                    fovy=float(rng.uniform(0.3, 2.0)), near=float(rng.uniform(0.05, 2.0)))


def _f32_down(x):
    y = x.astype(np.float32)
    return np.where(y.astype(np.float64) > x, np.nextafter(y, np.float32(-np.inf)), y).astype(np.float32)


def _f32_up(x):
    y = x.astype(np.float32)
    return np.where(y.astype(np.float64) < x, np.nextafter(y, np.float32(np.inf)), y).astype(np.float32)


def test_conservative_on_random_cameras(oracle):
    """Evaluated in float64 on the f32 matrix: a box holding a point strictly inside the clip volume (NDC |x|, |y| <=
    0.95, depth in [0.02, 0.98]) is never culled; a box whose 8 corners all lie beyond one plane by a relative margin of
    1e-5 is always culled."""
    rng = np.random.default_rng(0x5EED0F21)
    kept = culled = 0
    for _ in range(40):
        m = _random_camera(rng)
        M = F.rows(m).astype(np.float64)
        # inside: a world point for a random NDC point, then a box around it rounded outwards to f32
        k = 200
        ndc = np.stack([rng.uniform(-0.95, 0.95, k), rng.uniform(-0.95, 0.95, k), rng.uniform(0.02, 0.98, k), np.ones(k)], 1)
        h = np.linalg.solve(M, ndc.T).T
        pt = h[:, :3] / h[:, 3:4]
        ext = np.abs(rng.normal(size=(k, 3))) * rng.choice([0.0, 0.01, 1.0, 30.0], k)[:, None]
        boxes = np.concatenate([_f32_down(pt - ext), np.ones((k, 1), np.float32), _f32_up(pt + ext),
                                np.ones((k, 1), np.float32)], 1)
        clip = np.concatenate([pt, np.ones((k, 1))], 1) @ M.T
        w = clip[:, 3]
        assert (np.abs(clip[:, 0]) < w).all() and (np.abs(clip[:, 1]) < w).all() and (clip[:, 2] > 0).all() and (clip[:, 2] < w).all()
        vis = F.oracle_visible(m, boxes)
        assert vis.all(), np.nonzero(~vis)[0][:8]
        kept += k
        # outside: random boxes, those wholly beyond some plane by the margin (the exact planes: f32 adds are exact in f64)
        k = 2000
        c = M[3, :3] * 0 + rng.uniform(-400, 400, (k, 3))
        e = np.abs(rng.normal(size=(k, 3))) * rng.choice([0.0, 1.0, 20.0], k)[:, None]
        boxes = np.concatenate([c - e, np.ones((k, 1)), c + e, np.ones((k, 1))], 1).astype(np.float32)
        lo, hi = boxes[:, 0:3].astype(np.float64), boxes[:, 4:7].astype(np.float64)
        P = [M[3] + M[0], M[3] - M[0], M[3] + M[1], M[3] - M[1], M[2], M[3] - M[2]]
        beyond = np.zeros(k, dtype=bool)
        for a in P:
            pv = np.where(a[:3] >= 0, hi, lo)
            s = pv @ a[:3] + a[3]
            mag = np.abs(pv) @ np.abs(a[:3]) + abs(a[3])
            beyond |= s < -1e-5 * mag
        vis = F.oracle_visible(m, boxes)
        assert not vis[beyond].any(), np.nonzero(beyond & vis)[0][:8]
        culled += int(beyond.sum())
    assert kept >= 8000 and culled >= 20000


def test_default_box_is_never_culled(oracle, cases):
    """SceneNode's default box (-inf..+inf): every p-vertex term is +inf or NaN, under any matrix -- infinite and NaN
    entries too."""
    rng = np.random.default_rng(0x5EED0F22)
    mats = [m for _, m, _ in cases]
    for _ in range(50):
        m = rng.normal(size=16).astype(np.float32)
        m[rng.choice(16, 5, replace=False)] = rng.choice(np.array([0.0, -0.0, np.inf, -np.inf, np.nan], np.float32), 5)
        mats.append(m)
    box = F.default_box()[None, :]
    for m in mats:
        assert F.frustum_visible(m, box)[0]
        assert F.oracle_visible(m, box)[0]


@pytest.mark.parametrize("n,tr,tc", [(130, 32, 24), (97, 16, 20), (40, 1, 7), (64, 100, 100)])
def test_compaction_and_index_ranges_same_as_reference_cull(oracle, n, tr, tc):
    """Boxes whose visibility under the identity is the same for both tests (tests/_terrain_limits.py cull_boxes): the
    two culls give the same flags, ids, index buffer and counts."""
    rng = np.random.default_rng(n * 1000 + tr)
    tiles_r, tiles_c = oracle.tile_count(n, tr, tc)
    for p in (0.0, 0.3, 1.0):
        vis = rng.random(tiles_r * tiles_c) < p
        boxes = L.cull_boxes(vis)
        ref = oracle.terrain_cull(boxes, n, tr, tc, L.IDENTITY)
        got = FO.terrain_cull_frustum(boxes, n, tr, tc, L.IDENTITY)
        assert np.array_equal(ref["visible"], vis.astype(np.uint32))
        for key in ("visible", "ids", "idx", "counts"):
            assert np.array_equal(got[key], ref[key]), (p, key)
    # idx_capacity: the buffer holds exactly the visible indices
    got = FO.terrain_cull_frustum(boxes, n, tr, tc, L.IDENTITY, idx_capacity=int(got["counts"][1]))
    assert got["idx"].size == int(got["counts"][1])


def _on_screen_tiles(vtx, n, tr, tc, m, margin=1e-3):
    """Per tile: does some vertex of it lie strictly inside the clip volume (float64; a relative margin in x and y, and
    1e-6 in depth, which a perspective projection crowds towards w)?"""
    pos = vtx.view(np.float32).reshape(n, n, 8)[:, :, :3].astype(np.float64).reshape(-1, 3)
    M = F.rows(m).astype(np.float64)
    q = np.concatenate([pos, np.ones((len(pos), 1))], 1) @ M.T
    w = q[:, 3]
    inside = ((np.abs(q[:, 0]) < (1 - margin) * w) & (np.abs(q[:, 1]) < (1 - margin) * w) & (q[:, 2] > 1e-6 * w)
              & (q[:, 2] < (1 - 1e-6) * w)).reshape(n, n)
    tiles_r, tiles_c = (n - 1 + tr - 1) // tr, (n - 1 + tc - 1) // tc
    out = np.zeros(tiles_r * tiles_c, dtype=bool)
    for a in range(tiles_r):
        for b in range(tiles_c):
            out[a * tiles_c + b] = inside[a * tr:min(a * tr + tr, n - 1) + 1, b * tc:min(b * tc + tc, n - 1) + 1].any()
    return out


@pytest.mark.parametrize("cam", ["reference", "far"])
def test_frustum_cull_keeps_every_tile_on_screen(oracle, cam):
    """A 1025^2 hash-noise terrain in 32 x 32-quad tiles.  Under a perspective camera the reference's test (no divide)
    drops tiles that have a vertex on screen (231 of 416 under the reference camera); the frustum test drops none and keeps
    only a few tiles off screen."""
    n, t = 1025, 32
    h = oracle.synth_heightmap_u16(0x5EED0001, n)
    boxes = oracle.terrain_tile_bounds(h, n, t, t)
    vtx, _ = oracle.terrain_build(h, n, want_idx=False)
    m = camera_matrix() if cam == "reference" else F.camera((-200.0, 70.0, -200.0), (0.0, 0.0, 0.0), 1200.0, 16 / 9)
    on = _on_screen_tiles(vtx, n, t, t, m)
    ref = oracle.terrain_cull(boxes, n, t, t, m, want_idx=False)["visible"].astype(bool)
    fr = FO.terrain_cull_frustum(boxes, n, t, t, m, want_idx=False)["visible"].astype(bool)
    assert on.sum() > 20
    assert (on & ~ref).any(), "the reference's test keeps every on-screen tile for this camera"
    assert not (on & ~fr).any(), np.nonzero(on & ~fr)[0][:8]
    assert (fr & ~on).sum() <= max(4, fr.sum() // 20)  # the conservative test keeps only a few tiles off screen
