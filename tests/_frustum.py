"""The six-plane frustum test of mr_terrain_cull_frustum: a numpy model, wrong variants of it, and cases that tell them apart.

Imported by tests/test_frustum_cull_cpu.py and tests/test_gpu_frustum_cull.py.

- frustum_visible(m, boxes, mutant): the header's test restated in numpy, every operation rounded in f32.  With
  mutant=None it is the contract of include/myrenderer_b200.h; the names in MUTANTS are plausible wrong implementations
  (contraction, evaluation order, precision, flush to zero, the p-vertex selection, the comparison, the depth range, a
  missing plane, and the clip-space-corners formulation).
- frustum_cases(seed): per matrix, the boxes that tell at least one mutant apart from the contract, plus boxes with +-inf
  or NaN in every slot.
- camera(...): view-projection images of the reference's camera (math.zig perspective * lookAt).
"""
import numpy as np

import _float_edges as E
import _frustum_oracle as FO
from test_terrain_cull_cpu import look_at, mat_image, perspective

F32 = np.float32

MUTANTS = ("fma", "reversed", "float64", "ftz_daz", "sign_bit", "gt_zero", "le_zero", "nan_culls", "gl_near", "no_near",
           "no_far", "corners")
# Every mutant is told apart by some generated box; none is equivalent to the contract.
EQUIVALENT_MUTANTS = ()

# ---- the test -------------------------------------------------------------------------------------------------------------
def rows(m):
    """R_i = (m[i], m[4+i], m[8+i], m[12+i]) of the column image m: [4, 4] f32, R[i, j] = m[4j + i]."""
    return np.asarray(m, dtype=np.float32).reshape(16).reshape(4, 4).T.copy()


def planes(m, mutant=None):
    """The six planes as [k, 4] (a, b, c, d), each component one rounded add or subtract (in f64 for 'float64')."""
    R = rows(m).astype(np.float64 if mutant == "float64" else np.float32)
    if mutant == "ftz_daz":
        R = E._ftz(R)
    with np.errstate(all="ignore"):
        out = [R[3] + R[0], R[3] - R[0], R[3] + R[1], R[3] - R[1], R[3] + R[2] if mutant == "gl_near" else R[2], R[3] - R[2]]
    if mutant == "no_near":
        del out[4]
    elif mutant == "no_far":
        del out[5]
    out = np.array(out)
    return E._ftz(out) if mutant == "ftz_daz" else out


def _select(coef, lo, hi, mutant):
    if mutant == "sign_bit":
        pick_hi = not np.signbit(coef)  # -0 picks lo, a NaN with its sign bit clear picks hi
    elif mutant == "gt_zero":
        pick_hi = coef > 0  # +0 picks lo
    else:
        pick_hi = coef >= 0  # the contract: -0 picks hi, NaN picks lo
    return hi if pick_hi else lo


def plane_values(m, boxes, mutant=None):
    """[N, k] s per box and plane under the contract or a plane-test mutant."""
    boxes = np.asarray(boxes, dtype=np.float32).reshape(-1, 8)
    lo, hi = boxes[:, 0:3], boxes[:, 4:7]
    wide = mutant == "float64"
    if wide:
        lo, hi = lo.astype(np.float64), hi.astype(np.float64)
    if mutant == "ftz_daz":
        lo, hi = E._ftz(lo), E._ftz(hi)
    fl = E._ftz if mutant == "ftz_daz" else (lambda x: x)
    P = planes(m, mutant)
    out = np.empty((len(boxes), len(P)), dtype=np.float64 if wide else np.float32)
    with np.errstate(all="ignore"):
        for k, (a, b, c, d) in enumerate(P):
            px, py, pz = (_select(co, lo[:, i], hi[:, i], mutant) for i, co in enumerate((a, b, c)))
            if mutant == "fma":  # contracted: fma(c, pz, fma(b, py, a * px)) + d
                s = E._fma(c, pz, E._fma(b, py, a * px)) + d
            elif mutant == "reversed":
                s = ((d + c * pz) + b * py) + a * px
            else:
                s = fl(fl(fl(fl(a * px) + fl(b * py)) + fl(c * pz)) + d)
            out[:, k] = s
    return out


def _corners_visible(m, boxes):
    """Transform the 8 corners (w = 1) with mach's mulVec, cull if all 8 fail one clip inequality."""
    boxes = np.asarray(boxes, dtype=np.float32).reshape(-1, 8)
    fail = np.ones((len(boxes), 6), dtype=bool)
    for k in range(8):
        p = np.stack([boxes[:, 4 * ((k >> i) & 1) + i] for i in range(3)] + [np.ones(len(boxes), np.float32)], 1)
        q = E.mul_vec(m, p)
        x, y, z, w = q.T
        with np.errstate(invalid="ignore"):
            fail &= np.stack([x < -w, x > w, y < -w, y > w, z < 0, z > w], 1)
    return ~fail.any(1)


def frustum_visible(m, boxes, mutant=None):
    """Visibility bit per box ([N, 8] f32: p0.xyzw, p1.xyzw) under the contract (mutant=None) or a named mutant."""
    if mutant == "corners":
        return _corners_visible(m, boxes)
    s = plane_values(m, boxes, mutant)
    with np.errstate(invalid="ignore"):
        if mutant == "le_zero":
            return ~(s <= 0).any(1)
        if mutant == "nan_culls":
            return ~(~(s >= 0)).any(1)
        return ~(s < 0).any(1)


def oracle_visible(m, boxes):
    """The C oracle's bits for many boxes at once: one tile row of one-quad-wide tiles, one tile per box."""
    boxes = np.ascontiguousarray(boxes, dtype=np.float32).reshape(-1, 8)
    n = len(boxes) + 1
    return FO.terrain_cull_frustum(boxes, n, n - 1, 1, m, want_idx=False)["visible"].astype(bool)


# ---- cameras ----------------------------------------------------------------------------------------------------------------
def camera(cam=(30.0, 25.0, -40.0), target=(0.0, 0.0, 0.0), far=200.0, aspect=1.0, fovy=1.2, near=0.1):
    """perspective(fovy, aspect, near, far) * lookAt(cam, target, +y) as a column image (math.zig:9-31)."""
    p = np.array(perspective(fovy, aspect, near, far), dtype=np.float32)
    return mat_image(p @ np.array(look_at(cam, target, (0, 1, 0)), dtype=np.float32))


# The cameras of scripts/bench_cull.py and the GPU tests: (name, eye, target, far), aspect 16/9.
CAMERAS = (
    ("near", (30.0, 25.0, -40.0), (0.0, 0.0, 0.0), 200.0),
    ("far", (-350.0, 120.0, -350.0), (0.0, 0.0, 0.0), 2000.0),
    ("down", (5.0, 400.0, 3.0), (0.0, 0.0, 0.0), 1000.0),
    ("grazing", (-400.0, 3.0, 10.0), (400.0, 1.0, -10.0), 1500.0),
)


def camera_by_name(name):
    for nm, eye, tgt, far in CAMERAS:
        if nm == name:
            return camera(eye, tgt, far, aspect=16.0 / 9.0)
    raise KeyError(name)


# ---- cases ------------------------------------------------------------------------------------------------------------------
def frustum_matrices(rng):
    """(kind, 16 f32 column image): cameras, normal() matrices, subnormal, huge and signed-zero entries, an infinite far
    plane (R2 == R3, so the far plane is all zeros), and small integer matrices on which s is often exactly 0."""
    out = [("camera", camera()), ("camera", camera_by_name("far")), ("camera", camera_by_name("grazing"))]
    for _ in range(2):
        out.append(("camera", camera(tuple(float(x) for x in rng.uniform(-80, 80, 3)),
                                     tuple(float(x) for x in rng.uniform(-20, 20, 3)), far=float(rng.uniform(50, 500)))))
    for _ in range(3):
        out.append(("normal", rng.normal(size=16).astype(np.float32)))
    out.append(("subnormal", (rng.normal(size=16) * 2.0 ** -132).astype(np.float32)))
    m = rng.normal(size=16).astype(np.float32)
    m[rng.choice(16, 6, replace=False)] = E.f32_from_bits(rng.integers(1, 0x800000, 6)) * F32(rng.choice([-1, 1]))
    out.append(("subnormal", m))
    out.append(("huge", (rng.normal(size=16) * 1e37).astype(np.float32)))
    m = rng.normal(size=16).astype(np.float32)
    m[rng.choice(16, 5, replace=False)] = F32(E.FLT_MAX) * rng.choice([-1, 1], 5).astype(np.float32)
    out.append(("huge", m))
    for _ in range(3):
        m = rng.choice(np.array([0.0, -0.0, 1.0, -1.0, 0.5, -2.0], dtype=np.float32), 16)
        m[rng.choice(16, 4, replace=False)] = rng.choice(np.array([0.0, -0.0], dtype=np.float32), 4)
        out.append(("zeros", m))
    R = rows(camera())
    R[2] = R[3]  # depth = w everywhere: the far plane R3 - R2 is (0, 0, 0, 0)
    out.append(("infinite_far", mat_image(R)))
    out.append(("integer", np.eye(4, dtype=np.float32).reshape(16)))
    out.append(("integer", rng.integers(-3, 4, 16).astype(np.float32)))
    return out


def _near_plane_boxes(rng, m, count):
    """Boxes whose p-vertex s for one plane lies within a few ulps of 0 (or at 0): one p-vertex coordinate solved for
    s = 0 in f64, then moved by -3..3 ulps; the other corner lies on the far side of the p-vertex (a proper box) or, for
    a quarter of them, on the near side (inverted), or at the p-vertex (flat)."""
    P = planes(m).astype(np.float64)
    out = []
    k = rng.integers(0, len(P), count)
    axis = rng.integers(0, 3, count)
    scale = rng.choice([1.0, 10.0, 100.0, 1e-3], count)
    for t in range(count):
        a = P[k[t]]
        if not np.isfinite(a).all() or a[axis[t]] == 0:
            continue
        p = rng.normal(size=3) * scale[t]
        rest = sum(a[i] * p[i] for i in range(3) if i != axis[t]) + a[3]
        p[axis[t]] = -rest / a[axis[t]]
        if not np.isfinite(p).all() or np.abs(p).max() > 1e38:
            continue
        p = p.astype(np.float32)
        p[axis[t]] = E.step_ulps(p[axis[t]], int(rng.integers(-3, 4)))
        ext = np.abs(rng.normal(size=3) * scale[t]).astype(np.float32)
        mode = rng.random()
        if mode < 0.15:
            ext[:] = 0  # flat
        elif mode < 0.4:
            ext = -ext  # inverted
        hi, lo = p.copy(), p.copy()
        for i in range(3):  # p is the p-vertex: hi where the coefficient is >= 0, else lo
            if a[i] >= 0:
                lo[i] = p[i] - ext[i]
            else:
                hi[i] = p[i] + ext[i]
        out.append(np.concatenate([lo, [1.0], hi, [1.0]]).astype(np.float32))
    return np.array(out, dtype=np.float32).reshape(-1, 8)


def _random_boxes(rng, count):
    """Proper, flat and inverted boxes around random points, scales from 1e-3 to 1e3."""
    c = rng.normal(size=(count, 3)) * rng.choice([1e-3, 1.0, 10.0, 100.0, 1000.0], count)[:, None]
    e = np.abs(rng.normal(size=(count, 3))) * rng.choice([0.0, 0.1, 1.0, 10.0], count)[:, None]
    e *= np.where(rng.random((count, 1)) < 0.2, -1.0, 1.0)
    ones = np.ones((count, 1))
    return np.concatenate([c - e, ones, c + e, ones], 1).astype(np.float32)


def _nonfinite_boxes(rng):
    """+inf, -inf and NaN in every slot (w included: it is not read), alone and two at a time, on random boxes and on
    boxes at the origin (where the planes' +-0 coefficients meet them)."""
    base = lambda: (np.concatenate([rng.normal(size=3) * 3, [1.0], rng.normal(size=3) * 3, [1.0]])
                    if rng.random() < 0.5 else np.array([0, 0, 0, 1, 0, 0, 0, 1], dtype=np.float64)).astype(np.float32)
    specials = (np.inf, -np.inf, np.nan)
    out = []
    for s in range(8):
        for v in specials:
            for _ in range(4):
                b = base()
                b[s] = v
                out.append(b)
    for s1 in range(8):
        for s2 in range(s1 + 1, 8):
            b = base()
            b[s1], b[s2] = rng.choice(specials), rng.choice(specials)
            out.append(b)
    out.append(np.full(8, np.nan, dtype=np.float32))
    out.append(np.array([-np.inf] * 3 + [1] + [np.inf] * 3 + [1], dtype=np.float32))  # SceneNode's default box
    return np.array(out, dtype=np.float32)


def frustum_cases(seed=0x5EED0F20, near=600, extreme=300, random=300):
    """[(kind, m, boxes)]: per matrix, the generated boxes that tell some mutant apart from the contract, plus the
    non-finite ones."""
    rng = np.random.default_rng(seed)
    out = []
    for kind, m in frustum_matrices(rng):
        # E._extreme_boxes: coordinates whose products with the planes are subnormal or overflow, mixed in sign
        cand = np.concatenate([_near_plane_boxes(rng, m, near), E._extreme_boxes(rng, extreme), _random_boxes(rng, random)])
        want = frustum_visible(m, cand)
        keep = np.zeros(len(cand), dtype=bool)
        for mu in MUTANTS:
            keep |= frustum_visible(m, cand, mu) != want
        out.append((kind, m, np.concatenate([cand[keep], _nonfinite_boxes(rng)])))
    return out


def default_box():
    return np.array([-np.inf, -np.inf, -np.inf, 1, np.inf, np.inf, np.inf, 1], dtype=np.float32)
