"""Float-edge cases for the terrain kernels, and CPU models to tell whether they can catch a wrong kernel.

Imported by tests/test_float_edges_cpu.py, tests/test_gpu_float_edges.py and scripts/fuzz_terrain.py / fuzz_session.py.

- should_render(m, boxes, mutant): the visibility test of mr_terrain_cull (SceneNode.zig:96-110) restated in numpy, every
  operation rounded in f32.  With mutant=None it is the contract of include/myrenderer_b200.h; the names in MUTANTS are
  plausible wrong implementations of it (evaluation order, precision, flush to zero, the +-inf skip rule, comparisons).
- cull_cases(seed): per matrix, the boxes that tell at least one mutant apart from the contract, plus boxes with +-inf or
  NaN in every slot.  Boxes drawn from real heightmaps almost never land within a few ulps of the thresholds.
- special_heightmap(rng, n): an f32 heightmap of NaNs, infinities, signed zeros, subnormals, +-FLT_MAX side by side and
  differences around the edges of the constant-divisor quotient's guarded range.
- float_mismatch(): compares output buffers word by word, any two NaNs equal (the header leaves a NaN's sign and payload
  unspecified); padding and index words stay exact.
"""
import math
from fractions import Fraction

import numpy as np

F32 = np.float32
FLT_MAX = float(np.finfo(np.float32).max)
MIN_NORMAL = F32(2.0 ** -126)

MUTANTS = ("fma", "reversed_j", "pairwise", "float64", "ftz_daz", "no_skip", "skip_any_inf", "compare_select_minmax",
           "three_components", "non_strict")
# fminf / fmaxf and a compare-select min / max differ only when an operand is NaN.  A point with a NaN component fails
# its clause whether it is transformed (NaN propagates to every component of M*p) or not, so no box can tell this
# mutant apart: it is kept as a check of that argument.
EQUIVALENT_MUTANTS = ("compare_select_minmax",)


def f32_from_bits(words):
    return np.asarray(words, dtype=np.uint32).view(np.float32)


# ---- the visibility test ----------------------------------------------------------------------------------------------
def round_f32(q: Fraction) -> np.float32:
    """The exact rational q rounded once to f32 (to nearest, ties to even, subnormals and overflow included)."""
    if q == 0:
        return F32(0.0)
    neg = q < 0
    a = -q if neg else q
    e = a.numerator.bit_length() - a.denominator.bit_length()  # 2^(e-1) < a < 2^(e+1)
    if a < Fraction(2) ** e:
        e -= 1
    e = max(e, -126)  # below the normal range the spacing stays 2^-149
    scaled = a * Fraction(2) ** (23 - e)
    m = scaled.numerator // scaled.denominator
    rem = scaled - m
    if rem > Fraction(1, 2) or (rem == Fraction(1, 2) and m & 1):
        m += 1
    v = m * 2.0 ** (e - 23)  # exact in f64
    if v >= 2.0 ** 128:
        v = math.inf
    return F32(-v if neg else v)


def _fma(a, b, c):
    """RN_f32(a * b + c) with a single rounding, a scalar, b and c f32 arrays."""
    a64 = np.float64(a)
    b64, c64 = b.astype(np.float64), c.astype(np.float64)
    with np.errstate(all="ignore"):
        p = a64 * b64  # exact: a product of two f32 fits in f64
        s = p + c64
        bb = s - p
        err = (p - (s - bb)) + (c64 - bb)  # s + err == p + c exactly (TwoSum)
        out = s.astype(np.float32)
        fin_p, fin_c = np.isfinite(p), np.isfinite(c64)
        out = np.where(fin_p, out, F32(a) * b + c)  # an infinite or NaN factor: fused and unfused agree
        out = np.where(fin_p & ~fin_c, c, out)      # a finite product plus +-inf or NaN is c
    for k in np.nonzero(fin_p & fin_c & (err != 0))[0]:  # s was rounded: round the exact value instead
        out[k] = round_f32(Fraction(float(a64)) * Fraction(float(b64[k])) + Fraction(float(c64[k])))
    return out


def _ftz(x):
    return np.where(np.abs(x) < MIN_NORMAL, np.copysign(F32(0.0), x), x).astype(np.float32)


def mul_vec(m, v, mutant=None):
    """mach Mat4x4.mulVec on the column image m (16 f32) for rows of v ([N, 4] f32): r[i] = sum_j m[4j+i] * v[j]."""
    m = np.asarray(m, dtype=np.float32).reshape(16)
    v = np.asarray(v, dtype=np.float32)
    out = np.empty(v.shape, dtype=np.float64 if mutant == "float64" else np.float32)
    with np.errstate(all="ignore"):
        if mutant == "ftz_daz":
            m, v = _ftz(m), _ftz(v)
        for i in range(4):
            if mutant == "float64":
                acc = np.zeros(len(v))
                for j in range(4):
                    acc = acc + np.float64(m[4 * j + i]) * v[:, j].astype(np.float64)
            elif mutant == "fma":
                acc = np.zeros(len(v), dtype=np.float32)
                for j in range(4):
                    acc = _fma(m[4 * j + i], v[:, j], acc)
            else:
                t = [m[4 * j + i] * v[:, j] for j in range(4)]
                if mutant == "ftz_daz":
                    t = [_ftz(x) for x in t]
                if mutant == "pairwise":
                    acc = (t[0] + t[1]) + (t[2] + t[3])
                else:
                    acc = np.zeros(len(v), dtype=np.float32)
                    for j in ((3, 2, 1, 0) if mutant == "reversed_j" else (0, 1, 2, 3)):
                        acc = acc + t[j]
                        if mutant == "ftz_daz":
                            acc = _ftz(acc)
            out[:, i] = acc
    return out


def _min4(p, mutant):
    if mutant == "compare_select_minmax":
        cs = lambda a, b: np.where(a < b, a, b)
        return cs(cs(p[:, 0], p[:, 1]), cs(p[:, 2], p[:, 3]))
    return np.fmin(np.fmin(p[:, 0], p[:, 1]), np.fmin(p[:, 2], p[:, 3]))  # fminf: a NaN operand is ignored


def _max4(p, mutant):
    if mutant == "compare_select_minmax":
        cs = lambda a, b: np.where(a > b, a, b)
        return cs(cs(p[:, 0], p[:, 1]), cs(p[:, 2], p[:, 3]))
    return np.fmax(np.fmax(p[:, 0], p[:, 1]), np.fmax(p[:, 2], p[:, 3]))


def should_render(m, boxes, mutant=None):
    """Visibility bit per box ([N, 8] f32: p0.xyzw, p1.xyzw) under the contract (mutant=None) or a named mutant."""
    boxes = np.asarray(boxes, dtype=np.float32).reshape(-1, 8)
    p0, p1 = boxes[:, :4], boxes[:, 4:]
    if mutant == "no_skip":
        skip0 = skip1 = np.zeros(len(boxes), dtype=bool)
    elif mutant == "skip_any_inf":
        skip0, skip1 = np.isinf(p0).any(1), np.isinf(p1).any(1)
    else:
        skip0, skip1 = _min4(p0, mutant) == -np.inf, _max4(p1, mutant) == np.inf
    q0 = np.where(skip0[:, None], p0, mul_vec(m, p0, mutant))
    q1 = np.where(skip1[:, None], p1, mul_vec(m, p1, mutant))
    k = 3 if mutant == "three_components" else 4
    with np.errstate(invalid="ignore"):
        if mutant == "non_strict":
            return (q1[:, :k] >= 0).all(1) | (q0[:, :k] <= 1).all(1)
        return (q1[:, :k] > 0).all(1) | (q0[:, :k] < 1).all(1)


def oracle_should_render(oracle, m, boxes):
    """The oracle's visibility bits for many boxes at once: one tile row of one-quad-wide tiles, one tile per box."""
    boxes = np.ascontiguousarray(boxes, dtype=np.float32).reshape(-1, 8)
    n = len(boxes) + 1
    return oracle.terrain_cull(boxes, n, n - 1, 1, m, want_idx=False)["visible"].astype(bool)


# ---- cull cases ---------------------------------------------------------------------------------------------------------
def step_ulps(x, k):
    """x moved by k ulps along the f32 number line (through zero, not past +-inf)."""
    b = np.asarray(x, dtype=np.float32).view(np.int32).astype(np.int64)
    lin = np.where(b < 0, -(b & 0x7FFFFFFF), b) + np.asarray(k, dtype=np.int64)  # monotone integer image of the floats
    lin = np.clip(lin, -0x7F800000, 0x7F800000)
    back = np.where(lin < 0, (-lin) | 0x80000000, lin).astype(np.uint32)
    return back.view(np.float32)


def cull_matrices(rng):
    """(kind, 16 f32 column image) pairs: cameras, normal() matrices, subnormal, huge and signed-zero entries."""
    from test_terrain_cull_cpu import camera_matrix

    out = [("camera", camera_matrix())]
    for _ in range(2):
        out.append(("camera", camera_matrix(tuple(float(x) for x in rng.uniform(-80, 80, 3)),
                                            tuple(float(x) for x in rng.uniform(-20, 20, 3)))))
    for _ in range(3):
        out.append(("normal", rng.normal(size=16).astype(np.float32)))
    out.append(("subnormal", (rng.normal(size=16) * 2.0 ** -132).astype(np.float32)))  # entries and products subnormal
    m = rng.normal(size=16).astype(np.float32)
    m[rng.choice(16, 6, replace=False)] = f32_from_bits(rng.integers(1, 0x800000, 6)) * F32(rng.choice([-1, 1]))
    out.append(("subnormal", m))
    out.append(("huge", (rng.normal(size=16) * 1e37).astype(np.float32)))  # products overflow
    m = rng.normal(size=16).astype(np.float32)
    m[rng.choice(16, 5, replace=False)] = F32(FLT_MAX) * rng.choice([-1, 1], 5).astype(np.float32)
    out.append(("huge", m))
    for _ in range(2):
        m = rng.normal(size=16).astype(np.float32)
        m[rng.choice(16, 7, replace=False)] = rng.choice(np.array([0.0, -0.0], dtype=np.float32), 7)
        out.append(("zeros", m))
    return out


def _near_threshold(rng, m, count):
    """Boxes with one component of M*p1 near 0 or one of M*p0 near 1: one coordinate solved for it, then moved by a few
    ulps; some other coordinate is sometimes -0."""
    m = np.asarray(m, dtype=np.float64).reshape(4, 4)  # m[j, i] = xform[4j + i]
    scale = rng.choice([1.0, 10.0, 100.0, 1e-3], count)[:, None]
    p = rng.normal(size=(count, 4)) * scale
    p[:, 3] = np.where(rng.random(count) < 0.7, 1.0, p[:, 3])
    which = rng.integers(0, 2, count)  # 1: p1 against 0, 0: p0 against 1
    i, k = rng.integers(0, 4, count), rng.integers(0, 4, count)
    z = rng.integers(0, 4, count)
    negz = (rng.random(count) < 0.3) & (z != k)
    p[negz, z[negz]] = -0.0
    p = p.astype(np.float32).astype(np.float64)
    target = np.where(which == 1, 0.0, 1.0)
    with np.errstate(all="ignore"):
        rest = (p * m[:, i].T).sum(1) - p[np.arange(count), k] * m[k, i]  # sum over j != k of m[j, i] * p[j]
        sol = (target - rest) / m[k, i]
    ok = np.isfinite(sol) & (np.abs(sol) < 1e38)
    p, which, k, sol = p[ok].astype(np.float32), which[ok], k[ok], sol[ok]
    p[np.arange(len(p)), k] = step_ulps(sol.astype(np.float32), rng.integers(-3, 4, len(p)))
    other = (rng.normal(size=(len(p), 4)) * rng.choice([1.0, 10.0, 100.0], len(p))[:, None]).astype(np.float32)
    other[:, 3] = 1.0
    return np.where((which == 1)[:, None], np.concatenate([other, p], 1), np.concatenate([p, other], 1)).astype(np.float32)


def _extreme_boxes(rng, count):
    """Components whose products are subnormal or overflow, mixed in sign, so that a sum can be inf - inf."""
    vals = np.array([FLT_MAX, 3e38, 1e38, 1e20, 1e-20, 1e-38, 1e-40, 1e-45, 2.0 ** -140, 1.0, 0.5], dtype=np.float32)
    b = rng.choice(vals, size=(count, 8)) * rng.choice(np.array([-1, 1], dtype=np.float32), size=(count, 8))
    mix = rng.random((count, 8)) < 0.3
    b[mix] = rng.normal(size=mix.sum()).astype(np.float32)
    return b.astype(np.float32)


def _nonfinite_boxes(rng):
    """+inf, -inf and NaN in every slot (w included), and -inf / +inf with NaN in one point, in both orders."""
    base = lambda: np.concatenate([rng.normal(size=3) * 3, [1.0], rng.normal(size=3) * 3, [1.0]]).astype(np.float32)
    out = []
    for s in range(8):
        for v in (np.inf, -np.inf, np.nan):
            for _ in range(4):  # +inf in p0 (-inf in p1) changes the bit only when M sends it below 1 (above 0)
                b = base()
                b[s] = v
                out.append(b)
    for pt in (0, 4):
        for a in range(4):
            for c in range(4):
                if a != c:
                    for inf in (-np.inf, np.inf):
                        b = base()
                        b[pt + a], b[pt + c] = inf, np.nan
                        out.append(b)
    out.append(np.full(8, np.nan, dtype=np.float32))
    out.append(np.array([-np.inf] * 3 + [1] + [np.inf] * 3 + [1], dtype=np.float32))  # SceneNode's default box
    return np.array(out, dtype=np.float32)


def cull_cases(seed=0x5EED0F10, near=600, extreme=300):
    """[(kind, m, boxes)]: per matrix, the boxes that tell some mutant apart from the contract, plus the non-finite ones."""
    rng = np.random.default_rng(seed)
    out = []
    for kind, m in cull_matrices(rng):
        cand = np.concatenate([_near_threshold(rng, m, near), _extreme_boxes(rng, extreme)])
        want = should_render(m, cand)
        keep = np.zeros(len(cand), dtype=bool)
        for mu in MUTANTS:
            keep |= should_render(m, cand, mu) != want
        out.append((kind, m, np.concatenate([cand[keep], _nonfinite_boxes(rng)])))
    return out


# ---- heightmaps ---------------------------------------------------------------------------------------------------------
NAN_WORDS = (0x7FC00000, 0x7FA00001, 0xFFC00000, 0x7FC12345, 0xFF800001, 0x7FBFFFFF)  # quiet, signalling, negative, payloads
SPECIAL_WORDS = NAN_WORDS + (0x7F800000, 0xFF800000, 0x00000000, 0x80000000, 0x00000001, 0x80000001, 0x007FFFFF, 0x807FFFFF,
                             0x7F7FFFFF, 0xFF7FFFFF)


def special_heightmap(rng, n, tiles=((8, 24),), height_scale=5.0):
    """[n, n] f32 heightmap of special values on a uniform(-3, 3) ground.

    Scattered: NaN (quiet, signalling, negative, with payloads), +-inf, +-0, the smallest and largest subnormals, +-FLT_MAX.
    +FLT_MAX and -FLT_MAX side by side and two apart along rows and columns, at the borders too (their difference
    overflows).  Height differences d with height_scale * d within a few ulps of 2^-63 and 2^64, the ends of the range in
    which the kernels divide by grid_step with the reciprocal-and-correct scheme.  For every (tile_rows, tile_cols) in
    `tiles` that fits: one tile all NaN, one tile whose first and last texels are NaN, one tile of positive heights whose
    minimum is the smallest subnormal."""
    w = rng.uniform(-3.0, 3.0, size=(n, n)).astype(np.float32).view(np.uint32)
    k = max(1, n * n // 40)
    w.reshape(-1)[rng.choice(n * n, k, replace=n * n < k)] = rng.choice(np.array(SPECIAL_WORDS, dtype=np.uint32), k)
    if n >= 3:
        big, nbig = 0x7F7FFFFF, 0xFF7FFFFF
        for r in {0, n // 2, n - 1}:
            c = int(rng.integers(0, n - 2))
            w[r, c], w[r, c + 1], w[r, c + 2] = big, nbig, nbig if r else big
            c = int(rng.integers(0, n - 2))
            w[c, r], w[c + 1, r], w[c + 2, r] = nbig, big, big
        # hs * d straddling 2^-63 and 2^64: neighbours two apart differ by d (the centre keeps its value)
        ys = []
        for y0 in (2.0 ** -63, 2.0 ** 64):
            for s in (1.0, -1.0):
                y = step_ulps(np.full(7, y0 * s, dtype=np.float32), np.arange(-3, 4))
                ys.extend(np.float32(yv) / np.float32(height_scale) for yv in y)
        for t, d in enumerate(ys):
            r, c = int(rng.integers(1, n - 1)), int(rng.integers(1, n - 1))
            if t % 2:
                w[r, c - 1], w[r, c + 1] = 0, np.float32(d).view(np.uint32)
            else:
                w[r - 1, c], w[r + 1, c] = 0, np.float32(d).view(np.uint32)
    for tr, tc in tiles:
        tiles_r, tiles_c = (n - 1 + tr - 1) // tr, (n - 1 + tc - 1) // tc
        if tiles_r < 2 or tiles_c < 2:
            continue
        spots = [(a, b) for a in range(tiles_r) for b in range(tiles_c)]
        picks = rng.choice(len(spots), min(3, len(spots)), replace=False)
        for role, p in enumerate(picks):
            a, b = spots[p]
            r0, c0 = a * tr, b * tc
            r1, c1 = min(r0 + tr, n - 1), min(c0 + tc, n - 1)
            if role == 0:
                w[r0:r1 + 1, c0:c1 + 1] = rng.choice(np.array(NAN_WORDS, dtype=np.uint32), (r1 - r0 + 1, c1 - c0 + 1))
            elif role == 1:
                w[r0, c0], w[r1, c1] = NAN_WORDS[1], NAN_WORDS[2]
            else:
                w[r0:r1 + 1, c0:c1 + 1] = rng.uniform(1.0, 3.0, (r1 - r0 + 1, c1 - c0 + 1)).astype(np.float32).view(np.uint32)
                w[int(rng.integers(r0, r1 + 1)), int(rng.integers(c0, c1 + 1))] = 0x00000001
    return w.view(np.float32)


# ---- comparing outputs --------------------------------------------------------------------------------------------------
def is_nan_word(w):
    return (np.asarray(w, dtype=np.uint32) & 0x7FFFFFFF) > 0x7F800000


def vertex_float_mask(nbytes, layout):
    """Per 32-bit word of a vertex buffer: True where the kernels write a float (position / normal x, y, z)."""
    stride, attrs = layout
    mask = np.zeros((nbytes // stride, stride // 4), dtype=bool)
    for off, _ in attrs:
        mask[:, off // 4: off // 4 + 3] = True
    return mask.reshape(-1)


def float_mismatch(got, want, float_mask=True):
    """None if the buffers agree, else a description.  Words under float_mask (True: every word) agree when they are
    bit-equal or both NaN; all other words, padding included, must be bit-equal."""
    g = np.ascontiguousarray(got).reshape(-1).view(np.uint32)
    w = np.ascontiguousarray(want).reshape(-1).view(np.uint32)
    if g.shape != w.shape:
        return "sizes differ: %d vs %d words" % (g.size, w.size)
    ok = (g == w) | (np.asarray(float_mask) & is_nan_word(g) & is_nan_word(w))
    if ok.all():
        return None
    i = int(np.argmin(ok))
    return "%d of %d words differ, first at word %d: got 0x%08x, want 0x%08x" % ((~ok).sum(), ok.size, i, g[i], w[i])


def nan_words(buf, float_mask=True):
    """The distinct NaN bit patterns in the float words of a buffer."""
    b = np.ascontiguousarray(buf).reshape(-1).view(np.uint32)
    return sorted({int(x) for x in np.unique(b[np.asarray(float_mask) & is_nan_word(b)])})
