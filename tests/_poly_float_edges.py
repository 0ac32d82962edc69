"""Float-edge cases for the polygon triangulation, and the proof that they can catch a wrong kernel.

Imported by tests/test_poly_float_edges_cpu.py and tests/test_gpu_poly_float_edges.py.

The reference's float rules are three predicates of Triangulation.zig (is_left_of :117-126, point_is_above :128-136,
push_triangle_if_acute :398-425), render_point's bbox rule (Polygon.zig:73-76) and the non-finite rejection; the kernels
restate each of them once per execution path.  The oracle (oracle/o_triangulation.c, o_polygon.c) carries test-only
mutants of every rule (oracle.MUTANTS): a plausible wrong restatement each.  kill_cases() draws polygons from families that
put these rules at their edges -- signed zeros, subnormal and overflowing side tests, near-collinear triples, corners
whose atan2 difference lies within an ulp of pi -- in every size class of the kernels, and keeps the polygons on which some
mutant changes the output (status, triangle count, vertex bytes or bbox bits).  nonfinite_cases() puts NaNs and
infinities in x only or y only, at the first, a middle and the last point, in every size class.
"""
import numpy as np

F32 = np.float32
FLT_MAX = float(np.finfo(np.float32).max)

# (name, smallest n, largest n) of the kernels' size classes: one warp per polygon up to 64 points, independent warps up
# to 288, warp teams up to 1024, one polygon per SM up to 3072, the general path above.
CLASSES = (("le64", 3, 64), ("w128", 65, 128), ("w168", 129, 168), ("w216", 169, 216), ("w288", 217, 288),
           ("t368", 289, 368), ("t504", 369, 504), ("t608", 505, 608), ("t768", 609, 768), ("t1024", 769, 1024),
           ("xl3072", 1025, 3072), ("gt3072", 3073, 4096))
# A few sizes per class: both ends, and an interior size up to 1024 points.  The first class also gets the small sizes that
# tests/test_poly_float_edges_cpu.py can run through oracle/pyref.py.
CLASS_SIZES = {"le64": (4, 5, 6, 7, 8, 10, 12, 16, 33, 64)}
for _name, _lo, _hi in CLASSES[1:]:
    CLASS_SIZES[_name] = (_lo, (_lo + _hi) // 2, _hi) if _hi <= 1024 else (_lo, _hi)

# Every mutant runs its rule in every size class, and the kill set must catch each of them in every class: the float
# rules are restated once per execution path, so a mistake confined to one path (say the XL class) must fail a test.
# The non-finite mutants are caught by nonfinite_cases(), the others by kill_cases().

MAX_KEEP = 3  # killing cases kept per (mutant, class)
PAD_SOURCES = 12  # small killing polygons padded per (mutant, class) that pass 1 did not reach
PAD_KEEP = 1
PYREF_MAX_N = 16


def size_class(n):
    for name, lo, hi in CLASSES:
        if lo <= n <= hi:
            return name
    raise ValueError(n)


def _f(a):
    return np.ascontiguousarray(a, dtype=np.float32)


def _sound(oracle, n, fam, seed):
    """A polygon of the reference-sound families (ellipse, zipper) or a star, moved to the origin: coordinates of both
    signs, magnitude about 100."""
    xy = oracle.synth_polygons(seed, np.array([0, n], dtype=np.uint64), family=fam).astype(np.float64)
    return xy - 100.0


def _mirror(xy, k):
    """One of the eight exact symmetries of the square (k = 0..7): rotations by 90 degrees and reflections."""
    xy = np.array(xy, dtype=np.float64)
    if k & 4:
        xy = xy[:, ::-1].copy()
    if k & 1:
        xy[:, 0] = -xy[:, 0]
    if k & 2:
        xy[:, 1] = -xy[:, 1]
    return xy


# ---- families ---------------------------------------------------------------------------------------------------------
def fam_grid_pm0(oracle, rng, n):
    """A sound polygon on a quarter or integer grid, centred so that points fall on both axes: rounding a small negative
    coordinate gives -0, a small positive one +0.  The grid spacing keeps most neighbours apart; coincident points that
    remain send the polygon to the general path."""
    q = float(rng.choice([0.25, 1.0]))
    xy = _mirror(_sound(oracle, n, int(rng.integers(0, 3)), int(rng.integers(1 << 30))), int(rng.integers(8)))
    s = max(1.0, n / 100.0) * float(rng.uniform(0.5, 2.0))
    xy = np.round(xy * s / q) * q
    return _f(xy)


def fam_ylevels(oracle, rng, n):
    """y near zero snapped to -0 or +0 (sign drawn per point), x left distinct: ties in y between -0 and +0 that the x
    coordinates decide.  Also x near zero snapped to a signed zero."""
    xy = _mirror(_sound(oracle, n, int(rng.integers(0, 2)), int(rng.integers(1 << 30))), int(rng.integers(8)))
    band = float(rng.uniform(5, 30))
    sub = rng.random() < 0.4  # snap to distinct subnormals of either sign instead: the order of those must not flush
    for c in (1, 0) if rng.random() < 0.5 else (1,):
        m = np.abs(xy[:, c]) < band
        sign = np.where(rng.random(m.sum()) < 0.5, -1.0, 1.0)
        xy[m, c] = sign * (rng.integers(1, 1 << 20, m.sum()) * 2.0 ** -149 if sub else 0.0)
        if c == 1 and not sub and m.sum() >= 2:  # at least one -0 / +0 pair
            j = np.nonzero(m)[0]
            xy[j[0], 1], xy[j[-1], 1] = -0.0, 0.0
    return _f(xy)


def fam_edge0(oracle, rng, n):
    """A sound polygon moved so that its smallest (or, mirrored, largest) x and y are exactly zero, with the zero's sign
    drawn per point: render_point's bbox accumulators start at +0 and a tie must keep them."""
    xy = _sound(oracle, n, int(rng.integers(0, 3)), int(rng.integers(1 << 30)))
    xy = _f(xy - xy.min(0))
    for c in (0, 1):
        z = xy[:, c] == 0
        xy[z, c] = np.where(rng.random(z.sum()) < 0.7, -0.0, 0.0)
    return _f(_mirror(xy, int(rng.integers(8))))


def fam_twins(oracle, rng, n):
    """A grid polygon with a -0 / +0 twin: a point with a zero coordinate repeated with the zero's sign flipped.  The
    two are equal in the (y, x) order, i.e. coincident."""
    xy = fam_grid_pm0(oracle, rng, n).astype(np.float32)
    zeros = np.nonzero((xy == 0).any(1))[0]
    k = int(zeros[rng.integers(len(zeros))]) if len(zeros) else int(rng.integers(n))
    if not len(zeros):
        xy[k, 1] = -0.0
    j = (k + 1 + int(rng.integers(0, max(1, n - 1)))) % n if rng.random() < 0.5 else (k + 1) % n
    if j != k:
        xy[j] = np.where(xy[k] == 0, np.copysign(np.float32(0), -np.copysign(np.float32(1), xy[k])), xy[k])
    return _f(xy)


SCALES = (2.0 ** -140, 2.0 ** -75, 2.0 ** 121)  # subnormal coordinates; subnormal products; overflowing differences


def fam_scaled(oracle, rng, n):
    """A sound family or a star scaled so that the coordinates and differences are subnormal (2^-140), the products of
    differences are subnormal (2^-75), or the differences overflow to inf and inf*0 gives NaN in the side test (2^121 at
    magnitude 100 after centring: 2^121 * 200 > FLT_MAX)."""
    sc = SCALES[int(rng.integers(len(SCALES)))]
    xy = _mirror(_sound(oracle, n, int(rng.integers(0, 3)), int(rng.integers(1 << 30))), int(rng.integers(8)))
    if sc > 1:
        xy = np.clip(xy * sc, -FLT_MAX, FLT_MAX)
    else:
        xy = xy * sc
    return _f(xy)


def fam_collinear(oracle, rng, n):
    """Every few vertices of a sound polygon of magnitude 1e3 moved onto the line through its two neighbours, then a few
    ulps off it in x or y.  The neighbours' directions cover all eight octants."""
    xy = _mirror(_sound(oracle, n, int(rng.integers(0, 2)), int(rng.integers(1 << 30))), int(rng.integers(8)))
    xy = _f(xy * 10.0 + rng.uniform(-1e3, 1e3, 2))
    step = int(rng.integers(2, 4))
    for k in range(1, n - 1, step):
        a, b = xy[k - 1].astype(np.float64), xy[k + 1].astype(np.float64)
        t = rng.uniform(0.2, 0.8)
        p = _f(a + t * (b - a))
        c = int(rng.integers(2))
        u = int(rng.integers(-3, 4))
        v = p[c]
        for _ in range(abs(u)):
            v = np.nextafter(v, np.float32(np.inf if u > 0 else -np.inf), dtype=np.float32)
        p[c] = v
        xy[k] = p
    return xy


ACUTE_SLOPES = (0.0, 1e-45, 5e-41, 1e-38, 1e-12, 1e-9, 1.4e-8, 1.6e-8, 3e-8, 3.15e-8, 3.2e-8, 3.25e-8, 3.3e-8, 5e-8, 1e-7,
                1.2e-7, 2e-7, 2.4e-7, 3e-7, 1e-6, 1.1e-6)


def fam_acute(oracle, rng, n):
    """The corners of test_acute_test_near_the_negative_x_axis as a polygon of any size: a chain whose consecutive
    points rise by slopes from 0 and subnormal through the 1e-8 .. 1e-6 range where atan2 rounds to pi or to the float
    below it, closed by an apex below; rotated into any quadrant and mirrored.  The mountain loop then compares
    differences of atan2 values within an ulp of pi."""
    w = float(rng.choice([1.0, 1e-3, 1e8, 3e-20])) * (1.0 + rng.random())
    m = n - 1
    x = np.arange(m, dtype=np.float64) * w
    sl = np.array(ACUTE_SLOPES)[rng.integers(len(ACUTE_SLOPES), size=m)] * (1.0 + 0.05 * rng.random(m))
    y = np.cumsum(np.concatenate([[0.0], w * sl[1:] * np.where(rng.random(m - 1) < 0.7, 1.0, -1.0)]))
    if rng.random() < 0.5:
        y = y - y[int(rng.integers(m))]
    if m > 8 and rng.random() < 0.7:  # a short flat chain on top of a convex arc of the remaining points
        m = int(rng.integers(3, 7))
        x, y = x[:m], y[:m]
        t = np.linspace(0.0, np.pi, n - m + 2)[1:-1]
        r = x[-1] / 2
        below = np.stack([r + r * np.cos(t), -r * rng.uniform(0.2, 2.0) * np.sin(t)], 1)
    else:
        below = np.array([[x[-1] * rng.uniform(0.3, 0.7), -w * rng.uniform(0.5, 3.0) * max(1.0, m / 8)]])
    chain = np.stack([x, y], 1)
    xy = np.concatenate([chain, below])
    if rng.random() < 0.5:
        xy = xy[::-1].copy()
    return _f(_mirror(xy, int(rng.integers(8))))


def fam_acute_small(oracle, rng, n):
    """The thin triangles and quadrilaterals of test_acute_test_near_the_negative_x_axis, rotated into every quadrant."""
    w = float(rng.choice([1.0, 1e-3, 1e10, 3e-20, 1e-41])) * (1.0 + rng.random())
    slope = float(rng.choice(ACUTE_SLOPES + (0.5, 0.25)))
    y_far = w * slope * (1.0 + 0.5 * rng.random())
    if n == 3:
        xy = np.array([[0.0, 0.0], [2.0 * w, y_far], [w, 0.5 * y_far * rng.random()]])
    else:
        xy = np.array([[0.0, 0.0], [w, w * slope], [2 * w, 2.5 * w * slope], [w, -w]])
    if rng.random() < 0.5:
        xy = xy[::-1].copy()
    return _f(_mirror(xy, int(rng.integers(8))))


PI_EDGE_SLOPE = 3.1786509e-8  # atan2(y, -1) rounds to (f32)pi below this slope and to the float below pi above it


def fam_pi_edge(oracle, rng, n):
    """A corner whose two atan2 values are (f32)pi or the float below it, and exactly 0: the centre sees one neighbour
    along a slope within a few parts in 10^7 of PI_EDGE_SLOPE, with |dx| not a power of two so that y/x is rounded before
    atan, and the other neighbour along a horizontal edge.  Whether the corner is acute then depends on the last bit of
    atan2 near pi."""
    x1 = float(rng.uniform(0.5, 4.0))
    y1 = -x1 * PI_EDGE_SLOPE * (1.0 + float(rng.uniform(-3e-7, 3e-7)))
    xy = np.array([[-float(rng.uniform(1.0, 4.0)), -float(rng.uniform(0.5, 3.0))], [x1, y1], [0.0, 0.0],
                   [-float(rng.uniform(0.5, 4.0)), 0.0]])
    xy = np.roll(xy, int(rng.integers(4)), axis=0)
    return pad(_f(xy[::-1] if rng.random() < 0.5 else xy), n, rng)


def fam_subnormal_axis(oracle, rng, n):
    """An integer-grid sound polygon with only its y (or only its x) coordinates scaled by 2^-140 into the subnormal
    range.  Differences along that axis are subnormal or +-0 while the other axis stays ordinary, so the side-test
    products are subnormal but not zero, and atan2 sees (subnormal, +-0) vectors: pi/2, which a flushed atan2 turns
    into 0 or +-pi."""
    xy = _sound(oracle, n, int(rng.integers(0, 2)), int(rng.integers(1 << 30)))
    xy = np.round(xy * max(0.1, n / 200.0) * float(rng.uniform(0.5, 2.0)))
    xy[:, int(rng.integers(2))] *= 2.0 ** -140
    return _f(_mirror(xy, int(rng.integers(4))))


def pad(p, n, rng):
    """p with n - len(p) points inserted on a shallow outward arc over one of its edges: a polygon of any size class
    that keeps p's corners.  The arc points are in general position."""
    p = np.asarray(p, dtype=np.float64)
    m = n - len(p)
    if m <= 0:
        return _f(p)
    i = int(rng.integers(len(p)))
    a, b = p[i], p[(i + 1) % len(p)]
    area = np.sum(p[:, 0] * np.roll(p[:, 1], -1) - np.roll(p[:, 0], -1) * p[:, 1])
    d = b - a
    out = np.array([d[1], -d[0]]) * (1.0 if area > 0 else -1.0)
    t = (np.arange(m) + 1.0) / (m + 1.0)
    arc = a + t[:, None] * d + (0.25 * np.sin(np.pi * t))[:, None] * out
    return _f(np.concatenate([p[: i + 1], arc, p[i + 1:]]))


# small-polygon families: run at the small sizes; pad() carries their killing cases into the larger classes
SMALL_FAMILIES = {"pi_edge": fam_pi_edge, "subnormal_axis": fam_subnormal_axis}

FAMILIES = {"grid_pm0": fam_grid_pm0, "ylevels": fam_ylevels, "twins": fam_twins, "scaled": fam_scaled,
            "collinear": fam_collinear, "acute": fam_acute, "edge0": fam_edge0}


# ---- running the oracle -------------------------------------------------------------------------------------------------
def pack(polys):
    xy = np.concatenate([p.reshape(-1, 2) for p in polys]).astype(np.float32) if polys else np.zeros((0, 2), np.float32)
    fp = np.concatenate([[0], np.cumsum([len(p) for p in polys])]).astype(np.uint64)
    return xy, fp


def per_polygon_outputs(oracle, xy, fp, op, layout=None):
    """Oracle outputs split per polygon: (status, ntri, vertex bytes, bbox bits) tuples."""
    kw = {} if layout is None else {"layout": layout}
    r = oracle.polygon_batch(xy, fp, offset_prime=op, nthreads=0, want_ids=False, **kw)
    per = (layout or oracle.GPUVERTEX_DECL)[0] * 3
    ft = r["first_tri"]
    bb = r["bbox"].view(np.uint32)
    return [(int(r["status"][i]), int(r["ntri"][i]), r["vtx"][int(ft[i]) * per:int(ft[i + 1]) * per].tobytes(),
             tuple(bb[i].tolist())) for i in range(len(fp) - 1)], r


def kill_matrix(oracle, xy, fp, op):
    """{mutant: boolean array over the polygons: the mutant changes that polygon's output}, and the reference outputs."""
    with oracle.mutant(None):
        ref, r = per_polygon_outputs(oracle, xy, fp, op)
    kills = {}
    for name in oracle.MUTANTS:
        with oracle.mutant(name):
            got, _ = per_polygon_outputs(oracle, xy, fp, op)
        kills[name] = np.array([a != b for a, b in zip(ref, got)], dtype=bool)
    return kills, r


class CaseSet:
    """Polygons with their explicit (offset, prime) edge orders, family names and size classes."""

    def __init__(self, polys, op, fams):
        self.polys, self.op, self.fams = list(polys), np.asarray(op, dtype=np.uint32).reshape(-1, 2), list(fams)
        self.classes = [size_class(len(p)) for p in self.polys]

    def __len__(self):
        return len(self.polys)

    def packed(self, idx=None):
        idx = range(len(self.polys)) if idx is None else idx
        xy, fp = pack([self.polys[i] for i in idx])
        return xy, fp, self.op[list(idx)]


def _orders(oracle, rng, n, k):
    """k explicit (offset, prime) pairs: what unirand_seed produces for n (a permutation of the edges)."""
    return [oracle.unirand_seed(n, int(rng.integers(1 << 62)), int(rng.integers(1 << 30))) for _ in range(k)]


_CACHE = {}


def _run_one(oracle, name, xy, fp, op):
    with oracle.mutant(name):
        out, _ = per_polygon_outputs(oracle, xy, fp, op)
    return out


def kill_cases(oracle, seed=20261020):
    """The kill set: for every (mutant, size class) up to MAX_KEEP polygons on which the mutant changes the output, and
    two polygons per class whose differences overflow and two with a -0 / +0 tie in y.  Returns (CaseSet, {mutant: kill array over the set}).

    Pass 1 draws FAMILIES at every class size and SMALL_FAMILIES / fam_acute_small at the small sizes, with seeded edge
    orders.  Pass 2 fills the (mutant, class) pairs that pass 1 left empty: it pads small polygons that kill the mutant
    to sizes of that class (pad()) and keeps the padded polygons that still kill it."""
    if seed in _CACHE:
        return _CACHE[seed]
    rng = np.random.default_rng(seed)
    polys, ops, fams = [], [], []

    def add(p, fname, k=1):
        for o in _orders(oracle, rng, len(p), k):
            polys.append(p)
            ops.append(o)
            fams.append(fname)

    for cname, _, _ in CLASSES:
        for n in CLASS_SIZES[cname]:
            reps = 4 if n <= 16 else 2 if n <= 1024 else 1
            for fname, fn in FAMILIES.items():
                for _ in range(reps):
                    add(fn(oracle, rng, n), fname, 2 if n <= 1024 else 1)
            if n <= 8:
                for fname, fn in SMALL_FAMILIES.items():
                    for _ in range(40):
                        add(fn(oracle, rng, n), fname)
            if n <= 4:
                for _ in range(24):
                    add(fam_acute_small(oracle, rng, n if rng.random() < 0.5 else 3), "acute_small")
    cand = CaseSet(polys, ops, fams)
    with np.errstate(all="ignore"):
        kills, _ = kill_matrix(oracle, *cand.packed())
    keep, count = [], {}
    for i in range(len(cand)):
        want = False
        for m, k in kills.items():
            if k[i] and count.get((m, cand.classes[i]), 0) < MAX_KEEP:
                count[(m, cand.classes[i])] = count.get((m, cand.classes[i]), 0) + 1
                want = True
        for feature, has in (("overflow", has_overflowing_difference), ("pm0_tie", has_pm0_y_tie)):
            if not want and has(cand.polys[i]):  # kept whether or not a mutant sees it
                want = count.get((feature, cand.classes[i]), 0) < 2
                count[(feature, cand.classes[i])] = count.get((feature, cand.classes[i]), 0) + 1
        if want:
            keep.append(i)
    kept = [(cand.polys[i], cand.op[i], cand.fams[i]) for i in keep]
    final = {m: k[keep] for m, k in kills.items()}

    # pass 2: pad small killers into the classes pass 1 missed
    pp, pop, pfam, pmut = [], [], [], []
    for m, k in kills.items():
        src = [i for i in np.nonzero(k)[0] if len(cand.polys[i]) <= 16][:PAD_SOURCES]
        if not src:
            continue
        for cname, lo, hi in CLASSES[1:]:
            if count.get((m, cname), 0):
                continue
            for j, i in enumerate(src):
                n = CLASS_SIZES[cname][j % len(CLASS_SIZES[cname])]
                p = pad(cand.polys[i], n, rng)
                for o in _orders(oracle, rng, n, 2):
                    pp.append(p)
                    pop.append(o)
                    pfam.append("padded_" + cand.fams[i])
                    pmut.append(m)
    padded = []
    if pp:
        pc = CaseSet(pp, pop, pfam)
        with np.errstate(all="ignore"):
            ref = _run_one(oracle, None, *pc.packed())
            for m in dict.fromkeys(pmut):
                idx = [i for i, mm in enumerate(pmut) if mm == m]
                got = _run_one(oracle, m, *pc.packed(idx))
                for i, g in zip(idx, got):
                    if g != ref[i] and count.get((m, pc.classes[i]), 0) < PAD_KEEP:
                        count[(m, pc.classes[i])] = count.get((m, pc.classes[i]), 0) + 1
                        padded.append(i)
        if padded:  # every mutant on the padded polygons kept
            padded.sort()
            with np.errstate(all="ignore"):
                pk, _ = kill_matrix(oracle, *pc.packed(padded))
            kept += [(pc.polys[i], pc.op[i], pc.fams[i]) for i in padded]
            final = {m: np.concatenate([final[m], pk[m]]) for m in final}
    cs = CaseSet([k[0] for k in kept], [k[1] for k in kept], [k[2] for k in kept])
    _CACHE[seed] = (cs, final)
    return cs, final


# ---- non-finite input -----------------------------------------------------------------------------------------------------
NONFINITE_WORDS = {"qnan": 0x7FC00000, "snan": 0x7FA00001, "neg_nan_payload": 0xFFC01234, "pinf": 0x7F800000,
                   "ninf": 0xFF800000}


def nonfinite_cases(oracle, seed=20261021):
    """Sound polygons of every size class with one non-finite word in x only or in y only, at the first, a middle and the
    last point (quiet, signalling and negative-payload NaN, +inf, -inf), and finite polygons that reach +-FLT_MAX, which
    must not be flagged.  Returns (CaseSet, expected_nonfinite bool array, description list)."""
    rng = np.random.default_rng(seed)
    polys, ops, fams, flagged, desc = [], [], [], [], []
    names = list(NONFINITE_WORDS)
    for cname, lo, hi in CLASSES:
        for k, n in enumerate(CLASS_SIZES[cname][-2:] if cname != "le64" else (4, 7, 64)):
            base = _f(_sound(oracle, n, oracle.FAMILY_ELLIPSE if k % 2 else oracle.FAMILY_ZIPPER, int(rng.integers(1 << 30))))
            for c in (0, 1):
                for where, at in (("first", 0), ("middle", n // 2), ("last", n - 1)):
                    w = names[(len(polys) + c) % len(names)]
                    p = base.copy()
                    p.view(np.uint32)[at, c] = NONFINITE_WORDS[w]
                    polys.append(p)
                    flagged.append(True)
                    desc.append((cname, n, "xy"[c], where, w))
            m = base.copy().astype(np.float64)
            m = m / np.abs(m).max(0) * FLT_MAX
            p = _f(np.clip(m, -FLT_MAX, FLT_MAX))
            p[int(np.argmax(p[:, 0]))] = (FLT_MAX, p[int(np.argmax(p[:, 0])), 1])
            p[int(np.argmin(p[:, 1])), 1] = -FLT_MAX
            polys.append(p)
            flagged.append(False)
            desc.append((cname, n, "-", "flt_max", "finite"))
    for p in polys:
        ops.append(_orders(oracle, rng, len(p), 1)[0])
        fams.append("nonfinite")
    return CaseSet(polys, ops, fams), np.array(flagged), desc


# ---- properties the tests check on the cases ------------------------------------------------------------------------------
def has_pm0_y_tie(p):
    """Two points with y == 0 of opposite zero signs and distinct x."""
    z = p[:, 1] == 0
    s = np.signbit(p[z, 1])
    return bool(s.any() and (~s).any() and len(np.unique(p[z, 0])) > 1)


def side_test_terms(p):
    """The products and differences of is_left_of for the consecutive triples of a polygon, rounded in f32."""
    a, b, q = p, np.roll(p, -1, 0), np.roll(p, -2, 0)
    with np.errstate(all="ignore"):
        d = [b[:, 0] - a[:, 0], q[:, 1] - a[:, 1], b[:, 1] - a[:, 1], q[:, 0] - a[:, 0]]
        return d, [d[0] * d[1], d[2] * d[3]]


def has_subnormal_product(p):
    _, prods = side_test_terms(p)
    return any(bool(((x != 0) & (np.abs(x) < np.float32(2.0 ** -126))).any()) for x in prods)


def has_overflowing_difference(p):
    if not np.isfinite(p).all():
        return False
    diffs, _ = side_test_terms(p)
    return any(bool(np.isinf(x).any()) for x in diffs)
