"""Parity fuzz: the CUDA triangulation through the C ABI vs the CPU oracle, byte for byte, on inputs the unit tests
do not enumerate -- every synthetic family under exact geometric transformations (reversal, mirrors, axis swap,
power-of-two scaling), quantised coordinates (ties in y, collinear runs), duplicated vertices (the coincident-point
path), random self-intersecting rings (where the reference mostly fails: the failure must be the same failure),
and size mixes around every class boundary.  Test infrastructure: the oracle is the checker, not the product.

    python scripts/fuzz_parity.py --rounds 60 --seed 1 --out gpurun_out/fuzz.json     # on a GPU box
    MR_B200_LIB=myrenderer_b200/lib/libmyrenderer_b200_checked.so python scripts/fuzz_parity.py ...   # bounds-checked build

Every case appends one line to <out>.log before and after it runs, so a hang names its case.
On a shared GPU box always run it under `timeout -s KILL <seconds>`: --budget-s only stops NEW cases from starting.
"""
import argparse
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "oracle"))

BOUNDARIES = [64, 128, 168, 216, 288, 368, 504, 608, 768, 1024]


def sizes_for(rng, mix):
    if mix == "small":
        return rng.integers(3, 65, size=int(rng.integers(2000, 20000)))
    if mix == "tiny":
        return rng.integers(2, 9, size=int(rng.integers(1000, 5000)))
    if mix == "loguniform":
        k = int(rng.integers(300, 2500))
        return np.exp(rng.uniform(np.log(8), np.log(1024), size=k)).astype(np.int64)
    if mix == "boundaries":
        s = np.array([b + d for b in BOUNDARIES for d in (-1, 0, 1)])
        return rng.permutation(np.repeat(s, int(rng.integers(1, 4))))
    if mix == "xl":
        return np.concatenate([rng.integers(1025, 3073, size=6), rng.integers(3073, 4097, size=2), rng.integers(3, 1025, size=40)])
    if mix == "few":  # the small-batch path when the buffers are host memory
        return rng.integers(3, 300, size=int(rng.integers(1, 40)))
    raise ValueError(mix)


def per_polygon(xy, fp, fn):
    out = xy.copy()
    for i in range(len(fp) - 1):
        a, z = int(fp[i]), int(fp[i + 1])
        out[a:z] = fn(out[a:z], i)
    return out


def transform(rng, xy, fp, how):
    if how == "identity":
        return xy
    if how == "reverse":
        return per_polygon(xy, fp, lambda p, i: p[::-1])
    if how == "rotate_start":
        return per_polygon(xy, fp, lambda p, i: np.roll(p, int(rng.integers(0, len(p))), axis=0))
    if how == "swap_axes":
        return np.ascontiguousarray(xy[:, ::-1])
    if how == "negate_y":
        return xy * np.array([1.0, -1.0], dtype=np.float32)
    if how == "negate_x":
        return xy * np.array([-1.0, 1.0], dtype=np.float32)
    if how == "scale_up":
        return xy * np.float32(2.0 ** 40)
    if how == "scale_down":
        return xy * np.float32(2.0 ** -60)
    if how == "quantise":
        q = np.float32(rng.choice([0.25, 1.0, 4.0]))
        return (np.round(xy / q) * q).astype(np.float32)
    if how == "duplicate":
        def dup(p, i):
            if len(p) >= 4 and (i % 3) == 0:
                k = int(rng.integers(0, len(p) - 1))
                p = p.copy()
                p[k + 1] = p[k] if (i % 2) else p[(k + 2) % len(p)]
            return p
        return per_polygon(xy, fp, dup)
    if how == "same_y":  # a handful of y levels: the order by (y, x) is decided by x almost everywhere
        out = xy.copy()
        out[:, 1] = np.round(out[:, 1] / np.float32(16.0)) * np.float32(16.0)
        return out
    if how == "collinear":
        def mid(p, i):
            if len(p) >= 5:
                p = p.copy()
                for k in range(1, len(p) - 1, 3):
                    p[k] = (p[k - 1] + p[k + 1]) * np.float32(0.5)
            return p
        return per_polygon(xy, fp, mid)
    if how == "scale_huge":  # products overflow to inf in the acute test and the side tests
        return xy * np.float32(2.0 ** 100)
    if how == "float_edges":  # signed zeros, subnormal coordinates / products, overflowing differences, mirrors
        def edge(p, i):
            k = int(rng.integers(0, 4))
            c = p.astype(np.float64) - p.astype(np.float64).mean(0)
            c = c * np.array([1.0 if rng.random() < 0.5 else -1.0, 1.0 if rng.random() < 0.5 else -1.0])
            if k == 0:  # quarter grid: small negative coordinates round to -0
                return (np.round(c * 4.0) / 4.0).astype(np.float32)
            return (c * (2.0 ** -140, 2.0 ** -75, 2.0 ** 121)[k - 1]).clip(-3.4e38, 3.4e38).astype(np.float32)
        return per_polygon(xy, fp, edge)
    if how == "mixed":
        pool = ["identity", "reverse", "quantise", "noise", "duplicate", "collinear", "float_edges"]
        out = xy.copy()
        for i in range(len(fp) - 1):
            a, z = int(fp[i]), int(fp[i + 1])
            sub_fp = np.array([0, z - a], dtype=np.uint64)
            out[a:z] = transform(rng, np.ascontiguousarray(out[a:z]), sub_fp, pool[int(rng.integers(0, len(pool)))])
        return out
    if how == "noise":
        return (rng.uniform(-100, 100, size=xy.shape)).astype(np.float32)
    if how == "noise_grid":
        return rng.integers(-8, 9, size=xy.shape).astype(np.float32)
    raise ValueError(how)


TRANSFORMS = ["identity", "reverse", "rotate_start", "swap_axes", "negate_y", "negate_x", "scale_up", "scale_down", "quantise",
              "duplicate", "noise", "noise_grid", "same_y", "collinear", "scale_huge", "float_edges", "mixed"]
MIXES = ["small", "small", "tiny", "loguniform", "loguniform", "boundaries", "xl", "few"]


def draw_layout(rng, which):
    """(stride, attrs) for GPUVertex-like vertices: x (2 floats) and optionally a colour (3 or 4 floats)."""
    if which == "decl":
        return (32, ((0, 2), (16, 3)))
    if which == "zigauto":
        return (32, ((16, 2), (0, 3)))
    for _ in range(100):
        stride = 4 * int(rng.integers(2, 17))
        slots = stride // 4
        a = int(rng.integers(0, slots - 1))
        if rng.integers(0, 4) == 0:
            return (stride, ((4 * a, 2),))
        cc = int(rng.choice([3, 4]))
        b = int(rng.integers(0, max(slots - cc + 1, 1)))
        if b + cc <= slots and (a + 2 <= b or b + cc <= a):
            return (stride, ((4 * a, 2), (4 * b, cc)))
    return (32, ((0, 2), (16, 3)))


def compare(ctx, mr, oracle, xy, fp, *, offset_prime, seed, poly_index0, layout, host, split, skip):
    """Runs the batch through mr_triangulate_batch -- whole, or cut into sub-range calls that write into the same buffers --
    and compares every output byte with the oracle.  Returns (None, ref) when they agree, else a description.
      host : False (device memory) | True / "host" (pageable host memory: staged / small-batch paths) | "pinned" |
             a dict placing each buffer on its own ("dev" / "host" / "pinned")
      split: None | "abs" (sub-calls index the full xy / vtx buffers: point_base = tri_base = 0)
                  | "rel" (sub-calls get pointers to their own slices: point_base = first_point[cut], tri_base = first_tri[cut])
      skip : subset of {"bbox", "status", "ntri"} passed as NULL"""
    import torch

    lay = mr.VertexLayout(layout[0], layout[1])
    ref = oracle.polygon_batch(xy, fp, offset_prime=offset_prime, seed=seed, poly_index0=poly_index0, layout=layout, nthreads=0)
    npoly = len(fp) - 1
    stride = layout[0]
    ft = ref["first_tri"].astype(np.uint64)
    nv = int(ft[-1]) * 3 * stride
    op = None if offset_prime is None else np.ascontiguousarray(offset_prime, dtype=np.uint32).reshape(-1)
    xyh = np.ascontiguousarray(xy, dtype=np.float32).reshape(-1)
    SENT = 0xA5
    h = dict(xy=xyh, fp=fp, ft=ft, op=op, vtx=np.full(nv + 32, SENT, dtype=np.uint8), bbox=np.full(4 * npoly, np.float32(-7.0), dtype=np.float32),
             st=np.full(npoly, 0xA5A5A5A5, dtype=np.uint32), nt=np.full(npoly, 0xA5A5A5A5, dtype=np.uint32))
    # where each buffer lives: "host" (pageable), "pinned" (page-locked: outputs are written zero-copy) or "dev"
    def signed(x):
        return x.view(np.int64) if x.dtype == np.uint64 else x.view(np.int32) if x.dtype == np.uint32 else x
    d, back = {}, {}
    for k, v in h.items():
        where = host if isinstance(host, str) else ("host" if host else "dev")
        if isinstance(host, dict):
            where = host[k]
        if v is None:
            d[k] = None
        elif where == "host":
            d[k] = v
        elif where == "pinned":
            t = torch.empty(v.shape, dtype=torch.from_numpy(signed(v)).dtype, pin_memory=True)
            t.copy_(torch.from_numpy(signed(v)))
            d[k] = t
        else:
            d[k] = torch.from_numpy(signed(v)).cuda()
    cuts = [0, npoly]
    if split and npoly >= 2:
        cuts = sorted(set([0, npoly] + [int(c) for c in np.random.default_rng(seed & 0xFFFF).integers(1, npoly, size=3)]))
    p = mr.Polygon(ctx, lay)
    for a, z in zip(cuts[:-1], cuts[1:]):
        pa, ta = int(fp[a]), int(ft[a])
        rel = split == "rel"
        p.triangulate(p.job(d["xy"][2 * pa:] if rel else d["xy"], d["fp"][a:], z - a,
                            vtx_out=d["vtx"][ta * 3 * stride:] if rel else d["vtx"], first_tri=d["ft"][a:],
                            bbox_out=None if "bbox" in skip else d["bbox"][4 * a:], status_out=None if "status" in skip else d["st"][a:],
                            ntri_out=None if "ntri" in skip else d["nt"][a:], offset_prime=None if op is None else d["op"][2 * a:],
                            seed=seed, poly_index0=poly_index0 + a, point_base=pa if rel else 0, tri_base=ta if rel else 0))
    ctx.sync()
    def fetch(k):
        x = d[k]
        return x if isinstance(x, np.ndarray) else x.cpu().numpy()
    gv, gb = fetch("vtx"), fetch("bbox")
    gs, gn = fetch("st").view(np.uint32), fetch("nt").view(np.uint32)
    if not (gv[nv:] == SENT).all():
        return "bytes behind the vertex range were written"
    gv = gv[:nv]
    if "status" in skip:
        if not (gs == 0xA5A5A5A5).all():
            return "status_out was NULL but the buffer was written"
    else:
        bad = np.where(gs != ref["status"])[0]
        if bad.size:
            i = int(bad[0])
            return "status of polygon %d (n=%d): gpu %d oracle %d (%d differ)" % (i, int(fp[i + 1] - fp[i]), int(gs[i]), int(ref["status"][i]), bad.size)
    if "ntri" not in skip and not np.array_equal(gn, ref["ntri"]):
        return "ntri differs"
    if not np.array_equal(gv, ref["vtx"][:nv]):
        per = stride * 3
        for i in range(npoly):
            a, z = int(ft[i]) * per, int(ft[i + 1]) * per
            if not np.array_equal(gv[a:z], ref["vtx"][a:z]):
                return "vertices of polygon %d (n=%d, oracle status %d) differ" % (i, int(fp[i + 1] - fp[i]), int(ref["status"][i]))
        return "vertex bytes differ outside every polygon range"
    if "bbox" not in skip and not np.array_equal(gb.view(np.uint32).reshape(-1), ref["bbox"].view(np.uint32).reshape(-1)):
        return "bbox differs"
    return None, ref


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=40)
    ap.add_argument("--seed", type=int, default=1)
    ap.add_argument("--out", default=os.path.join(ROOT, "gpurun_out", "fuzz.json"))
    ap.add_argument("--budget-s", type=float, default=600.0, help="stop starting new cases after this many seconds")
    a = ap.parse_args()
    import oracle as orc
    import myrenderer_b200 as mr

    ctx = mr.Context(0)
    flags = int(ctx.lib.mr_build_flags())
    log = open(a.out + ".log", "a")
    rng = np.random.default_rng(a.seed)
    t0 = time.time()
    cases, failures = [], []
    totals = {"polygons": 0, "points": 0, "status_ok": 0}
    families = [orc.FAMILY_STAR, orc.FAMILY_ELLIPSE, orc.FAMILY_ZIPPER]
    for r in range(a.rounds):
        if time.time() - t0 > a.budget_s:
            break
        mix = MIXES[r % len(MIXES)] if r < 2 * len(MIXES) else str(rng.choice(MIXES))
        how = TRANSFORMS[r % len(TRANSFORMS)] if r < 2 * len(TRANSFORMS) else str(rng.choice(TRANSFORMS))
        fam = families[int(rng.integers(0, 3))]
        sizes = np.maximum(sizes_for(rng, mix), 2)
        fp = np.concatenate([[0], np.cumsum(sizes)]).astype(np.uint64)
        seed = int(rng.integers(1, 2 ** 62))
        idx0 = int(rng.integers(0, 2 ** 40)) if r % 3 == 0 else 0
        xy = transform(rng, orc.synth_polygons(seed, fp, poly_index0=idx0, family=fam), fp, how)
        op = None
        if r % 4 == 1:  # explicit (offset, prime) pairs, including ones unirand_seed would never hand out
            n = sizes.astype(np.uint32)
            op = np.stack([rng.integers(0, 2 ** 31, size=len(n)).astype(np.uint32) % np.maximum(n, 1),
                           rng.choice(np.array([1, 2, 3, 5, 7, 11, 13, 1723, 10001567], dtype=np.uint32), size=len(n))], axis=1)
        host = (mix == "few") or (r % 5 == 2)
        if r % 5 in (3, 4) or (mix == "few" and r % 2):  # every buffer placed on its own
            host = {k: str(rng.choice(["dev", "host", "pinned"])) for k in ("xy", "fp", "ft", "op", "vtx", "bbox", "st", "nt")}
        elif r % 10 == 7:
            host = "pinned"
        layout = draw_layout(rng, ["decl", "decl", "zigauto", "generic", "generic"][int(rng.integers(0, 5))])
        split = [None, None, "abs", "rel"][int(rng.integers(0, 4))]
        skip = [s_ for s_ in ("bbox", "status", "ntri") if rng.integers(0, 6) == 0]
        desc = {"round": r, "mix": mix, "transform": how, "family": int(fam), "npoly": int(len(sizes)), "points": int(fp[-1]),
                "explicit_order": op is not None, "host_buffers": host, "layout": layout, "split": split, "null_outputs": skip}
        log.write("start " + json.dumps(desc) + "\n")
        log.flush()
        try:
            res = compare(ctx, mr, orc, xy, fp, offset_prime=op, seed=seed, poly_index0=idx0, layout=layout, host=host, split=split, skip=skip)
        except Exception as e:  # an error code for a job this script believes valid is a finding too
            res = "raised " + repr(e)
        if isinstance(res, tuple):
            ok = int((res[1]["status"] == 0).sum())
            desc["status_ok"] = ok
            totals["polygons"] += len(sizes)
            totals["points"] += int(fp[-1])
            totals["status_ok"] += ok
        else:
            desc["mismatch"] = res
            desc["seed"] = seed
            failures.append(desc)
            np.savez_compressed(a.out + ".fail%d.npz" % r, xy=xy, fp=fp, seed=seed, idx0=idx0, op=op if op is not None else np.zeros(0))
        cases.append(desc)
        log.write("done  " + json.dumps(desc) + "\n")
        log.flush()
    out = {"seed": a.seed, "cases": len(cases), "mismatches": len(failures), "totals": totals, "build_flags": flags,
           "library": os.environ.get("MR_B200_LIB", "default"), "seconds": round(time.time() - t0, 1), "failures": failures,
           "by_transform": {t: sum(1 for c in cases if c["transform"] == t) for t in TRANSFORMS},
           "by_mix": {m: sum(1 for c in cases if c["mix"] == m) for m in sorted(set(MIXES))}, "case_list": cases}
    json.dump(out, open(a.out, "w"), indent=1)
    print(json.dumps({k: out[k] for k in ("seed", "cases", "mismatches", "totals", "build_flags", "seconds")}))
    sys.exit(1 if failures else 0)


if __name__ == "__main__":
    main()
