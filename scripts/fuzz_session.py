"""Session fuzz: ONE context, a long random sequence of calls -- terrain builds (on the heights of fuzz_terrain, NaN and
infinite texels among them), tile boxes, culls, polygon batches of every shape, deliberately invalid calls (which must
fail with an error code and leave the context usable), scratch trims and tier-count queries in between -- every result
compared with the CPU oracle.  Looks for state that leaks from one call into the next (scratch growth and trim, the
cached launch plan, side streams, staging buffers).  Test infrastructure: the oracle is the checker.

    python scripts/fuzz_session.py --steps 400 --seed 1 --out gpurun_out/fuzz_session.json     # on a GPU box

On a shared GPU box always run it under `timeout -s KILL <seconds>`: --budget-s only stops NEW cases from starting.
"""
import argparse
import ctypes as C
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "oracle"))
sys.path.insert(0, os.path.join(ROOT, "tests"))
sys.path.insert(0, os.path.join(ROOT, "scripts"))
import _float_edges as E  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=300)
    ap.add_argument("--seed", type=int, default=1)
    ap.add_argument("--out", default=os.path.join(ROOT, "gpurun_out", "fuzz_session.json"))
    ap.add_argument("--budget-s", type=float, default=240.0)
    a = ap.parse_args()
    import torch
    import oracle as orc
    import myrenderer_b200 as mr
    import fuzz_parity as FP
    import fuzz_terrain as FT

    ctx = mr.Context(0)
    lib = ctx.lib
    rng = np.random.default_rng(a.seed)
    log = open(a.out + ".log", "a")
    t0 = time.time()
    counts = {"terrain": 0, "polygons": 0, "invalid": 0, "trim": 0, "tiers": 0}
    failures = []
    fams = [orc.FAMILY_STAR, orc.FAMILY_ELLIPSE, orc.FAMILY_ZIPPER]
    placements = ["dev", "host", "pinned"]

    def fail(step, what):
        failures.append({"step": step, "what": what})
        log.write("FAIL %d %s\n" % (step, what))
        log.flush()

    for step in range(a.steps):
        if time.time() - t0 > a.budget_s:
            break
        kind = str(rng.choice(["terrain", "polygons", "polygons", "invalid", "trim", "tiers"], p=[0.25, 0.3, 0.2, 0.15, 0.05, 0.05]))
        log.write("step %d %s\n" % (step, kind))
        log.flush()
        try:
            if kind == "terrain":
                n = FT.draw_n(rng)
                h = FT.draw_height(rng, orc, n)
                params = FT.draw_params(rng)
                lay_t = FT.draw_layout(rng)
                t = mr.Terrain(ctx, mr.VertexLayout(lay_t[0], lay_t[1]), params)
                host = {x: str(rng.choice(placements)) for x in ("height", "vtx", "idx")}
                vbytes, icount = n * n * lay_t[0], 6 * max(n - 1, 0) ** 2
                gv, gi = FT.run_build(ctx, t, torch, h, n, host, 0, n, 0, max(n - 1, 0), 0, n, 0, 0, vbytes, icount)
                ovtx, oidx = orc.terrain_build(h, n, layout=lay_t, params=params, nthreads=0)
                vbad = vbytes and E.float_mismatch(gv[:vbytes], ovtx, E.vertex_float_mask(vbytes, lay_t)) is not None
                if vbad or (icount and not np.array_equal(gi[:icount], oidx)):
                    fail(step, "terrain n=%d differs" % n)
                counts["terrain"] += 1
            elif kind == "polygons":
                mix = str(rng.choice(FP.MIXES))
                sizes = np.maximum(FP.sizes_for(rng, mix), 2)
                if len(sizes) > 4000:
                    sizes = sizes[:4000]
                fp = np.concatenate([[0], np.cumsum(sizes)]).astype(np.uint64)
                seed = int(rng.integers(1, 2 ** 62))
                xy = FP.transform(rng, orc.synth_polygons(seed, fp, family=fams[int(rng.integers(0, 3))]), fp, str(rng.choice(FP.TRANSFORMS)))
                host = {k: str(rng.choice(placements)) for k in ("xy", "fp", "ft", "op", "vtx", "bbox", "st", "nt")}
                if rng.integers(0, 3) == 0:
                    host = bool(rng.integers(0, 2))
                res = FP.compare(ctx, mr, orc, xy, fp, offset_prime=None, seed=seed, poly_index0=0,
                                 layout=FP.draw_layout(rng, str(rng.choice(["decl", "zigauto", "generic"]))), host=host,
                                 split=[None, "abs", "rel"][int(rng.integers(0, 3))], skip=[])
                if not isinstance(res, tuple):
                    fail(step, "polygons (%s): %s" % (mix, res))
                counts["polygons"] += 1
            elif kind == "invalid":
                which = int(rng.integers(0, 7))
                n = 64
                hd = torch.zeros(n * n, dtype=torch.int16, device="cuda")
                vtx = torch.empty(n * n * 32 + 64, dtype=torch.uint8, device="cuda")
                idx = torch.empty(6 * (n - 1) * (n - 1) + 16, dtype=torch.int32, device="cuda")
                T = mr.Terrain(ctx)
                P = mr.Polygon(ctx)
                ok = False
                try:
                    if which == 0:
                        T.build(T.job(hd, n, vtx_out=vtx, idx_out=idx.data_ptr() + 4))          # misaligned index buffer
                    elif which == 1:
                        T.build(T.job(hd, n, rows=(10, 5), vtx_out=vtx, idx_out=idx))           # reversed band
                    elif which == 2:
                        T.build(T.job(hd, n, rows=(0, n), height_row0=3, height_rows=n - 3, vtx_out=vtx))  # halo not covered
                    elif which == 3:
                        bad = mr.Terrain(ctx, mr.VertexLayout(30, ((0, 3),)))                    # stride not a multiple of 4
                        bad.build(bad.job(hd, n, vtx_out=vtx))
                    elif which == 4:
                        xy = np.zeros(8, dtype=np.float32)
                        fp = np.array([0, 4], dtype=np.uint64)
                        P.triangulate(P.job(xy, fp, 1, vtx_out=None, first_tri=np.array([0, 2], dtype=np.uint64)))  # no output buffer
                    elif which == 5:
                        ctx.check(lib.mr_terrain_tile_bounds(ctx.handle, hd.data_ptr(), 0, n, 0, 8, None, vtx.data_ptr()), "tile bounds")  # tile_rows 0
                    else:
                        badp = mr.Polygon(ctx, mr.VertexLayout(32, ((0, 2), (30, 3))))           # colour beyond the stride
                        xy = np.zeros(8, dtype=np.float32)
                        fp = np.array([0, 4], dtype=np.uint64)
                        badp.triangulate(badp.job(xy, fp, 1, vtx_out=np.zeros(192, dtype=np.uint8), first_tri=np.array([0, 2], dtype=np.uint64)))
                except mr.MrError:
                    ok = True
                if not ok:
                    fail(step, "invalid call %d was accepted" % which)
                counts["invalid"] += 1
            elif kind == "trim":
                ctx.check(lib.mr_context_trim(ctx.handle), "trim")
                counts["trim"] += 1
            else:
                tc = (C.c_uint32 * 8)()
                ctx.check(lib.mr_triangulate_tier_counts(ctx.handle, tc), "tier counts")
                counts["tiers"] += 1
        except Exception as e:
            fail(step, "%s raised %r" % (kind, e))
    ctx.sync()
    out = {"seed": a.seed, "steps": sum(counts.values()), "counts": counts, "mismatches": len(failures), "failures": failures[:50],
           "library": os.environ.get("MR_B200_LIB", "default"), "seconds": round(time.time() - t0, 1),
           "command": "python scripts/fuzz_session.py --steps %d --seed %d" % (a.steps, a.seed)}
    json.dump(out, open(a.out, "w"), indent=1)
    print(json.dumps({k: out[k] for k in ("seed", "steps", "counts", "mismatches", "seconds")}))
    sys.exit(1 if failures else 0)


if __name__ == "__main__":
    main()
