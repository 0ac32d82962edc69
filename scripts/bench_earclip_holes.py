"""Ear clipping of polygons with holes on one GPU: mr_triangulate_earclip_holes, and mr_triangulate_earclip on the same
outer rings without their holes (the cost of the bridging), device-resident inputs and outputs.

Workloads (star outer rings, radius 50..90 about the origin, triangle holes of side 1.5 on a 10 x 10 lattice within radius 30):
  holes0to4   100k polygons of 8..64 outer points with 0..4 holes
  holes1to16  100k polygons of 16..64 outer points with 1..16 holes
  holes100    10k polygons of 64 outer points with 100 holes
Per workload and entry point: milliseconds per call (CUDA events, mean of --calls calls after --warmup, a 256 MiB buffer
written between calls), polygons/s and the fraction of polygons with status MR_POLY_OK.  Prints one JSON line with the
card's name and power limit, read with nvidia-smi in the same run; --out also writes it to a file.

    python scripts/bench_earclip_holes.py --calls 5 --warmup 2 --out profiles/r06_bench_earclip_holes.json
"""
import argparse
import ctypes as C
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "scripts"))

from bench_earclip import gpu_info  # noqa: E402

WORKLOADS = (("holes0to4", 100_000, 8, 64, 0, 4), ("holes1to16", 100_000, 16, 64, 1, 16), ("holes100", 10_000, 64, 64, 100, 100))
SEED = 0x5EED0006


def make(np, rng, npoly, nmin, nmax, hmin, hmax):
    """(xy, first_point, first_ring, ring_start, outer-only xy, outer first_point)."""
    n = rng.integers(nmin, nmax + 1, npoly)
    h = rng.integers(hmin, hmax + 1, npoly)
    grid = np.stack(np.meshgrid(np.arange(-4.5, 5.0), np.arange(-4.5, 5.0)), -1).reshape(-1, 2) * 4.0  # 100 cells
    tri = np.array([(0.0, 0.0), (0.0, 1.5), (1.5, 0.75)])  # clockwise
    polys, outers = [], []
    for i in range(npoly):
        ang = (np.arange(n[i]) + 0.8 * rng.random(n[i])) * (2 * np.pi / n[i])  # gaps below 1.8 steps: the holes stay inside
        r = 50 + rng.random(n[i]) * 40
        outer = np.stack([r * np.cos(ang), r * np.sin(ang)], 1)
        cells = grid[rng.choice(len(grid), h[i], replace=False)] + rng.random((h[i], 2))
        holes = (cells[:, None, :] + tri[None]).reshape(-1, 2)
        polys.append(np.concatenate([outer, holes]))
        outers.append(outer)
    fp = np.zeros(npoly + 1, np.uint64)
    fp[1:] = np.cumsum(n + 3 * h)
    fr = np.zeros(npoly + 1, np.uint64)
    fr[1:] = np.cumsum(1 + h)
    rs = np.concatenate([fp[i] + np.concatenate([[0], n[i] + 3 * np.arange(h[i])]) for i in range(npoly)]).astype(np.uint64)
    ofp = np.zeros(npoly + 1, np.uint64)
    ofp[1:] = np.cumsum(n)
    return (np.concatenate(polys).astype(np.float32), fp, fr, rs, np.concatenate(outers).astype(np.float32), ofp)


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--calls", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--scale", type=float, default=1.0, help="fraction of each workload's polygon count")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()

    import numpy as np
    import torch

    import myrenderer_b200 as mr
    from myrenderer_b200 import _capi
    from myrenderer_b200.host import polygon_offsets_host, polygon_offsets_rings_host

    if not torch.cuda.is_available():
        raise SystemExit("bench_earclip_holes.py needs a CUDA device")
    ctx = mr.Context(0)
    lib = ctx.lib
    dev = torch.device("cuda", 0)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    layout = mr.Polygon(ctx).layout.native
    rng = np.random.default_rng(SEED)
    results = []

    def d(a):
        return torch.from_numpy(a.view(np.int64) if a.dtype == np.uint64 else a).to(dev)

    for wname, npoly, nmin, nmax, hmin, hmax in WORKLOADS:
        npoly = max(1, int(npoly * args.scale))
        xy, fp, fr, rs, oxy, ofp = make(np, rng, npoly, nmin, nmax, hmin, hmax)
        for entry in ("mr_triangulate_earclip_holes", "mr_triangulate_earclip"):
            holes = entry.endswith("holes")
            pts, firsts = (xy, fp) if holes else (oxy, ofp)
            ft = polygon_offsets_rings_host(fp, fr) if holes else polygon_offsets_host(ofp)
            bufs = dict(xy=d(pts), fp=d(firsts), ft=d(ft), fr=d(fr), rs=d(rs))
            vtx = torch.empty(int(ft[-1]) * 3 * 32, dtype=torch.uint8, device=dev)
            bbox = torch.empty((npoly, 4), dtype=torch.float32, device=dev)
            status = torch.empty(npoly, dtype=torch.int32, device=dev)
            ntri = torch.empty(npoly, dtype=torch.int32, device=dev)
            job = _capi.MrPolygonJob()
            job.xy, job.first_point, job.point_base, job.npoly = bufs["xy"].data_ptr(), bufs["fp"].data_ptr(), 0, npoly
            job.layout = layout
            job.vtx_out, job.first_tri, job.tri_base = vtx.data_ptr(), bufs["ft"].data_ptr(), 0
            job.bbox_out, job.status_out, job.ntri_out = bbox.data_ptr(), status.data_ptr(), ntri.data_ptr()
            rg = _capi.MrPolygonRings(bufs["fr"].data_ptr(), 0, bufs["rs"].data_ptr())

            def call():
                if holes:
                    ctx.check(lib.mr_triangulate_earclip_holes(ctx.handle, C.byref(job), C.byref(rg)), entry)
                else:
                    ctx.check(lib.mr_triangulate_earclip(ctx.handle, C.byref(job)), entry)

            for _ in range(args.warmup):
                call()
            times = []
            for _ in range(args.calls):
                flush.zero_()
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                call()
                e1.record()
                torch.cuda.synchronize()
                times.append(e0.elapsed_time(e1))
            ms = sum(times) / len(times)
            ok = float((status == 0).double().mean().item())
            results.append(dict(workload=wname, entry=entry, npoly=npoly, points=int(firsts[-1]),
                                holes=int(fr[-1]) - npoly if holes else 0, ms=round(ms, 3),
                                polygons_per_s=round(npoly / ms * 1e3), status_ok_fraction=round(ok, 6)))
            print(json.dumps(results[-1]), file=sys.stderr, flush=True)
    line = json.dumps(dict(bench="earclip_holes", gpu=gpu_info(), calls=args.calls, warmup=args.warmup,
                           l2="256 MiB written between calls", results=results))
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")
    ctx.close()


if __name__ == "__main__":
    main()
