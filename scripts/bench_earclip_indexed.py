"""Indexed ear clipping on one GPU: the same device-resident polygons written as vertices (mr_triangulate_earclip /
mr_triangulate_earclip_holes, 96 bytes per triangle in the GPUVertex layout), as indices only
(mr_triangulate_earclip_indexed with a NULL vtx_out, 12 bytes per triangle) and as both.

Workloads: 100k polygons of 8..64 points (uniform sizes, the config-3 shape of bench_earclip.py) for the star, ellipse
and zipper families; 1M polygons of 8..1024 points (log-uniform) for star and zipper; and the 100k-polygon 0..4-hole
batch of bench_earclip_holes.py.  The arms of a workload alternate call by call.  A last pair of arms writes the 100k
star batch's triangles into pinned host memory (vertices, or indices only), where the output crosses PCIe.  Per arm:
milliseconds per call (CUDA events, mean of --calls calls after --warmup, a 256 MiB buffer written before every call),
output bytes and the fraction of polygons with status MR_POLY_OK.  Prints one JSON line with the card's name and power
limit, read with nvidia-smi in the same run; --out also writes it to a file.

    python scripts/bench_earclip_indexed.py --calls 5 --warmup 2 --out profiles/r07_bench_earclip_indexed.json
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
import bench_earclip_holes as BH  # noqa: E402

SEED = 0x5EED0005
WORKLOADS = (("config3", 100_000, 8, 64, 0, ("star", "ellipse", "zipper")), ("config5", 1_000_000, 8, 1024, 1, ("star", "zipper")))
FAMILY = {"star": 0, "ellipse": 1, "zipper": 2}
ARMS = ("vertices", "indices", "both")


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
        raise SystemExit("bench_earclip_indexed.py needs a CUDA device")
    ctx = mr.Context(0)
    lib = ctx.lib
    dev = torch.device("cuda", 0)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    layout = mr.Polygon(ctx).layout.native
    results = []

    def d(a):
        return torch.from_numpy(a.view(np.int64) if a.dtype == np.uint64 else a).to(dev)

    def run(name, npoly, npts, xy, fp, ft, rings=None, host=False, arms=ARMS):
        """Times the arms on one batch, alternating them call by call; host: vtx / idx in pinned host memory."""
        ntri = int(ft[-1])
        fp_d, ft_d = d(fp), d(ft)

        def out(nbytes):
            return torch.empty(nbytes, dtype=torch.uint8, pin_memory=True) if host else \
                torch.empty(nbytes, dtype=torch.uint8, device=dev)

        vtx, idx = out(ntri * 96), out(ntri * 12)
        bbox = torch.empty((npoly, 4), dtype=torch.float32, device=dev)
        status = torch.empty(npoly, dtype=torch.int32, device=dev)
        nt = torch.empty(npoly, dtype=torch.int32, device=dev)
        job = _capi.MrPolygonJob()
        job.xy, job.first_point, job.point_base, job.npoly = xy.data_ptr(), fp_d.data_ptr(), 0, npoly
        job.layout = layout
        job.first_tri, job.tri_base = ft_d.data_ptr(), 0
        job.bbox_out, job.status_out, job.ntri_out = bbox.data_ptr(), status.data_ptr(), nt.data_ptr()
        rg = keep = None
        if rings is not None:
            keep = (d(rings[0]), d(rings[1]))
            rg = _capi.MrPolygonRings(keep[0].data_ptr(), 0, keep[1].data_ptr())
        ix = _capi.MrPolygonIndices(idx.data_ptr(), 0)

        def call(arm):
            job.vtx_out = None if arm == "indices" else vtx.data_ptr()
            if arm != "vertices":
                ctx.check(lib.mr_triangulate_earclip_indexed(ctx.handle, C.byref(job), None if rg is None else C.byref(rg),
                                                             C.byref(ix)), "mr_triangulate_earclip_indexed")
            elif rg is None:
                ctx.check(lib.mr_triangulate_earclip(ctx.handle, C.byref(job)), "mr_triangulate_earclip")
            else:
                ctx.check(lib.mr_triangulate_earclip_holes(ctx.handle, C.byref(job), C.byref(rg)), "mr_triangulate_earclip_holes")

        for _ in range(args.warmup):
            for arm in arms:
                call(arm)
        times = {arm: [] for arm in arms}
        for _ in range(args.calls):
            for arm in arms:
                flush.zero_()
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                call(arm)
                e1.record()
                torch.cuda.synchronize()
                times[arm].append(e0.elapsed_time(e1))
        ok = float((status == 0).double().mean().item())
        for arm in arms:
            ms = sum(times[arm]) / len(times[arm])
            out_bytes = ntri * ((96 if arm != "indices" else 0) + (12 if arm != "vertices" else 0))
            results.append(dict(workload=name, arm=arm, outputs="pinned host" if host else "device", npoly=npoly,
                                points=npts, triangles=ntri, ms=round(ms, 3), ms_min=round(min(times[arm]), 3),
                                output_bytes=out_bytes, status_ok_fraction=round(ok, 6)))
            print(json.dumps(results[-1]), file=sys.stderr, flush=True)

    for wname, npoly, nmin, nmax, dist, fams in WORKLOADS:
        npoly = max(1, int(npoly * args.scale))
        fp = np.zeros(npoly + 1, dtype=np.uint64)
        ctx.check(lib.mr_synth_polygon_sizes(SEED, 0, npoly, nmin, nmax, dist, fp.ctypes.data), "sizes")
        npts = int(fp[-1])
        ft = polygon_offsets_host(fp)
        xy = torch.empty((npts, 2), dtype=torch.float32, device=dev)
        fp_d = d(fp)
        for fname in fams:
            ctx.check(lib.mr_synth_polygons_family(ctx.handle, FAMILY[fname], SEED, 0, fp_d.data_ptr(), npoly, xy.data_ptr()),
                      "synth")
            run(f"{wname}_{fname}", npoly, npts, xy, fp, ft)
            if wname == "config3" and fname == "star":
                run(f"{wname}_{fname}", npoly, npts, xy, fp, ft, host=True, arms=("vertices", "indices"))
        del xy

    npoly = max(1, int(100_000 * args.scale))
    hxy, hfp, hfr, hrs, _, _ = BH.make(np, np.random.default_rng(BH.SEED), npoly, 8, 64, 0, 4)
    run("holes0to4", npoly, int(hfp[-1]), d(hxy), hfp, polygon_offsets_rings_host(hfp, hfr), rings=(hfr, hrs))

    line = json.dumps(dict(bench="earclip_indexed", gpu=gpu_info(), calls=args.calls, warmup=args.warmup,
                           l2="256 MiB written before every call", results=results))
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")
    ctx.close()


if __name__ == "__main__":
    main()
