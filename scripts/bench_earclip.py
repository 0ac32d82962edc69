"""Polygon triangulation on one GPU: mr_triangulate_earclip (ear clipping) and mr_triangulate_batch (the reference's
triangulator) on the same device-resident polygons, outputs on the device.

Workloads: 100k polygons of 8..64 points (uniform sizes, the config-3 shape) and 1M polygons of 8..1024 points
(log-uniform, the config-5 shape), each for the star, ellipse and zipper families of mr_synth_polygons_family.  Per
workload and algorithm: milliseconds per call (CUDA events around each call, mean of --calls calls after --warmup, a
256 MiB buffer written between calls so that no call starts with its inputs in L2), polygons/s, points/s and the
fraction of polygons with status MR_POLY_OK.  Prints one JSON line with the card's name and power limit, read with
nvidia-smi in the same run; --out also writes it to a file.

    python scripts/bench_earclip.py --calls 5 --warmup 2 --out /tmp/bench_earclip.json
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

WORKLOADS = (("config3", 100_000, 8, 64, 0), ("config5", 1_000_000, 8, 1024, 1))  # (name, npoly, nmin, nmax, size dist)
FAMILIES = (("star", 0), ("ellipse", 1), ("zipper", 2))
ALGORITHMS = (("earclip", "mr_triangulate_earclip"), ("reference", "mr_triangulate_batch"))
SEED = 0x5EED0005


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                             text=True, timeout=30).stdout.strip().splitlines()[0]
        name, power = (s.strip() for s in out.split(","))
        return {"name": name, "power_limit": power}
    except Exception as e:  # the numbers stay, marked as from an unnamed card
        return {"name": None, "power_limit": None, "error": str(e)}


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--calls", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()

    import numpy as np
    import torch

    import myrenderer_b200 as mr
    from myrenderer_b200 import _capi

    if not torch.cuda.is_available():
        raise SystemExit("bench_earclip.py needs a CUDA device")
    ctx = mr.Context(0)
    lib = ctx.lib
    dev = torch.device("cuda", 0)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    layout = mr.Polygon(ctx).layout.native
    results = []
    for wname, npoly, nmin, nmax, dist in WORKLOADS:
        fp = np.zeros(npoly + 1, dtype=np.uint64)
        ctx.check(lib.mr_synth_polygon_sizes(SEED, 0, npoly, nmin, nmax, dist, fp.ctypes.data), "sizes")
        npts = int(fp[-1])
        ft = np.zeros(npoly + 1, dtype=np.uint64)
        ft[1:] = np.cumsum(np.diff(fp.astype(np.int64)) - 2)
        fp_d = torch.from_numpy(fp.view(np.int64)).to(dev)
        ft_d = torch.from_numpy(ft.view(np.int64)).to(dev)
        xy = torch.empty((npts, 2), dtype=torch.float32, device=dev)
        vtx = torch.empty(int(ft[-1]) * 3 * 32, dtype=torch.uint8, device=dev)
        bbox = torch.empty((npoly, 4), dtype=torch.float32, device=dev)
        status = torch.empty(npoly, dtype=torch.int32, device=dev)
        ntri = torch.empty(npoly, dtype=torch.int32, device=dev)
        for fname, fam in FAMILIES:
            ctx.check(lib.mr_synth_polygons_family(ctx.handle, fam, SEED, 0, fp_d.data_ptr(), npoly, xy.data_ptr()), "synth")
            job = _capi.MrPolygonJob()
            job.xy, job.first_point, job.point_base, job.npoly = xy.data_ptr(), fp_d.data_ptr(), 0, npoly
            job.offset_prime, job.seed, job.poly_index0 = None, SEED, 0
            job.layout = layout
            job.vtx_out, job.first_tri, job.tri_base = vtx.data_ptr(), ft_d.data_ptr(), 0
            job.bbox_out, job.status_out, job.ntri_out = bbox.data_ptr(), status.data_ptr(), ntri.data_ptr()
            for aname, fn_name in ALGORITHMS:
                fn = getattr(lib, fn_name)

                def call():
                    ctx.check(fn(ctx.handle, C.byref(job)), fn_name)

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
                results.append(dict(workload=wname, family=fname, algorithm=aname, npoly=npoly, points=npts,
                                    ms=round(ms, 3), polygons_per_s=round(npoly / ms * 1e3), points_per_s=round(npts / ms * 1e3),
                                    status_ok_fraction=round(ok, 6)))
                print(json.dumps(results[-1]), file=sys.stderr, flush=True)
        del vtx, xy
    line = json.dumps(dict(bench="earclip", gpu=gpu_info(), calls=args.calls, warmup=args.warmup,
                           l2="256 MiB written between calls", results=results))
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")
    ctx.close()


if __name__ == "__main__":
    main()
