"""Terrain tile culls on one GPU: mr_terrain_cull (the reference's SceneNode test) and mr_terrain_cull_frustum (the
six-plane test) on the same device-resident tile boxes, with the compacted index buffer on the device.

Cases: 4096^2 in 64 x 64-quad tiles (4,096 tiles), 16384^2 in 64 x 64 (65,536) and in 32 x 32 (262,144), each under the
four cameras of tests/_frustum.py (near, far, looking down, grazing; math.zig perspective * lookAt, aspect 16/9).  The
boxes are mr_terrain_tile_bounds of the hash-noise heightmap mr_synth_heightmap_u16 draws (the bench.py terrain).

Per case and test: visible tiles, indices written, microseconds per call (CUDA events around each call, mean of --calls
calls after --warmup, a 256 MiB buffer written between calls so that no call finds the boxes or outputs in L2), and the
index-write rate (4 bytes per index over the call time).  Prints one JSON line with the card's name and power limit,
read with nvidia-smi in the same run; --out also writes it to a file.

    python scripts/bench_cull.py --calls 100 --warmup 10 --out /tmp/bench_cull.json
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import _frustum as F  # noqa: E402

CASES = ((4096, 64), (16384, 64), (16384, 32))  # (n, square tile size in quads)
SEED = 0x5EED0001
TESTS = (("reference", "mr_terrain_cull"), ("frustum", "mr_terrain_cull_frustum"))


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
    ap.add_argument("--calls", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()

    import torch

    import myrenderer_b200 as mr
    from myrenderer_b200 import _capi

    if not torch.cuda.is_available():
        raise SystemExit("bench_cull.py needs a CUDA device")
    ctx = mr.Context(0)
    lib = ctx.lib
    dev = torch.device("cuda", 0)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    params = _capi.MrTerrainParams(0.2, 0.1, 5.0)
    results = []
    for n, t in CASES:
        h = torch.empty(n * n, dtype=torch.int16, device=dev)
        ctx.check(lib.mr_synth_heightmap_u16(ctx.handle, SEED, n, 0, n, h.data_ptr()), "synth")
        tiles_r, tiles_c = (n - 1 + t - 1) // t, (n - 1 + t - 1) // t
        ntiles = tiles_r * tiles_c
        boxes = torch.empty(ntiles * 8, dtype=torch.float32, device=dev)
        ctx.check(lib.mr_terrain_tile_bounds(ctx.handle, h.data_ptr(), _capi.MR_HEIGHT_U16, n, t, t, C.byref(params),
                                             boxes.data_ptr()), "tile_bounds")
        del h
        vis = torch.empty(ntiles, dtype=torch.int32, device=dev)
        ids = torch.empty(ntiles, dtype=torch.int32, device=dev)
        idx = torch.empty(6 * (n - 1) * (n - 1), dtype=torch.int32, device=dev)
        cnt = torch.zeros(2, dtype=torch.int64, device=dev)
        for cam, *_ in F.CAMERAS:
            m = np.ascontiguousarray(F.camera_by_name(cam), dtype=np.float32)
            for test, fn_name in TESTS:
                fn = getattr(lib, fn_name)

                def call():
                    ctx.check(fn(ctx.handle, boxes.data_ptr(), n, t, t, m.ctypes.data, vis.data_ptr(), ids.data_ptr(),
                                 idx.data_ptr(), cnt.data_ptr()), fn_name)

                for _ in range(args.warmup):
                    call()
                times = []
                for _ in range(args.calls):
                    flush.zero_()
                    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    a.record()
                    call()
                    b.record()
                    times.append((a, b))
                torch.cuda.synchronize()
                us = [a.elapsed_time(b) * 1e3 for a, b in times]
                visible, indices = (int(x) for x in cnt.cpu().tolist())
                mean = float(np.mean(us))
                results.append({"n": n, "tile": t, "tiles": ntiles, "camera": cam, "test": test, "visible_tiles": visible,
                                "indices": indices, "us_per_call": round(mean, 2),
                                "us_min": round(float(np.min(us)), 2), "us_median": round(float(np.median(us)), 2),
                                "index_write_GBps": round(indices * 4 / (mean * 1e-6) / 1e9, 1)})
        del boxes, vis, ids, idx, cnt
        torch.cuda.empty_cache()
    line = {"bench": "terrain_cull", "gpu": gpu_info(), "calls": args.calls, "warmup": args.warmup,
            "l2": "256 MiB buffer written before every timed call", "results": results}
    s = json.dumps(line)
    print(s)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(s + "\n")
    ctx.close()


if __name__ == "__main__":
    main()
