#!/usr/bin/env python
"""bench.py -- the geometry hot path on N B200s of one node.

One *step* = one pass of the hot path over one batch of synthetic input:
    terrain   n x n hash-noise u16 heightmap  ->  vertices (pos + normal, 32 B) + u32 index buffer
    polygons  star-shaped simple polygons, 8..64 vertices, device-seeded unirand edge order
At N=1 the workload is BASELINE.json configs[1] + configs[2]: n = 4096 and 100,000 polygons
(SURVEY 8-d configs 2 and 3).  At N>1 the work is sharded with no data-path collective (weak
scaling): the terrain becomes an n_G x n_G heightmap with n_G = round(4096*sqrt(N)) cut into N
row bands with a one-row halo, the polygon batch becomes 100,000*N polygons cut into N
cost-balanced contiguous ranges; every rank produces its shard into its own HBM.

Headline `value` = terrain Mverts/s (unique grid vertices produced per second, vertices + normals +
indices all written), inputs resident in HBM.  The polygon throughput of the same steps is in
"polygons".  `e2e` is the same terrain metric through the reference-facing C-ABI call with pinned
HOST buffers (H2D of the heightmap and D2H of vertices + indices inside the timed region).

The same line also carries, at every N (strong scaling: the total work is fixed, cut into N shards):
    config4   BASELINE configs[3]: 16384^2 terrain, row bands; compute-only and -- N > 1 -- with the
              vertex bands stored straight into rank 0's buffer over NVLink (rank 0 generates the
              whole index buffer locally)
    config5   BASELINE configs[4]: 1,000,000 polygons, sizes log-uniform 8..1024, cost-balanced
              ranges, for the two families the reference triangulates correctly (convex ellipses and
              the non-convex zipper family); compute-only and gathered into rank 0's buffer
and, for N > 1, `gather` (the weak-scaled terrain built into rank 0's buffer, checked against a local
build), plus `single_polygon_us` (N = 1): Polygon.create_polygon's own call shape.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--dump-outputs DIR]
"""
from __future__ import annotations

import argparse
import ctypes as C
import hashlib
import json
import os
import statistics
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

TERRAIN_N1 = 4096
POLYS_PER_GPU = 100_000
SEED_TERRAIN = 0x5EED0001
SEED_POLY = 0x5EED0003
POLY_NMIN, POLY_NMAX = 8, 64
STRIDE = 32
CFG4_N, CFG4_SEED = 16384, 0x5EED0004
CFG5_NPOLY, CFG5_SEED = 1_000_000, 0x5EED0005
FAMILY_STAR, FAMILY_ELLIPSE, FAMILY_ZIPPER = 0, 1, 2
APP_POLYGON1 = [[62.742857, 106.97143], [93.085712, 65.828571], [147.08571, 85.628572], [122.14285, 144.77143],
                [102.34286, 93.857142], [79.199998, 130.37143], [81.00000, 105.17143]]  # App/App.zig:68-76


def terrain_size(world: int) -> int:
    return int(round(TERRAIN_N1 * world ** 0.5))


def terrain_bytes(n: int, rows: int, qrows: int):
    """Algorithmic bytes (SURVEY 8-d, u16 conversion fused so the read term is 2 B/texel)."""
    return 2 * rows * n + STRIDE * rows * n, 24 * qrows * (n - 1)


def peaks():
    try:
        p = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        return float(p["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md)"


def host_info():
    """What the end-to-end numbers at N > 1 are bound by: the box's host side (NUMA nodes, CPUs)."""
    nodes = None
    try:
        txt = open("/sys/devices/system/node/online").read().strip()  # e.g. "0" or "0-1"
        nodes = sum((int(b) - int(a) + 1) if "-" in part else 1
                    for part in txt.split(",") for a, _, b in [part.partition("-")])
    except Exception:
        pass
    return {"numa_nodes": nodes, "cpus": os.cpu_count()}


def fresh_traffic():
    """DRAM bytes per launch of the vertex kernel from an `ncu --set full` capture -- only when the capture was
    taken from THIS terrain.cu (the file's sha256 is stored beside it); otherwise None."""
    try:
        tj = json.load(open(os.path.join(ROOT, "profiles", "r03_traffic.json")))["terrain_vertices_k"]
        src = hashlib.sha256(open(os.path.join(ROOT, "myrenderer_b200", "csrc", "terrain.cu"), "rb").read()).hexdigest()
        if tj.get("terrain_cu_sha256") == src:
            return int(tj["traffic"]), tj.get("source")
    except Exception:
        pass
    return None, None


class ClockSampler:
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.p = None
        try:
            self.p = subprocess.Popen(
                ["nvidia-smi", f"--id={index}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "20"],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except Exception:
            self.p = None

    def stop(self):
        if self.p is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.p.terminate()
        try:
            out, _ = self.p.communicate(timeout=5)
        except Exception:
            self.p.kill()
            out = ""
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for line in out.strip().splitlines():
            f = [x.strip() for x in line.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0]))
                mx.append(float(f[1]))
            except ValueError:
                continue
            for name, v in zip(names, f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons)}


def workload_name(world: int) -> str:
    n = terrain_size(world)
    return (f"terrain {n}x{n} u16 hash-noise heightmap -> pos+normal vertices (32 B) + u32 indices, "
            f"row-band sharded x{world}; {POLYS_PER_GPU * world} star polygons n in [{POLY_NMIN},{POLY_NMAX}], "
            f"cost-balanced x{world}")


def config_dict(world: int) -> dict:
    """The `config` object -- the SAME for the b200 arm and the reference arm."""
    return {"workload": workload_name(world), "terrain_n": terrain_size(world), "polygons": POLYS_PER_GPU * world,
            "l2": "256 MiB buffer written between timed iterations; each step also writes >1.2 GB",
            "timing": "b200 arm: CUDA events on the launching stream, value = vertices / (vertex kernel + index kernel) "
                      "time, max over ranks; reference arm: wall clock of the CPU port on a bounded sample"}


# ------------------------------------------------------------------------------------------------
def cpu_reference_rates(world: int, nthreads: int, budget_polys: int = 200_000):
    """Times the CPU oracle (C restatement of the Zig source, prints removed) on a bounded sample of
    the N-GPU workload.  Returns rates + a description.  Only called for cpu_baseline / --impl reference."""
    from oracle import oracle as O

    n = terrain_size(world)
    rows = min(n, max(1, (TERRAIN_N1 * TERRAIN_N1) // n))  # ~one GPU's share of rows
    lo, hi = 0, min(n, rows + 1)
    h = O.synth_heightmap_u16(SEED_TERRAIN, n, 0, hi - lo)
    t0 = time.perf_counter()
    O.terrain_build(h, n, rows=(0, rows), qrows=(0, min(rows, n - 1)), nthreads=nthreads)
    t_terrain = time.perf_counter() - t0
    npoly = min(POLYS_PER_GPU * world, budget_polys)
    fp = O.synth_polygon_sizes(SEED_POLY, npoly, POLY_NMIN, POLY_NMAX)
    xy = O.synth_polygons(SEED_POLY, fp)
    t0 = time.perf_counter()
    O.polygon_batch(xy, fp, seed=SEED_POLY, nthreads=nthreads, want_ids=False)
    t_poly = time.perf_counter() - t0
    return {
        "terrain_mverts_per_s": rows * n / t_terrain / 1e6,
        "polygons_per_s": npoly / t_poly,
        "terrain_s": t_terrain, "polygons_s": t_poly,
        "sample": f"terrain rows [0,{rows}) of a {n}x{n} heightmap (vertices+normals+indices); "
                  f"first {npoly} polygons of the batch",
    }


def cpu_config5_rates(nthreads: int, sample: int = 4000):
    """CPU port on the first `sample` polygons of config 5 (both sound families)."""
    from oracle import oracle as O

    fp = O.synth_polygon_sizes(CFG5_SEED, sample, 8, 1024, dist=1)
    out = {"sample": f"first {sample} of the 1,000,000 polygons", "points": int(fp[-1])}
    for name, fam in (("ellipse", FAMILY_ELLIPSE), ("zipper", FAMILY_ZIPPER)):
        xy = O.synth_polygons(CFG5_SEED, fp, family=fam)
        t0 = time.perf_counter()
        O.polygon_batch(xy, fp, seed=CFG5_SEED, nthreads=nthreads, want_ids=False)
        dt = time.perf_counter() - t0
        out[name] = {"polygons_per_s": sample / dt, "mpoints_per_s": int(fp[-1]) / dt / 1e6}
    return out


def cpu_single_polygon_us(reps: int = 20000):
    """The CPU port on App.zig's polygon1, one call per polygon with reusable arenas (timed inside C)."""
    from oracle import oracle as O

    O.time_create_polygon(APP_POLYGON1, 3, 2, 2000)  # warm-up
    return O.time_create_polygon(APP_POLYGON1, 3, 2, reps) * 1e6


def run_reference_arm(args):
    """--impl reference: the reference's own CPU implementation of the path.  The Zig reference cannot
    be built here (no Zig toolchain, un-vendored deps), so this is the C restatement (oracle port)
    with debug prints removed, on all host threads."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from oracle import oracle as O

    T = O.hardware_threads()
    for _ in range(max(args.warmup, 0)):
        cpu_reference_rates(args.gpus, T, budget_polys=20_000)
    ts, tp, last = [], [], None
    for _ in range(args.steps):
        last = cpu_reference_rates(args.gpus, T)
        ts.append(last["terrain_mverts_per_s"])
        tp.append(last["polygons_per_s"])
    val = statistics.mean(ts)
    line = {
        "impl": "reference", "metric": "terrain_mverts_per_s", "value": val, "unit": "Mverts/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": 1e3 * (last["terrain_s"] + last["polygons_s"]), "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": config_dict(args.gpus),
        "polygons": {"value": statistics.mean(tp), "unit": "polygons/s"},
        "config5": cpu_config5_rates(T),
        "single_polygon_us": cpu_single_polygon_us(),
        "cpu_baseline": {"value": val, "unit": "Mverts/s", "cores": T, "kind": "port",
                         "sample": last["sample"], "polygons_per_s": statistics.mean(tp),
                         "note": "CPU = naive C restatement of the Zig source (oracle/), not the Zig binary; mean of "
                                 f"{args.steps} runs after {args.warmup} warm-ups"},
        "e2e": {"value": val, "unit": "Mverts/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    emit(line)


DUMP_SEED = 0x5EED00D0
# sample sizes of --dump-outputs (rows of each buffer), divided among the ranks: at most 52 MiB of .npy in all
DUMP_VERTICES, DUMP_QUADS, DUMP_TRIANGLES, DUMP_POLYGONS = 1 << 19, 1 << 18, 1 << 18, 1 << 17


def dump_sample(count: int, k: int, *key) -> np.ndarray:
    """Sorted ids of k of the `count` rows (all of them when k >= count); fixed by DUMP_SEED and `key`."""
    if k >= count:
        return np.arange(count, dtype=np.int64)
    return np.sort(np.random.default_rng([DUMP_SEED, *key]).choice(count, size=k, replace=False))


def dump_outputs(out_dir, rank, world, rows, qrows, n, vtx, idx, tlayout, ptri_base, pvtx, pbbox, pstat, pntri, player,
                 poly_base):
    """Writes what one step of the timed path produced, as a caller receives it, to out_dir/<name>.npy
    (<name>.rank<r>.npy at N > 1): the terrain's vertex attributes and index buffer, the polygon batch's vertex
    attributes, bounding boxes, status words and triangle counts.  Buffers with more rows than the sample size are
    represented by a seeded sample of their rows; `*_ids` holds the global row numbers of what was kept (a
    terrain vertex is row-major r * n + c, a terrain quad r * (n - 1) + c with 6 indices each)."""
    import torch

    def rows_of(buf, dtype, width, ids):
        return buf.view(dtype).view(-1, width)[torch.from_numpy(ids).to(buf.device)].cpu().numpy()

    def attribute_columns(layout):  # the float components of every attribute, in attribute order
        return [off // 4 + c for off, ncomp in layout.attributes for c in range(ncomp)]

    out = {}
    (r0, r1), (q0, q1) = rows, qrows
    vids = dump_sample((r1 - r0) * n, DUMP_VERTICES // world, rank, 0)
    out["terrain_vertex_ids"] = (r0 * n + vids).astype(np.float64)
    out["terrain_vertices"] = rows_of(vtx, torch.float32, tlayout.stride // 4, vids)[:, attribute_columns(tlayout)]
    qids = dump_sample((q1 - q0) * (n - 1), DUMP_QUADS // world, rank, 1)
    out["terrain_quad_ids"] = (q0 * (n - 1) + qids).astype(np.float64)
    out["terrain_indices"] = rows_of(idx[:(q1 - q0) * 6 * (n - 1)], torch.int32, 6, qids).view(np.uint32).astype(np.float64)
    tids = dump_sample(pvtx.numel() // (3 * player.stride), DUMP_TRIANGLES // world, rank, 2)
    out["polygon_triangle_ids"] = (ptri_base + tids).astype(np.float64)
    tri = rows_of(pvtx, torch.float32, 3 * player.stride // 4, tids).reshape(-1, 3, player.stride // 4)
    out["polygon_vertices"] = tri[:, :, attribute_columns(player)]
    pids = dump_sample(pstat.numel(), DUMP_POLYGONS // world, rank, 3)
    out["polygon_ids"] = (poly_base + pids).astype(np.float64)
    out["polygon_bbox"] = rows_of(pbbox, torch.float32, 4, pids)
    out["polygon_status"] = rows_of(pstat, torch.int32, 1, pids).view(np.uint32)[:, 0].astype(np.float64)
    out["polygon_ntri"] = rows_of(pntri, torch.int32, 1, pids).view(np.uint32)[:, 0].astype(np.float64)
    os.makedirs(out_dir, exist_ok=True)
    suffix = "" if world == 1 else f".rank{rank}"
    for name, a in out.items():
        np.save(os.path.join(out_dir, name + suffix + ".npy"), np.ascontiguousarray(a))


_STDOUT_FD = None


def emit(line: dict):
    data = (json.dumps(line) + "\n").encode()
    if _STDOUT_FD is None:
        sys.stdout.write(data.decode())
        sys.stdout.flush()
    else:
        os.write(_STDOUT_FD, data)


# ------------------------------------------------------------------------------------------------
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-gather", action="store_true", help="N>1: skip the NVLink gather legs (they are on by default)")
    ap.add_argument("--no-configs45", action="store_true", help="skip the BASELINE config 4 / config 5 legs")
    ap.add_argument("--gather", action="store_true", help="(accepted for compatibility: the gather is on by default)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last one computed to DIR/<name>.npy (a seeded sample "
                         "of the large buffers, 52 MiB at most) so that two builds can be compared output for output")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes the outputs of the b200 arm")
    args.warmup = max(args.warmup, 3) if args.impl == "b200" else args.warmup
    # stdout carries exactly one JSON line: anything a library prints there (NCCL's version banner, ...) goes to stderr
    global _STDOUT_FD
    sys.stdout.flush()
    _STDOUT_FD = os.dup(1)
    os.dup2(2, 1)

    if args.impl == "reference":
        run_reference_arm(args)
        return

    import torch
    import torch.distributed as dist

    import myrenderer_b200 as mr

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus:
        if world == 1 and args.gpus > 1:
            raise SystemExit("launch with torch.distributed.run --nproc-per-node N for --gpus N")
    torch.cuda.set_device(local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))

    dev = torch.device("cuda", local)
    ctx = mr.Context(local)  # runs on torch's current stream
    lib = ctx.lib
    T = mr.Terrain(ctx)
    P = mr.Polygon(ctx)

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    ev = lambda: torch.cuda.Event(enable_timing=True)

    def reduce_max(x):
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def reduce_sum(x):
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.SUM)
        return float(t.item())

    def timed(fn, reps, warm=1):
        """Device time of fn per call: events around each call, barrier between calls, mean; max over ranks."""
        for _ in range(warm):
            fn()
        barrier()
        ts = []
        for _ in range(reps):
            a, b = ev(), ev()
            a.record()
            fn()
            b.record()
            torch.cuda.synchronize()
            ts.append(a.elapsed_time(b))
            barrier()
        return reduce_max(sum(ts) / len(ts))

    def shared_buffer(nbytes):
        """rank 0 allocates; the other ranks map it through CUDA IPC (peer pointer over NVLink)."""
        base = C.c_void_p()
        handle = torch.zeros(64, dtype=torch.uint8, device=dev)
        if rank == 0:
            ctx.check(lib.mr_device_alloc(ctx.handle, nbytes, C.byref(base)), "alloc gather buffer")
            hb = (C.c_ubyte * 64)()
            ctx.check(lib.mr_ipc_export(ctx.handle, base, hb), "ipc export")
            handle.copy_(torch.frombuffer(bytearray(hb), dtype=torch.uint8))
        dist.broadcast(handle, src=0)
        if rank != 0:
            hb = (C.c_ubyte * 64).from_buffer_copy(bytes(handle.cpu().numpy().tobytes()))
            ctx.check(lib.mr_ipc_open(ctx.handle, hb, C.byref(base)), "ipc open")
        return base

    def release(base):
        barrier()
        if rank != 0:
            lib.mr_ipc_close(ctx.handle, base)
        barrier()
        if rank == 0:
            lib.mr_device_free(ctx.handle, base)

    def checksum(ptr, nbytes):
        """64-bit sum of the buffer's u64 words (nbytes multiple of 8), computed on the device in chunks."""
        total = 0
        chunk = 1 << 30
        tmp = torch.empty(min(chunk, nbytes) // 8, dtype=torch.int64, device=dev)
        off = 0
        while off < nbytes:
            m = min(chunk, nbytes - off)
            ctx.check(lib.mr_copy(ctx.handle, tmp.data_ptr(), ptr + off, m), "copy")
            ctx.sync()
            total = (total + int(tmp[: m // 8].sum().item())) & 0xFFFFFFFFFFFFFFFF
            off += m
        return total

    # ---- this rank's shard ---------------------------------------------------------------------
    n = terrain_size(world)
    rows_p = (C.c_uint32 * (world + 1))()
    qrows_p = (C.c_uint32 * (world + 1))()
    lib.mr_terrain_partition(n, world, rows_p, qrows_p)
    r0, r1, q0, q1 = rows_p[rank], rows_p[rank + 1], qrows_p[rank], qrows_p[rank + 1]
    lo, hi = max(r0 - 1, 0), min(r1 + 1, n)
    height = torch.empty((hi - lo) * n, dtype=torch.int16, device=dev)  # band + halo, u16
    ctx.check(lib.mr_synth_heightmap_u16(ctx.handle, SEED_TERRAIN, n, lo, hi - lo, height.data_ptr()), "synth heightmap")
    vtx = torch.empty((r1 - r0) * n * STRIDE, dtype=torch.uint8, device=dev)
    idx = torch.empty(max((q1 - q0) * 6 * (n - 1), 1), dtype=torch.int32, device=dev)
    job_v = T.job(height, n, rows=(r0, r1), qrows=(q0, q0), height_row0=lo, height_rows=hi - lo, vtx_out=vtx, vtx_row0=r0)
    job_i = T.job(height, n, rows=(r0, r0), qrows=(q0, q1), height_row0=lo, height_rows=hi - lo, idx_out=idx, idx_qrow0=q0)

    npoly_total = POLYS_PER_GPU * world
    fp_all = np.zeros(npoly_total + 1, dtype=np.uint64)
    lib.mr_synth_polygon_sizes(SEED_POLY, 0, npoly_total, POLY_NMIN, POLY_NMAX, 0, fp_all.ctypes.data)
    ranges = (C.c_uint32 * (world + 1))()
    lib.mr_polygon_partition(fp_all.ctypes.data, npoly_total, world, ranges)
    pa, pb = ranges[rank], ranges[rank + 1]
    fp = np.ascontiguousarray(fp_all[pa:pb + 1])
    ft = mr.polygon_offsets_host(fp)  # local triangle offsets
    npoly, npts, ntri = pb - pa, int(fp[-1] - fp[0]), int(ft[-1])
    fp_d = torch.from_numpy(fp.view(np.int64)).to(dev)
    ft_d = torch.from_numpy(ft.view(np.int64)).to(dev)
    xy = torch.empty(npts * 2, dtype=torch.float32, device=dev)
    ctx.check(lib.mr_synth_polygons(ctx.handle, SEED_POLY, pa, fp_d.data_ptr(), npoly, xy.data_ptr()), "synth polygons")
    pvtx = torch.empty(ntri * 3 * STRIDE, dtype=torch.uint8, device=dev)
    pbbox = torch.empty(npoly * 4, dtype=torch.float32, device=dev)
    pstat = torch.empty(npoly, dtype=torch.int32, device=dev)
    pntri = torch.empty(npoly, dtype=torch.int32, device=dev)
    job_p = P.job(xy, fp_d, npoly, vtx_out=pvtx, first_tri=ft_d, bbox_out=pbbox, status_out=pstat, ntri_out=pntri,
                  seed=SEED_POLY, poly_index0=pa, point_base=int(fp[0]))
    # second polygon workload: convex polygons of the same sizes (MR_FAMILY_ELLIPSE: every one is triangulated
    # correctly by the reference algorithm, so all of them end with status OK)
    cxy = torch.empty(npts * 2, dtype=torch.float32, device=dev)
    ctx.check(lib.mr_synth_polygons_family(ctx.handle, FAMILY_ELLIPSE, SEED_POLY, pa, fp_d.data_ptr(), npoly, cxy.data_ptr()), "synth")
    cstat = torch.empty(npoly, dtype=torch.int32, device=dev)
    job_c = P.job(cxy, fp_d, npoly, vtx_out=pvtx, first_tri=ft_d, bbox_out=pbbox, status_out=cstat, ntri_out=pntri,
                  seed=SEED_POLY, poly_index0=pa, point_base=int(fp[0]))
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)  # 2x L2
    ctx.sync()

    def step(timers=None):
        e0, e1, e2, e3 = ev(), ev(), ev(), ev()
        e0.record()
        T.build(job_v)
        e1.record()
        T.build(job_i)
        e2.record()
        P.triangulate(job_p)
        e3.record()
        if timers is not None:
            timers.append((e0, e1, e2, e3))

    for _ in range(args.warmup):
        step()
        flush.zero_()
    barrier()
    sampler = ClockSampler(local) if rank == 0 else None
    launches0 = ctx.launch_count
    timers = []
    wall0 = time.perf_counter()
    for _ in range(args.steps):
        step(timers)
        flush.zero_()  # L2 flush between timed iterations (outside the per-step event pairs)
    barrier()
    wall = time.perf_counter() - wall0
    launches = ctx.launch_count - launches0
    clocks = sampler.stop() if sampler else None
    tv = [a.elapsed_time(b) for a, b, _, _ in timers]
    ti = [b.elapsed_time(c) for _, b, c, _ in timers]
    tp = [c.elapsed_time(d) for _, _, c, d in timers]
    ms_v, ms_i, ms_p = (sum(x) / len(x) for x in (tv, ti, tp))
    ok_star = int((pstat == 0).sum().item())
    tiers = (C.c_uint32 * 8)()
    lib.mr_triangulate_tier_counts(ctx.handle, tiers)  # how the star batch was spread over the arena tiers
    if args.dump_outputs:  # before the convex batch below reuses the polygon output buffers
        ptri_base = int(mr.polygon_offsets_host(fp_all[:pa + 1])[-1])
        dump_outputs(args.dump_outputs, rank, world, (r0, r1), (q0, q1), n, vtx, idx, T.layout, ptri_base, pvtx, pbbox,
                     pstat, pntri, P.layout, pa)

    # ---- convex batch, same protocol -----------------------------------------------------------------
    for _ in range(2):
        P.triangulate(job_c)
    barrier()
    tc = []
    for _ in range(args.steps):
        a_, b_ = ev(), ev()
        a_.record()
        P.triangulate(job_c)
        b_.record()
        flush.zero_()
        tc.append((a_, b_))
    barrier()
    ms_c = sum(x.elapsed_time(y) for x, y in tc) / len(tc)
    ok_c = int((cstat == 0).sum().item())

    # ---- terrain tiles: bounding boxes + the reference's visibility test with compaction (SURVEY 8-f rank 4) -------
    cull = None
    if world == 1:
        tile = 64
        tr_, tc_ = C.c_uint32(), C.c_uint32()
        lib.mr_terrain_tile_count(n, tile, tile, C.byref(tr_), C.byref(tc_))
        ntiles = tr_.value * tc_.value
        boxes = torch.empty(ntiles * 8, dtype=torch.float32, device=dev)
        cidx = torch.empty(6 * (n - 1) * (n - 1), dtype=torch.int32, device=dev)
        ccnt = torch.zeros(2, dtype=torch.int64, device=dev)
        # q = (x, y + 1, z, 1): a tile passes iff its box reaches into the quadrant x > 0, z > 0 (about a quarter of them)
        m = np.ascontiguousarray(np.array([[1, 0, 0, 0], [0, 1, 0, 1], [0, 0, 1, 0], [0, 0, 0, 1]], dtype=np.float32).T.reshape(16))

        def do_bounds():
            ctx.check(lib.mr_terrain_tile_bounds(ctx.handle, height.data_ptr(), 0, n, tile, tile, None, boxes.data_ptr()), "tile bounds")

        def do_cull():
            ctx.check(lib.mr_terrain_cull(ctx.handle, boxes.data_ptr(), n, tile, tile, m.ctypes.data, None, None, cidx.data_ptr(),
                                          ccnt.data_ptr()), "cull")

        ms_tb = timed(do_bounds, reps=10, warm=2)
        ms_cu = timed(do_cull, reps=10, warm=2)
        cc = ccnt.cpu().numpy()
        cull = {"tile_quads": tile, "tiles": int(ntiles), "tile_bounds_us": ms_tb * 1e3, "cull_us": ms_cu * 1e3,
                "visible_tiles": int(cc[0]), "indices_written": int(cc[1]),
                "index_write_gb_per_s": int(cc[1]) * 4 / (ms_cu * 1e-3) / 1e9,
                "what": "mr_terrain_tile_bounds (per-tile min/max, reads the u16 heightmap once) and mr_terrain_cull "
                        "(SceneNode.zig:96-110 per tile + ordered compaction + compacted index buffer)"}
        del boxes, cidx

    # ---- end to end through the C ABI with pinned host buffers --------------------------------
    e2e = None
    if not args.no_e2e:
        h_height = torch.empty((hi - lo) * n, dtype=torch.int16, pin_memory=True)
        h_height.copy_(height)
        h_vtx = torch.empty((r1 - r0) * n * STRIDE, dtype=torch.uint8, pin_memory=True)
        h_idx = torch.empty(max((q1 - q0) * 6 * (n - 1), 1), dtype=torch.int32, pin_memory=True)
        h_xy = torch.empty(npts * 2, dtype=torch.float32, pin_memory=True)
        h_xy.copy_(xy)
        h_pvtx = torch.empty(ntri * 3 * STRIDE, dtype=torch.uint8, pin_memory=True)
        h_bbox = torch.empty(npoly * 4, dtype=torch.float32, pin_memory=True)
        h_stat = torch.empty(npoly, dtype=torch.int32, pin_memory=True)
        h_ntri = torch.empty(npoly, dtype=torch.int32, pin_memory=True)
        torch.cuda.synchronize()
        job_e = T.job(h_height, n, rows=(r0, r1), qrows=(q0, q1), height_row0=lo, height_rows=hi - lo,
                      vtx_out=h_vtx, vtx_row0=r0, idx_out=h_idx, idx_qrow0=q0)
        job_pe = P.job(h_xy, fp, npoly, vtx_out=h_pvtx, first_tri=ft, bbox_out=h_bbox, status_out=h_stat,
                       ntri_out=h_ntri, seed=SEED_POLY, poly_index0=pa, point_base=int(fp[0]))
        esteps = max(3, min(args.steps, 10))
        for _ in range(2):
            T.build(job_e)
            P.triangulate(job_pe)
        barrier()
        te, tpe = [], []
        for _ in range(esteps):
            a, b, c = ev(), ev(), ev()
            a.record()
            T.build(job_e)   # H2D heightmap -> kernels -> D2H vertices + indices, returns when the host buffers are filled
            b.record()
            P.triangulate(job_pe)
            c.record()
            torch.cuda.synchronize()
            te.append(a.elapsed_time(b))
            tpe.append(b.elapsed_time(c))
        barrier()
        # PCIe floor of the terrain call: the same bytes moved by plain pinned copies (D2H of vertices + indices, H2D of
        # the heightmap on a second stream -- the two directions overlap), all ranks at once like the call itself
        side = torch.cuda.Stream()
        tf = []
        for _ in range(3):
            a, b = ev(), ev()
            barrier()
            a.record()
            side.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(side):
                height.copy_(h_height, non_blocking=True)
            h_vtx.copy_(vtx, non_blocking=True)
            h_idx.copy_(idx, non_blocking=True)
            torch.cuda.current_stream().wait_stream(side)
            b.record()
            torch.cuda.synchronize()
            tf.append(a.elapsed_time(b))
        barrier()
        e2e = {"ms_terrain": sum(te) / len(te), "ms_polygons": sum(tpe) / len(tpe),
               "h2d_terrain": h_height.numel() * 2, "d2h_terrain": h_vtx.numel() + h_idx.numel() * 4,
               "h2d_poly": h_xy.numel() * 4 + fp.nbytes + ft.nbytes,
               "d2h_poly": h_pvtx.numel() + h_bbox.numel() * 4 + h_stat.numel() * 4 + h_ntri.numel() * 4,
               "status_ok": int((h_stat.numpy() == 0).sum()), "pcie_floor_ms": min(tf)}
        del h_vtx, h_idx, h_pvtx, h_height, h_xy

    # ---- single polygon: Polygon.create_polygon's own call shape (host pointers, one 7-gon) ------------
    single = None
    if world == 1:
        p1 = np.array(APP_POLYGON1, dtype=np.float32)
        sfp, sft = np.array([0, 7], dtype=np.uint64), np.array([0, 5], dtype=np.uint64)
        svtx = np.zeros(5 * 96, dtype=np.uint8)
        sbb, sst, snt = np.zeros(4, dtype=np.float32), np.zeros(1, dtype=np.uint32), np.zeros(1, dtype=np.uint32)
        sop = np.array([3, 2], dtype=np.uint32)
        sj = P.job(p1, sfp, 1, vtx_out=svtx, first_tri=sft, bbox_out=sbb, status_out=sst, ntri_out=snt, offset_prime=sop)
        for _ in range(50):
            P.triangulate(sj)
        l0 = ctx.launch_count
        ts_ = []
        for _ in range(1000):
            t0 = time.perf_counter()
            P.triangulate(sj)
            ts_.append(time.perf_counter() - t0)
        single = {"us": statistics.median(ts_) * 1e6, "p90_us": sorted(ts_)[900] * 1e6,
                  "launches_per_call": (ctx.launch_count - l0) / 1000, "status": int(sst[0]), "triangles": int(snt[0]),
                  "what": "mr_triangulate_batch, npoly = 1 (App.zig polygon1), every buffer in host memory, wall clock of "
                          "the blocking call, median of 1000"}

    # ---- N>1: weak-scaled terrain gathered into rank 0's buffer by NVLink peer stores -------------------
    gather = None
    want_gather = world > 1 and not args.no_gather
    if want_gather:
        try:
            total_bytes = n * n * STRIDE
            base = shared_buffer(total_bytes)
            job_g = T.job(height, n, rows=(r0, r1), qrows=(q0, q0), height_row0=lo, height_rows=hi - lo,
                          vtx_out=base.value, vtx_row0=0)  # global row origin: the band lands at its final offset
            ms_g = timed(lambda: T.build(job_g), reps=max(3, min(args.steps, 10)), warm=2)
            # check: every band in rank 0's buffer equals the band its owner built locally (sum of u64 words)
            T.build(job_v)
            ctx.sync()
            local_sum = checksum(vtx.data_ptr(), vtx.numel())
            sums = torch.tensor([local_sum & 0x7FFFFFFFFFFFFFFF], dtype=torch.int64, device=dev)
            allsums = [torch.zeros_like(sums) for _ in range(world)]
            dist.all_gather(allsums, sums)
            barrier()
            ok_gather = True
            if rank == 0:
                for g in range(world):
                    a_, z_ = rows_p[g] * n * STRIDE, rows_p[g + 1] * n * STRIDE
                    got = checksum(base.value + a_, z_ - a_) & 0x7FFFFFFFFFFFFFFF
                    ok_gather = ok_gather and got == int(allsums[g].item())
            # ceiling for the ingest rate: the same bands moved by plain peer copies (copy engines), all ranks at once
            def peer_copy():
                if rank != 0:
                    ctx.check(lib.mr_copy(ctx.handle, base.value + r0 * n * STRIDE, vtx.data_ptr(), vtx.numel()), "peer copy")
            ms_pc = timed(peer_copy, reps=3, warm=1)
            gather = {"ms": ms_g, "ok": bool(ok_gather), "peer_copy_ms": ms_pc}
            release(base)
        except Exception as exc:  # the gather figure is informative; never lose the main line over it
            gather = {"error": str(exc)[:200]}

    # ---- free the weak-scaling buffers before the full-size configs ---------------------------------------
    verts_local = (r1 - r0) * n
    bv, bi = terrain_bytes(n, r1 - r0, q1 - q0)
    del vtx, idx, height, pvtx, xy, cxy, job_v, job_i, job_p, job_c
    torch.cuda.empty_cache()
    lib.mr_context_trim(ctx.handle)

    cfg4 = cfg5 = None
    if not args.no_configs45:
        # (an exception in one of these legs must not cost the headline line; at N > 1 a one-sided failure would
        # still desynchronise the ranks, so the legs only catch what every rank hits alike, e.g. out of memory)
        try:
            cfg4 = run_config4(ctx, T, dev, rank, world, timed, shared_buffer, release, want_gather, checksum, barrier)
        except Exception as exc:
            cfg4 = {"error": str(exc)[:200]}
        torch.cuda.empty_cache()
        try:
            cfg5 = run_config5(ctx, P, dev, rank, world, timed, shared_buffer, release, want_gather, reduce_sum)
        except Exception as exc:
            cfg5 = {"error": str(exc)[:200]}
        torch.cuda.empty_cache()

    # ---- reduce over ranks: max time, sum of units ------------------------------------------------
    g_ms_v, g_ms_i, g_ms_p = reduce_max(ms_v), reduce_max(ms_i), reduce_max(ms_p)
    g_ms_terrain = reduce_max(ms_v + ms_i)
    g_ms_step = reduce_max(ms_v + ms_i + ms_p)
    verts_total = reduce_sum(verts_local)
    polys_total = reduce_sum(npoly)
    bytes_terrain_total = reduce_sum(bv + bi)
    launches_total = int(reduce_sum(launches))
    if e2e is not None:
        e_ms_t = reduce_max(e2e["ms_terrain"])
        e_ms_p = reduce_max(e2e["ms_polygons"])
        e_floor = reduce_max(e2e["pcie_floor_ms"])
        e_h2d = int(reduce_sum(e2e["h2d_terrain"] + e2e["h2d_poly"]))
        e_d2h = int(reduce_sum(e2e["d2h_terrain"] + e2e["d2h_poly"]))
    ok_total = reduce_sum(ok_star)
    g_ms_c = reduce_max(ms_c)
    ok_c_total = reduce_sum(ok_c)

    if rank == 0:
        peak, peak_src = peaks()
        value = verts_total / (g_ms_terrain * 1e-3) / 1e6
        achieved_v = bv / (ms_v * 1e-3) / 1e9  # rank 0's dominant kernel
        traffic, traffic_src = fresh_traffic() if (world == 1 and n == 4096) else (None, None)
        line = {
            "metric": "terrain_mverts_per_s",
            "value": value, "unit": "Mverts/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": g_ms_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic",
            "config": config_dict(world),
            "terrain": {"ms": g_ms_terrain, "ms_vertices_kernel": g_ms_v, "ms_indices_kernel": g_ms_i,
                        "achieved_gb_per_s": bytes_terrain_total / (g_ms_terrain * 1e-3) / 1e9,
                        "algorithmic_bytes": int(bytes_terrain_total)},
            "polygons": {"value": polys_total / (g_ms_p * 1e-3), "unit": "polygons/s", "ms": g_ms_p,
                         "status_ok_fraction": ok_total / polys_total,
                         "note": "star polygons of SURVEY 8-d config 3; the reference algorithm itself fails "
                                 "(overflow/underfill/null-unwrap) on the non-OK fraction and the kernel reproduces that"},
            "polygons_convex": {"value": polys_total / (g_ms_c * 1e-3), "unit": "polygons/s", "ms": g_ms_c,
                                "status_ok_fraction": ok_c_total / polys_total,
                                "note": "same sizes, MR_FAMILY_ELLIPSE (convex): a family the reference triangulates correctly"},
            "polygon_tiers": {"retried_with_contract_cap_arenas": int(sum(tiers[0:6])), "general_path": int(tiers[6]),
                              "note": "rank 0's star batch; everything else ran in the first shared-memory pass"},
            "gpu_launches": launches_total,
            "wall_s_timed_region": wall,
            "clocks": clocks,
            "roofline": {"bound": "hbm", "kernel": "terrain_vertices_k", "achieved": achieved_v, "peak": peak,
                         "unit": "GB/s", "frac": achieved_v / peak, "traffic": traffic, "traffic_source": traffic_src,
                         "peak_source": peak_src, "algorithmic_bytes_per_launch": int(bv),
                         "indices_kernel": {"achieved": bi / (ms_i * 1e-3) / 1e9, "frac": bi / (ms_i * 1e-3) / 1e9 / peak,
                                            "algorithmic_bytes_per_launch": int(bi)}},
        }
        if cfg4 is not None:
            line["config4"] = cfg4
        if cfg5 is not None:
            line["config5"] = cfg5
        if e2e is not None:
            line["e2e"] = {"value": verts_total / (e_ms_t * 1e-3) / 1e6, "unit": "Mverts/s",
                           "h2d_bytes_per_step": e_h2d, "d2h_bytes_per_step": e_d2h, "ms_terrain": e_ms_t,
                           "ms_polygons": e_ms_p, "polygons_per_s": polys_total / (e_ms_p * 1e-3),
                           "pcie_floor_ms": e_floor, "fraction_of_pcie_floor": e_floor / e_ms_t, "host": host_info(),
                           "path": "mr_terrain_build / mr_triangulate_batch with pinned host buffers; pcie_floor_ms = the "
                                   "terrain call's bytes moved by plain pinned copies (both directions at once)"}
        if cull is not None:
            line["terrain_cull"] = cull
        if single is not None:
            line["single_polygon_us"] = single["us"]
            line["single_polygon"] = single
        if gather is not None:
            if "ms" in gather:
                nv_bytes = n * n * STRIDE * (world - 1) / world
                gather.update({"what": "weak-scaled terrain: vertex bands stored directly into rank 0's buffer (IPC-mapped "
                                       "peer pointer); checked band by band against the local builds",
                               "nvlink_bytes": int(nv_bytes), "rank0_ingest_gb_per_s": nv_bytes / (gather["ms"] * 1e-3) / 1e9,
                               "peer_copy_gb_per_s": nv_bytes / (gather["peer_copy_ms"] * 1e-3) / 1e9,
                               "gather_inclusive_mverts_per_s": verts_total / (gather["ms"] * 1e-3) / 1e6})
            line["gather"] = gather
        if world == 1 and not args.no_cpu_baseline:
            from oracle import oracle as O  # CPU baseline leg only

            Tn = O.hardware_threads()
            cpu_reference_rates(1, Tn, budget_polys=20_000)  # warm-up
            runs = [cpu_reference_rates(1, Tn) for _ in range(3)]
            cpu1 = cpu_reference_rates(1, 1, budget_polys=20_000)
            line["cpu_baseline"] = {
                "value": statistics.mean(r["terrain_mverts_per_s"] for r in runs), "unit": "Mverts/s", "cores": Tn,
                "kind": "port", "sample": runs[-1]["sample"] + "; mean of 3 runs after a warm-up",
                "polygons_per_s": statistics.mean(r["polygons_per_s"] for r in runs),
                "single_thread": {"terrain_mverts_per_s": cpu1["terrain_mverts_per_s"],
                                  "polygons_per_s": cpu1["polygons_per_s"], "sample": cpu1["sample"]},
                "config5": cpu_config5_rates(Tn, sample=2000),
                "single_polygon_us": cpu_single_polygon_us(),
                "note": "CPU = NAIVE C restatement of the Zig source (oracle/), prints removed; not the Zig binary and "
                        "not tuned (five divisions per vertex, O(T*M) mountain search as in the reference)"}
        emit(line)
    if world > 1:
        dist.destroy_process_group()
    ctx.close()


def run_config4(ctx, T, dev, rank, world, timed, shared_buffer, release, want_gather, checksum, barrier):
    """BASELINE configs[3]: 16384^2 terrain, strong-scaled row bands."""
    import torch

    from myrenderer_b200 import sharding

    lib = ctx.lib
    n = CFG4_N
    sh = sharding.plan_terrain(n, rank, world)
    (r0, r1), (q0, q1), (lo, hi) = sh.rows, sh.qrows, sh.halo_rows
    height = torch.empty((hi - lo) * n, dtype=torch.int16, device=dev)
    ctx.check(lib.mr_synth_heightmap_u16(ctx.handle, CFG4_SEED, n, lo, hi - lo, height.data_ptr()), "synth")
    vtx = torch.empty((r1 - r0) * n * STRIDE, dtype=torch.uint8, device=dev)
    idx = torch.empty((q1 - q0) * 6 * (n - 1), dtype=torch.int32, device=dev)
    job_v = T.job(height, n, rows=(r0, r1), qrows=(q0, q0), height_row0=lo, height_rows=hi - lo, vtx_out=vtx, vtx_row0=r0)
    job_l = T.job(height, n, rows=(r0, r1), qrows=(q0, q1), height_row0=lo, height_rows=hi - lo, vtx_out=vtx, vtx_row0=r0,
                  idx_out=idx, idx_qrow0=q0)
    ms_c = timed(lambda: T.build(job_l), reps=5, warm=2)
    ms_v = timed(lambda: T.build(job_v), reps=5, warm=1)
    bytes4 = 34 * n * n + 24 * (n - 1) ** 2
    peak, _ = peaks()
    res = {"what": "16384 x 16384 heightmap, strong-scaled row bands with a one-row halo",
           "compute_ms": ms_c, "compute_gverts_per_s": n * n / (ms_c * 1e-3) / 1e9,
           "achieved_gb_per_s_aggregate": bytes4 / (ms_c * 1e-3) / 1e9,
           "frac_of_hbm_peak_per_gpu": bytes4 / (ms_c * 1e-3) / 1e9 / world / peak,
           "vertices_kernel_ms": ms_v, "vertices_kernel_frac_of_hbm_peak": 34 * n * (r1 - r0) / (ms_v * 1e-3) / 1e9 / peak,
           "algorithmic_bytes": bytes4}
    if world > 1 and want_gather:
        try:
            # one mesh on rank 0: the vertex bands travel over NVLink (peer stores from the kernel), the index buffer --
            # heightmap-independent, closed form -- is generated by rank 0 locally while the bands arrive
            local_sum = checksum(vtx.data_ptr(), vtx.numel()) & 0x7FFFFFFFFFFFFFFF
            del idx
            torch.cuda.empty_cache()
            gv = shared_buffer(n * n * STRIDE)
            gidx = torch.empty(6 * (n - 1) ** 2, dtype=torch.int32, device=dev) if rank == 0 else None
            if rank == 0:
                job_g = T.job(height, n, rows=(r0, r1), qrows=(0, n - 1), height_row0=lo, height_rows=hi - lo,
                              vtx_out=gv.value, vtx_row0=0, idx_out=gidx, idx_qrow0=0)
            else:
                job_g = T.job(height, n, rows=(r0, r1), qrows=(0, 0), height_row0=lo, height_rows=hi - lo,
                              vtx_out=gv.value, vtx_row0=0)
            ms_g = timed(lambda: T.build(job_g), reps=3, warm=1)
            import torch.distributed as dist

            sums = torch.tensor([local_sum], dtype=torch.int64, device=dev)
            allsums = [torch.zeros_like(sums) for _ in range(world)]
            dist.all_gather(allsums, sums)
            ok = True
            if rank == 0:
                rows_p = (C.c_uint32 * (world + 1))()
                lib.mr_terrain_partition(n, world, rows_p, None)
                for g in range(world):
                    a_, z_ = rows_p[g] * n * STRIDE, rows_p[g + 1] * n * STRIDE
                    ok = ok and (checksum(gv.value + a_, z_ - a_) & 0x7FFFFFFFFFFFFFFF) == int(allsums[g].item())
            nv = n * n * STRIDE * (world - 1) / world
            res.update({"gather_ms": ms_g, "gather_gverts_per_s": n * n / (ms_g * 1e-3) / 1e9,
                        "nvlink_bytes_into_rank0": int(nv), "rank0_ingest_gb_per_s": nv / (ms_g * 1e-3) / 1e9,
                        "gather_ok": bool(ok),
                        "gather_note": "vertex bands peer-stored into rank 0; all 6.4 GB of indices generated on rank 0"})
            del gidx
            release(gv)
        except Exception as exc:
            res["gather_error"] = str(exc)[:200]
    return res


def run_config5(ctx, P, dev, rank, world, timed, shared_buffer, release, want_gather, reduce_sum):
    """BASELINE configs[4]: 1M polygons, sizes log-uniform 8..1024, strong-scaled cost-balanced ranges."""
    import torch

    import myrenderer_b200 as mr
    from myrenderer_b200 import sharding

    lib = ctx.lib
    npoly = CFG5_NPOLY
    fp_all = np.zeros(npoly + 1, dtype=np.uint64)
    lib.mr_synth_polygon_sizes(CFG5_SEED, 0, npoly, 8, 1024, 1, fp_all.ctypes.data)
    ft_all = mr.polygon_offsets_host(fp_all)
    ps = sharding.plan_polygons(fp_all, ft_all, rank, world)
    fp = np.ascontiguousarray(fp_all[ps.begin:ps.end + 1])
    ft_glob = np.ascontiguousarray(ft_all[ps.begin:ps.end + 1])
    ft_loc = ft_glob - ft_glob[0]
    cnt = ps.end - ps.begin
    fp_d = torch.from_numpy(fp.view(np.int64)).to(dev)
    ftl_d = torch.from_numpy(ft_loc.view(np.int64)).to(dev)
    ftg_d = torch.from_numpy(ft_glob.view(np.int64)).to(dev)
    xy = torch.empty(int(fp[-1] - fp[0]) * 2, dtype=torch.float32, device=dev)
    pv = torch.empty(int(ft_loc[-1]) * 96, dtype=torch.uint8, device=dev)
    st = torch.empty(cnt, dtype=torch.int32, device=dev)
    points = int(fp_all[-1])
    res = {"what": "1,000,000 polygons, sizes log-uniform 8..1024, strong-scaled cost-balanced contiguous ranges",
           "points": points, "algorithmic_bytes": int(8 * points + 8 * npoly + 96 * int(ft_all[-1]))}
    gp = None
    for name, fam in (("ellipse", FAMILY_ELLIPSE), ("zipper", FAMILY_ZIPPER)):
        ctx.check(lib.mr_synth_polygons_family(ctx.handle, fam, CFG5_SEED, ps.begin, fp_d.data_ptr(), cnt, xy.data_ptr()), "synth")
        job = P.job(xy, fp_d, cnt, vtx_out=pv, first_tri=ftl_d, status_out=st, seed=CFG5_SEED, poly_index0=ps.begin,
                    point_base=int(fp[0]))
        ms = timed(lambda: P.triangulate(job), reps=2, warm=1)
        ok = int(reduce_sum(int((st == 0).sum().item())))
        r = {"compute_ms": ms, "polygons_per_s": npoly / (ms * 1e-3), "mpoints_per_s": points / (ms * 1e-3) / 1e6,
             "achieved_gb_per_s_aggregate": res["algorithmic_bytes"] / (ms * 1e-3) / 1e9, "status_ok": ok}
        if world > 1 and want_gather:
            try:
                if gp is None:
                    gp = shared_buffer(int(ft_all[-1]) * 96)
                jg = P.job(xy, fp_d, cnt, vtx_out=gp.value, first_tri=ftg_d, tri_base=0, status_out=st, seed=CFG5_SEED,
                           poly_index0=ps.begin, point_base=int(fp[0]))
                msg = timed(lambda: P.triangulate(jg), reps=2, warm=1)
                r.update({"gather_ms": msg, "gather_polygons_per_s": npoly / (msg * 1e-3),
                          "nvlink_bytes_into_rank0": int(int(ft_all[-1]) * 96 * (world - 1) / world)})
            except Exception as exc:
                r["gather_error"] = str(exc)[:200]
        res[name] = r
    if gp is not None:
        release(gp)
    res["note"] = ("ellipse = convex; zipper = non-convex y-monotone family on which the reference is sound for every edge order "
                   "(tests/test_reference_soundness_cpu.py); every polygon of both ends with status OK")
    return res


if __name__ == "__main__":
    main()
