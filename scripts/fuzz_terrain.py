"""Terrain fuzz: mr_terrain_build / mr_terrain_tile_bounds / mr_terrain_cull through the C ABI vs the CPU oracle, byte
for byte, on drawn cases -- sizes 1..1600 (odd, even, multiples of 8 and of 256), u16 and f32 heights (noise, constant,
extremes, steps, maps of NaN / +-inf / +-0 / subnormal / +-FLT_MAX texels), terrain parameters (the reference's
constants, other grid steps, negative and zero scales), vertex layouts (strides 12..64, position / normal at any 4-byte
offset, with and without a normal), row bands written into larger buffers, device and host pointers, tilings, cull
matrices, and the near-threshold and non-finite cull boxes of tests/_float_edges.py.  Any two NaN floats compare equal
(the header leaves a NaN's sign and payload unspecified); every other word, padding included, must be bit-equal.  Test
infrastructure: the oracle is the checker.

    python scripts/fuzz_terrain.py --rounds 300 --seed 1 --out gpurun_out/fuzz_terrain.json     # on a GPU box

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
import _float_edges as E  # noqa: E402


def draw_n(rng):
    k = int(rng.integers(0, 6))
    if k == 0:
        return int(rng.integers(1, 12))
    if k == 1:
        return int(rng.integers(12, 300))
    if k == 2:
        return 8 * int(rng.integers(2, 160))
    if k == 3:
        return 256 * int(rng.integers(1, 6)) + int(rng.integers(-1, 2))
    if k == 4:
        return int(rng.integers(300, 1600))
    return int(rng.choice([2, 3, 255, 256, 257, 511, 512, 513, 1024]))


def draw_height(rng, orc, n):
    k = int(rng.integers(0, 8))
    if k == 7:
        return E.special_heightmap(rng, n, ((int(rng.choice([1, 8, 33])), int(rng.choice([2, 24, 600]))),))
    if k <= 2:
        return orc.synth_heightmap_u16(int(rng.integers(1, 2 ** 62)), n)
    if k == 3:
        return rng.choice(np.array([0, 1, 32767, 65534, 65535], dtype=np.uint16), size=(n, n))
    if k == 4:
        return rng.uniform(-3.0, 3.0, size=(n, n)).astype(np.float32)
    if k == 5:  # steps and ridges: large gradients, long flat runs (zero gradients)
        a = np.zeros((n, n), dtype=np.float32)
        a[:, n // 2:] = np.float32(rng.uniform(-100, 100))
        a[n // 3: n // 3 + 1, :] += np.float32(1e6)
        return a
    return orc.heightmap_normalize(orc.synth_heightmap_u16(int(rng.integers(1, 2 ** 62)), n))


def draw_params(rng):
    k = int(rng.integers(0, 6))
    if k <= 2:
        return (0.2, 0.1, 5.0)
    if k == 3:
        return (float(np.float32(rng.choice([0.4, 0.25, 1.0, 0.3, 3.0]))), float(np.float32(rng.uniform(0, 1))), float(np.float32(rng.uniform(-9, 9))))
    if k == 4:
        return (0.2, 0.1, 0.0)
    return (float(np.float32(rng.uniform(0.01, 5))), float(np.float32(rng.uniform(-1, 1))), float(np.float32(rng.uniform(-50, 50))))


def draw_layout(rng):
    k = int(rng.integers(0, 5))
    if k <= 1:
        return (32, ((0, 3), (16, 3)))
    if k == 2:
        return (32, ((16, 3), (0, 3)))
    if k == 3:  # position only
        stride = 4 * int(rng.integers(3, 10))
        return (stride, ((4 * int(rng.integers(0, stride // 4 - 2)), 3),))
    stride = 4 * int(rng.integers(6, 17))
    slots = stride // 4
    for _ in range(100):
        a, b = int(rng.integers(0, slots - 2)), int(rng.integers(0, slots - 2))
        ca, cb = int(rng.choice([3, 4])), int(rng.choice([3, 4]))
        if a + ca <= b or b + cb <= a:
            if a + ca <= slots and b + cb <= slots:
                return (stride, ((4 * a, ca), (4 * b, cb)))
    return (32, ((0, 3), (16, 3)))


def run_build(ctx, t, torch, hs, n, host, rb, re, qb, qe, hlo, hhi, v0, q0, vbytes, icount):
    """host: {"height"|"vtx"|"idx": "dev"|"host"|"pinned"} -- every buffer placed on its own."""
    def place(x, where):
        if where == "host":
            return x
        v = x.view(np.int16) if x.dtype == np.uint16 else x.view(np.int32) if x.dtype == np.uint32 else x
        if where == "pinned":
            tt = torch.empty(v.shape, dtype=torch.from_numpy(v).dtype, pin_memory=True)
            tt.copy_(torch.from_numpy(v))
            return tt
        return torch.from_numpy(v).cuda()
    hd = place(hs, host["height"])
    gv = place(np.full(max(vbytes, 1), 0xA5, dtype=np.uint8), host["vtx"])
    gi = place(np.full(max(icount, 2), 0xA5A5A5A5, dtype=np.uint32), host["idx"])
    j = t.job(hd, n, rows=(rb, re), qrows=(qb, qe), height_row0=hlo, height_rows=hhi - hlo, vtx_out=gv if vbytes else None,
              vtx_row0=v0, idx_out=gi if icount else None, idx_qrow0=q0)
    j.height_fmt = 0 if hs.dtype == np.uint16 else 1
    t.build(j)
    ctx.sync()
    back = lambda x: x if isinstance(x, np.ndarray) else x.cpu().numpy()
    return back(gv), back(gi).view(np.uint32)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=100)
    ap.add_argument("--seed", type=int, default=1)
    ap.add_argument("--out", default=os.path.join(ROOT, "gpurun_out", "fuzz_terrain.json"))
    ap.add_argument("--budget-s", type=float, default=300.0)
    a = ap.parse_args()
    import torch
    import oracle as orc
    import myrenderer_b200 as mr
    from test_terrain_cull_cpu import camera_matrix, mat_image

    edge_cases = E.cull_cases(seed=a.seed)
    ctx = mr.Context(0)
    lib = ctx.lib
    rng = np.random.default_rng(a.seed)
    log = open(a.out + ".log", "a")
    t0 = time.time()
    failures, cases = [], 0
    totals = {"vertices": 0, "indices": 0, "tiles": 0, "cull_calls": 0}

    def fail(desc, what):
        d = dict(desc)
        d["mismatch"] = what
        failures.append(d)
        log.write("FAIL  " + json.dumps(d) + "\n")
        log.flush()

    for r in range(a.rounds):
        if time.time() - t0 > a.budget_s:
            break
        n = draw_n(rng)
        h = draw_height(rng, orc, n)
        params = draw_params(rng)
        lay_t = draw_layout(rng)
        lay = mr.VertexLayout(lay_t[0], lay_t[1])
        k = int(rng.integers(0, 4))
        host = ({x: "dev" for x in ("height", "vtx", "idx")} if k == 0 else {x: "host" for x in ("height", "vtx", "idx")} if k == 1
                else {x: str(rng.choice(["dev", "host", "pinned"])) for x in ("height", "vtx", "idx")})
        # a band of rows / quad rows written into a buffer that starts at an earlier row
        if n > 2 and rng.integers(0, 2):
            rb = int(rng.integers(0, n))
            re = int(rng.integers(rb, n + 1))
            qb = int(rng.integers(0, n - 1))
            qe = int(rng.integers(qb, n))
        else:
            rb, re, qb, qe = 0, n, 0, max(n - 1, 0)
        v0 = int(rng.integers(0, rb + 1))
        q0 = int(rng.integers(0, qb + 1))
        # the heightmap slice the job is given: the band plus its halo, sometimes more
        hlo = max(rb - 1, 0) if re > rb else 0
        hhi = min(re + 1, n) if re > rb else n
        if rng.integers(0, 2):
            hlo, hhi = int(rng.integers(0, hlo + 1)), int(rng.integers(hhi, n + 1))
        desc = {"round": r, "n": n, "dtype": str(h.dtype), "params": params, "layout": lay_t, "host": host, "rows": [rb, re], "qrows": [qb, qe],
                "vtx_row0": v0, "idx_qrow0": q0, "height_rows": [hlo, hhi]}
        log.write("start " + json.dumps(desc) + "\n")
        log.flush()
        cases += 1
        stride = lay_t[0]
        vbytes = (re - v0) * n * stride
        icount = (qe - q0) * 6 * max(n - 1, 0)
        ovtx, oidx = orc.terrain_build(h, n, layout=lay_t, params=params, rows=(rb, re), qrows=(qb, qe), nthreads=0)
        want_v = np.full(max(vbytes, 1), 0xA5, dtype=np.uint8)
        want_v[(rb - v0) * n * stride: (re - v0) * n * stride] = ovtx
        want_i = np.full(max(icount, 2), 0xA5A5A5A5, dtype=np.uint32)
        want_i[(qb - q0) * 6 * max(n - 1, 0): (qe - q0) * 6 * max(n - 1, 0)] = oidx
        hs = np.ascontiguousarray(h[hlo:hhi])
        t = mr.Terrain(ctx, lay, params)
        try:
            gv, gi = run_build(ctx, t, torch, hs, n, host, rb, re, qb, qe, hlo, hhi, v0, q0, vbytes, icount)
        except Exception as e:  # an error code for a job this script believes valid is a finding too
            fail(desc, "build raised " + repr(e))
            continue
        if not np.array_equal(gi, want_i):
            fail(desc, "index buffer (or the words around the band) differs")
        if (E.float_mismatch(gv, want_v, E.vertex_float_mask(vbytes, lay_t)) is not None if vbytes
                else not np.array_equal(gv, want_v)):
            fail(desc, "vertex bytes (or the bytes around the band) differ")
        totals["vertices"] += (re - rb) * n
        totals["indices"] += oidx.size
        # tiles and culling on the same heightmap
        if n >= 2 and r % 2 == 0:
            tr = int(rng.choice([1, 3, 8, 16, 33, 64, 100, 4096]))
            tc = int(rng.choice([1, 2, 8, 16, 24, 64, 256, 500, 4096]))
            want_box = orc.terrain_tile_bounds(h, n, tr, tc, params)
            ntiles = want_box.shape[0]
            hd = torch.from_numpy(h.view(np.int16) if h.dtype == np.uint16 else h).cuda()
            box_d = torch.empty(ntiles * 8, dtype=torch.float32, device="cuda")
            ctx.check(lib.mr_terrain_tile_bounds(ctx.handle, hd.data_ptr(), 0 if h.dtype == np.uint16 else 1, n, tr, tc, C.byref(t.params),
                                                 box_d.data_ptr()), "tile bounds")
            ctx.sync()
            if E.float_mismatch(box_d.cpu().numpy(), want_box) is not None:
                fail(dict(desc, tile=[tr, tc]), "tile boxes differ")
            totals["tiles"] += ntiles
            for _ in range(2):
                k = int(rng.integers(0, 5))
                boxes = want_box  # the cull is checked on the oracle's boxes
                if k == 0:
                    m = camera_matrix()
                elif k == 1:
                    eye = tuple(float(x) for x in rng.uniform(-80, 80, 3))
                    m = camera_matrix(eye, tuple(float(x) for x in rng.uniform(-40, 40, 3)))
                elif k == 2:
                    m = rng.uniform(-1, 1, 16).astype(np.float32)
                elif k == 3:
                    m = mat_image(np.array([[0, 0, 0, 1]] * 4, dtype=np.float32))
                else:  # boxes near the thresholds of the test, or with +-inf / NaN components, under their matrix
                    _, m, pool = edge_cases[int(rng.integers(0, len(edge_cases)))]
                    boxes = pool[rng.integers(0, len(pool), ntiles)]
                box_d = torch.from_numpy(np.ascontiguousarray(boxes).reshape(-1)).cuda()
                ref = orc.terrain_cull(boxes, n, tr, tc, m)
                vis = torch.empty(ntiles, dtype=torch.int32, device="cuda")
                ids = torch.empty(ntiles, dtype=torch.int32, device="cuda")
                idx = torch.full((6 * (n - 1) * (n - 1),), -1, dtype=torch.int32, device="cuda")
                cnt = torch.zeros(2, dtype=torch.int64, device="cuda")
                ctx.check(lib.mr_terrain_cull(ctx.handle, box_d.data_ptr(), n, tr, tc, m.ctypes.data, vis.data_ptr(), ids.data_ptr(),
                                              idx.data_ptr(), cnt.data_ptr()), "cull")
                ctx.sync()
                c = cnt.cpu().numpy()
                g = idx.cpu().numpy().view(np.uint32)
                if (c.tolist() != ref["counts"].tolist() or not np.array_equal(vis.cpu().numpy().view(np.uint32), ref["visible"])
                        or not np.array_equal(ids.cpu().numpy().view(np.uint32)[: c[0]], ref["ids"])
                        or not np.array_equal(g[: c[1]], ref["idx"]) or not (g[c[1]:] == 0xFFFFFFFF).all()):
                    fail(dict(desc, tile=[tr, tc], matrix=m.tolist()), "cull outputs differ")
                totals["cull_calls"] += 1
        log.write("done  %d\n" % r)
        log.flush()
    out = {"seed": a.seed, "cases": cases, "mismatches": len(failures), "totals": totals, "seconds": round(time.time() - t0, 1),
           "failures": failures[:50], "command": "python scripts/fuzz_terrain.py --rounds %d --seed %d" % (a.rounds, a.seed)}
    json.dump(out, open(a.out, "w"), indent=1)
    print(json.dumps({k: out[k] for k in ("seed", "cases", "mismatches", "totals", "seconds")}))
    sys.exit(1 if failures else 0)


if __name__ == "__main__":
    main()
