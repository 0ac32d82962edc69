"""The polygon kernels at float edges, against the CPU oracle: every case of the kill set of tests/_poly_float_edges.py
(signed zeros, subnormal and overflowing side tests, near-collinear triples, atan2 differences within an ulp of pi, bbox
ties at zero) and the non-finite set (NaN / inf in x only or y only, at the first, a middle and the last point, and finite
+-FLT_MAX polygons), through every path: device batches by size class in three vertex layouts, single host-memory polygons
(the small-batch path) and a mixed host batch.  Status, triangle count, vertex bytes and bbox bits must equal the oracle's.
tests/test_poly_float_edges_cpu.py shows that these cases tell each mutant of the float rules apart from the reference."""
import ctypes as C

import numpy as np
import pytest

import _poly_float_edges as E

pytestmark = pytest.mark.gpu

LAYOUTS = {"decl": None, "zigauto": None, "generic": (40, ((4, 2), (20, 3)))}


def _layout(mr, name):
    if LAYOUTS[name] is None:
        return mr.VertexLayout.create(mr.GPUVertex, name)
    return mr.VertexLayout(*LAYOUTS[name])


def _tier_counts(ctx):
    tc = (C.c_uint32 * 8)()
    ctx.check(ctx.lib.mr_triangulate_tier_counts(ctx.handle, tc), "tier counts")
    return list(tc)


def _compare(what, gs, gn, gv, gb, ref, stride, fp):
    bad = np.nonzero(gs != ref["status"])[0]
    assert bad.size == 0, (what, "status", bad[:5].tolist(), gs[bad[:5]].tolist(), ref["status"][bad[:5]].tolist())
    assert np.array_equal(gn, ref["ntri"]), (what, "ntri", np.nonzero(gn != ref["ntri"])[0][:5].tolist())
    if not np.array_equal(gv, ref["vtx"]):
        ft, per = ref["first_tri"], 3 * stride
        for i in range(len(fp) - 1):
            a, z = int(ft[i]) * per, int(ft[i + 1]) * per
            assert np.array_equal(gv[a:z], ref["vtx"][a:z]), (what, "vertex bytes of polygon", i, int(fp[i + 1] - fp[i]))
    bad = np.nonzero((gb.view(np.uint32) != ref["bbox"].view(np.uint32)).any(1))[0]
    assert bad.size == 0, (what, "bbox bits", bad[:5].tolist(), gb[bad[:5]].tolist(), ref["bbox"][bad[:5]].tolist())


def _device_batch(ctx, oracle, mr, xy, fp, op, layout_name, what):
    lay = _layout(mr, layout_name)
    b = mr.Polygon(ctx, lay).create_polygons(xy, fp, offset_prime=op)
    ctx.sync()
    with np.errstate(all="ignore"):
        ref = oracle.polygon_batch(xy, fp, offset_prime=op, layout=(lay.stride, lay.attributes), nthreads=0)
    _compare((what, layout_name), b.status.cpu().numpy().view(np.uint32), b.ntri.cpu().numpy().view(np.uint32),
             b.vertex_buffer.cpu().numpy(), b.bbox.cpu().numpy(), ref, lay.stride, fp)
    return ref


def _host_call(ctx, oracle, mr, xy, fp, op):
    P = mr.Polygon(ctx)
    with np.errstate(all="ignore"):
        ref = oracle.polygon_batch(xy, fp, offset_prime=op, nthreads=0)
    ft = ref["first_tri"]
    npoly = len(fp) - 1
    vtx = np.full(max(int(ft[-1]) * 96, 1), 0xEE, dtype=np.uint8)
    st = np.full(npoly, 77, dtype=np.uint32)
    nt = np.zeros(npoly, dtype=np.uint32)
    bbox = np.full((npoly, 4), np.nan, dtype=np.float32)
    opf = np.ascontiguousarray(op, dtype=np.uint32).reshape(-1)
    xy = np.ascontiguousarray(xy, dtype=np.float32)
    P.triangulate(P.job(xy, fp, npoly, vtx_out=vtx, first_tri=ft, bbox_out=bbox, status_out=st, ntri_out=nt, offset_prime=opf))
    return st, nt, vtx[: int(ft[-1]) * 96], bbox, ref


def _sets(oracle):
    cs, _ = E.kill_cases(oracle)
    nf, _, _ = E.nonfinite_cases(oracle)
    return (("kill", cs), ("nonfinite", nf))


def test_device_batches_by_class_every_layout(ctx, oracle):
    import myrenderer_b200 as mr

    for set_name, cs in _sets(oracle):
        for cname, _, _ in E.CLASSES:
            idx = [i for i, c in enumerate(cs.classes) if c == cname]
            xy, fp, op = cs.packed(idx)
            for lay in LAYOUTS:
                _device_batch(ctx, oracle, mr, xy, fp, op, lay, (set_name, cname))
        # and all classes in one batch, so that the classes share a launch
        _device_batch(ctx, oracle, mr, *cs.packed(), "decl", (set_name, "all"))


def test_single_polygon_host_calls(ctx, oracle):
    """Polygon.create_polygon's call shape: one polygon, every buffer in host memory (mr_triangulate_small)."""
    import myrenderer_b200 as mr

    for set_name, cs in _sets(oracle):
        for i in range(len(cs)):
            xy, fp, op = cs.packed([i])
            st, nt, vtx, bbox, ref = _host_call(ctx, oracle, mr, xy, fp, op)
            _compare((set_name, i, cs.fams[i], len(cs.polys[i])), st, nt, vtx, bbox, ref, 32, fp)


def test_mixed_small_host_batch(ctx, oracle):
    import myrenderer_b200 as mr

    rng = np.random.default_rng(5)
    for set_name, cs in _sets(oracle):
        small = [i for i, p in enumerate(cs.polys) if len(p) <= 1024]
        for _ in range(3):
            idx = sorted(rng.choice(small, size=min(24, len(small)), replace=False).tolist())
            big = [i for i, p in enumerate(cs.polys) if len(p) > 1024]
            idx += [int(rng.choice(big))]
            xy, fp, op = cs.packed(idx)
            st, nt, vtx, bbox, ref = _host_call(ctx, oracle, mr, xy, fp, op)
            _compare((set_name, "mixed"), st, nt, vtx, bbox, ref, 32, fp)


def test_signed_zero_routing(ctx, oracle):
    """A -0 / +0 twin is coincident in the (y, x) order and goes to the general path; a -0 / +0 tie in y between points
    of distinct x is an ordinary order decision and stays on the fast path -- exact either way."""
    import myrenderer_b200 as mr

    twin = np.array([[0.0, 0.0], [10.0, -0.0], [10.0, 10.0], [-0.0, 10.0], [0.0, 5.0], [-0.0, 0.0]], dtype=np.float32)
    ties = np.array([[0.0, 0.0], [10.0, -0.0], [10.0, 10.0], [5.0, 12.0], [-0.0, 10.0], [-3.0, -0.0]], dtype=np.float32)
    for p, general in ((twin, 1), (ties, 0)):
        xy, fp = E.pack([p])
        for op in ([0, 1], [2, 5], oracle.unirand_seed(len(p), 9, 0)):
            op = np.array([op], dtype=np.uint32)
            _device_batch(ctx, oracle, mr, xy, fp, op, "decl", ("routing", general))
            tc = _tier_counts(ctx)
            assert tc[6] == general and sum(tc[0:6]) == 0 and tc[7] == 0, (general, tc)


def test_nonfinite_above_3072_points_reach_the_general_path_check(ctx, oracle):
    import myrenderer_b200 as mr

    nf, flagged, desc = E.nonfinite_cases(oracle)
    idx = [i for i, d in enumerate(desc) if d[0] == "gt3072"]
    assert len(idx) >= 6 and flagged[idx].any()
    xy, fp, op = nf.packed(idx)
    ref = _device_batch(ctx, oracle, mr, xy, fp, op, "decl", "gt3072")
    assert _tier_counts(ctx)[7] == len(idx)
    assert np.array_equal(ref["status"] == 2, flagged[idx])
