"""CPU tests of the host-side mirror of the reference interface (no GPU work)."""
import numpy as np


def test_vertex_layout_create():
    import myrenderer_b200 as mr

    # VertexLayout.create(GPUVertex) -- Polygon.zig:26-29 with Vec2 = 8 B, Vec3 = 16 B @Vector
    decl = mr.VertexLayout.create(mr.GPUVertex, "decl")
    assert decl.stride == 32 and decl.attributes == ((0, 2), (16, 3))
    auto = mr.VertexLayout.create(mr.GPUVertex, "zigauto")
    assert auto.stride == 32 and auto.attributes == ((16, 2), (0, 3))
    t = mr.VertexLayout.create(mr.TerrainVertex)
    assert t.stride == 32 and t.attributes == ((0, 3), (16, 3))
    n = t.native
    assert (n.stride, n.nattr, n.attr[1].offset, n.attr[1].location) == (32, 2, 16, 1)
    v4 = mr.VertexLayout.create((("a", "Vec2"), ("b", "Vec2"), ("c", "Vec4")))
    assert v4.stride == 32 and v4.attributes == ((0, 2), (8, 2), (16, 4))


def test_vertex_buffer_descriptor():
    import myrenderer_b200 as mr

    vb = mr.VertexBuffer.new(4, 5, None)  # VertexBuffer.new(renderer, offset, primitive_count, void)
    assert (vb.vertex_count, vb.instance_count, vb.first_vertex, vb.first_instance) == (15, 1, 12, 0)
    assert vb.vertex_buffer is None


def test_unirand_mirror(oracle):
    import myrenderer_b200 as mr

    for top in (2, 7, 36, 64, 1000):
        r = mr.unirand_seed(top, 77, 5)
        assert (r.offset, r.prime) == oracle.unirand_seed(top, 77, 5)
        seq = []
        while True:
            v = r.next()
            if v is None:
                break
            seq.append(v)
        assert seq == oracle.unirand_sequence(top, r.offset, r.prime)
    assert mr.Unirand(0, 3, 1).next() is None  # unirand.zig:15: top == 0 yields null at once


def test_polygon_offsets_host(oracle):
    import myrenderer_b200 as mr

    fp = np.array([0, 0, 1, 3, 6, 10, 74], dtype=np.uint64)
    assert mr.polygon_offsets_host(fp).tolist() == [0, 0, 0, 0, 1, 3, 65]
    assert np.array_equal(mr.polygon_offsets_host(fp), oracle.polygon_offsets(fp))


def test_png_loader_matches_fixture():
    """The reference's HEIGHTMAP.png pixels, stored as a 16-bit grayscale PNG (tests/golden/make_golden.py), decode
    to the u16 array the reference's own PNG decoded to."""
    import os

    import myrenderer_b200 as mr

    golden = os.path.join(os.path.dirname(__file__), "golden")
    h = mr.load_heightmap_png(os.path.join(golden, "heightmap_100.png"))
    want = np.load(os.path.join(golden, "heightmap_100.npy"))
    assert h.dtype == np.uint16 and np.array_equal(h, want)


def test_roofline_traffic_evidence_is_not_stale():
    """bench.py reports `roofline.traffic` from profiles/r03_traffic.json only while that capture belongs to the
    committed terrain.cu (sha256 stored beside it); this keeps the two from drifting apart unnoticed."""
    import bench

    traffic, src = bench.fresh_traffic()
    assert traffic is not None and 0.5 * 570425344 < traffic < 1.5 * 570425344, "re-capture the vertex kernel: terrain.cu changed"
