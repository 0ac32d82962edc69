"""Host-side mirror of the reference's interface for the geometry hot path.

Names, argument meaning and error behaviour follow the Zig modules so the parity tests read like
tests of the reference:

    VertexLayout.create        Renderer/VertexLayout.zig:9-31
    VertexBuffer.new/.map      Renderer/VertexBuffer.zig:11-35
    Terrain.create_terrain     Terrain/Terrain.zig:88-129
    Polygon.create_polygon     Polygon/Polygon.zig:81-107
    Triangulation.create_polygon(points, ctx, emit)   Polygon/Triangulation.zig:446-451
    unirand_seed / Unirand.next   Polygon/unirand.zig:12-50

Everything computes through the C ABI of libmyrenderer_b200.so (include/myrenderer_b200.h).
torch is used only to own device memory and streams.  There is no CPU fallback: constructing a
`Context` without a CUDA device raises `MrError`.
"""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass, field
from typing import Callable, Optional, Sequence

import numpy as np

from . import _capi as capi
from ._capi import (MrDrawIndexedRange, MrError, MrLayout, MrPolygonIndices, MrPolygonJob, MrPolygonRings, MrTerrainJob,
                    MrTerrainParams)

try:  # torch is plumbing (device memory, streams); numpy host arrays work without it
    import torch
except Exception:  # pragma: no cover
    torch = None


# ----------------------------------------------------------------------------------------------
def _ptr(x) -> Optional[int]:
    """Address of a numpy array / torch tensor / int / None."""
    if x is None:
        return None
    if isinstance(x, int):
        return x
    if isinstance(x, np.ndarray):
        if not x.flags["C_CONTIGUOUS"]:
            raise ValueError("array must be C-contiguous")
        return x.ctypes.data
    if torch is not None and isinstance(x, torch.Tensor):
        if not x.is_contiguous():
            raise ValueError("tensor must be contiguous")
        return x.data_ptr()
    raise TypeError(f"unsupported buffer type {type(x)}")


def _is_cuda(x) -> bool:
    return torch is not None and isinstance(x, torch.Tensor) and x.is_cuda


class Context:
    """Owns an mr_context (stream + device scratch): the analogue of Triangulation.new/destroy."""

    def __init__(self, device: int = 0, use_torch_stream: bool = True):
        self.lib = capi.load()
        h = C.c_void_p()
        rc = self.lib.mr_context_create(device, C.byref(h))
        if rc != 0:
            raise MrError(rc, "mr_context_create", "no usable CUDA device (there is no CPU fallback)")
        self.handle = h
        self.device = device
        if use_torch_stream and torch is not None and torch.cuda.is_available():
            self.set_stream(torch.cuda.current_stream(device).cuda_stream)

    def check(self, rc: int, where: str):
        if rc != 0:
            raise MrError(rc, where, self.lib.mr_last_error(self.handle).decode())

    def set_stream(self, cuda_stream: int):
        self.check(self.lib.mr_context_set_stream(self.handle, C.c_void_p(cuda_stream)), "mr_context_set_stream")

    def sync(self):
        self.check(self.lib.mr_sync(self.handle), "mr_sync")

    @property
    def launch_count(self) -> int:
        return int(self.lib.mr_launch_count(self.handle))

    def close(self):
        if getattr(self, "handle", None):
            self.lib.mr_context_destroy(self.handle)
            self.handle = None

    def __del__(self):  # pragma: no cover
        try:
            self.close()
        except Exception:
            pass


# ---- VertexLayout / VertexBuffer -------------------------------------------------------------
_VEC = {"Vec2": (8, 8, 2), "Vec3": (16, 16, 3), "Vec4": (16, 16, 4)}  # size, align, components


@dataclass(frozen=True)
class VertexLayout:
    """VertexLayout.create(T): array_stride=@sizeOf(T), attribute i = {@offsetOf, format, location i}.

    `order` selects how field offsets are derived, because Zig may reorder a non-extern struct:
      "decl"    fields laid out in declaration order (what an `extern struct` would give)
      "zigauto" fields sorted by descending alignment (what the Zig compiler does today)
    A Zig caller passes the real @offsetOf values instead (see INTEGRATION.md)."""

    stride: int
    attributes: tuple  # ((offset, ncomp), ...) in field (shader_location) order

    @staticmethod
    def create(fields: Sequence[tuple], order: str = "decl") -> "VertexLayout":
        idx = list(range(len(fields)))
        if order == "zigauto":
            idx.sort(key=lambda i: -_VEC[fields[i][1]][1])
        elif order != "decl":
            raise ValueError(order)
        off, offsets, max_align = 0, {}, 1
        for i in idx:
            size, align, _ = _VEC[fields[i][1]]
            off = (off + align - 1) // align * align
            offsets[i] = off
            off += size
            max_align = max(max_align, align)
        stride = (off + max_align - 1) // max_align * max_align
        return VertexLayout(stride, tuple((offsets[i], _VEC[f[1]][2]) for i, f in enumerate(fields)))

    @property
    def native(self) -> MrLayout:
        L = MrLayout()
        L.stride = self.stride
        L.nattr = len(self.attributes)
        for i, (off, ncomp) in enumerate(self.attributes):
            L.attr[i].offset, L.attr[i].ncomp, L.attr[i].location = off, ncomp, i
        return L


GPUVertex = (("x", "Vec2"), ("color", "Vec3"))          # Polygon.zig:26-29
TerrainVertex = (("pos", "Vec3"), ("normal", "Vec3"))   # new type, SURVEY 8-a4


@dataclass
class VertexBuffer:
    """Mirror of Renderer/VertexBuffer.zig: a draw descriptor plus the (device) buffer."""

    vertex_buffer: object = None
    vertex_count: int = 3
    instance_count: int = 1
    first_vertex: int = 0
    first_instance: int = 0

    @staticmethod
    def new(offset: int, primitive_count: int, layout: Optional[VertexLayout], device="cuda") -> "VertexBuffer":
        # VertexBuffer.zig:11-31: size = primitive_count * @sizeOf(T) * 3, mapped at creation (zeroed)
        buf = None
        if layout is not None:
            buf = torch.zeros(max(primitive_count * layout.stride * 3, 1), dtype=torch.uint8, device=device)
        return VertexBuffer(buf, primitive_count * 3, 1, offset * 3, 0)

    def map(self) -> np.ndarray:
        """getMappedRange: the whole buffer as host bytes."""
        return self.vertex_buffer.cpu().numpy()


# ---- unirand ----------------------------------------------------------------------------------
class Unirand:
    """Polygon/unirand.zig:6-22."""

    def __init__(self, top: int, offset: int, prime: int):
        self.at, self.top, self.offset, self.prime = 0, top, offset, prime

    def next(self) -> Optional[int]:
        result = None
        if self.top > 0 and self.at < self.top:
            result = ((self.at * self.prime + self.offset) & 0xFFFFFFFF) % self.top
        self.at += 1
        return result


def unirand_seed(top: int, seed: int, index: int = 0) -> Unirand:
    """unirand_seed (unirand.zig:26-50) with std.crypto.random replaced by the documented stream."""
    lib = capi.load()
    off, prime = C.c_uint32(), C.c_uint32()
    rc = lib.mr_unirand_seed_host(top, seed, index, C.byref(off), C.byref(prime))
    if rc != 0:
        raise MrError(rc, "mr_unirand_seed_host")
    return Unirand(top, off.value, prime.value)


# ---- Terrain ------------------------------------------------------------------------------------
@dataclass
class TerrainMesh:
    size: int
    vertex_buffer: VertexBuffer
    index_buffer: object            # u32 tensor, 6*(n-1)^2
    index_count: int
    bounding_box_p0: tuple
    bounding_box_p1: tuple
    layout: VertexLayout


def load_heightmap_png(filename: str) -> np.ndarray:
    """PNG -> u16[n][n] (Terrain.zig:89-95,116: square, grayscale16)."""
    from PIL import Image

    img = Image.open(filename)
    if img.mode not in ("I;16", "I;16B", "I"):
        raise ValueError(f"{filename}: expected 16-bit grayscale, got mode {img.mode}")
    a = np.asarray(img).astype(np.uint16)
    if a.ndim != 2 or a.shape[0] != a.shape[1]:
        raise ValueError("heightmap must be square")
    return np.ascontiguousarray(a)


class Terrain:
    """Mirror of the Terrain module.  create_terrain builds the indexed mesh on the GPU."""

    def __init__(self, ctx: Context, layout: Optional[VertexLayout] = None, params=(0.2, 0.1, 5.0)):
        self.ctx = ctx
        self.layout = layout or VertexLayout.create(TerrainVertex)
        self.params = MrTerrainParams(*params)

    def job(self, height, n, *, rows=None, qrows=None, height_row0=0, height_rows=None, vtx_out=None,
            vtx_row0=0, idx_out=None, idx_qrow0=0) -> MrTerrainJob:
        if isinstance(height, np.ndarray):
            fmt = capi.MR_HEIGHT_U16 if height.dtype == np.uint16 else capi.MR_HEIGHT_F32
            nelem = height.size
        else:
            fmt = capi.MR_HEIGHT_U16 if height.dtype in (torch.uint16, torch.int16) else capi.MR_HEIGHT_F32
            nelem = height.numel()
        if fmt == capi.MR_HEIGHT_F32 and str(height.dtype).split(".")[-1] != "float32":
            raise TypeError("heightmap must be uint16 or float32")
        j = MrTerrainJob()
        j.n, j.height_fmt, j.height = n, fmt, _ptr(height)
        j.height_row0 = height_row0
        j.height_rows = nelem // n if height_rows is None else height_rows
        j.row_begin, j.row_end = (0, n) if rows is None else rows
        j.qrow_begin, j.qrow_end = (0, max(n - 1, 0)) if qrows is None else qrows
        j.vtx_out, j.vtx_row0 = _ptr(vtx_out), vtx_row0
        j.idx_out, j.idx_qrow0 = _ptr(idx_out), idx_qrow0
        j.layout, j.params = self.layout.native, self.params
        return j

    def build(self, job: MrTerrainJob):
        self.ctx.check(self.ctx.lib.mr_terrain_build(self.ctx.handle, C.byref(job)), "mr_terrain_build")

    def create_terrain(self, heightmap, device="cuda") -> TerrainMesh:
        """heightmap: PNG filename (Terrain.zig:88), u16/f32 numpy array or torch tensor (n x n)."""
        if isinstance(heightmap, (str, bytes)):
            heightmap = load_heightmap_png(heightmap)
        n = int(heightmap.shape[1]) if heightmap.ndim == 2 else int(round(heightmap.numel() ** 0.5))
        if isinstance(heightmap, np.ndarray):
            heightmap = np.ascontiguousarray(heightmap)
        vb = VertexBuffer.new(0, 0, None)
        vtx = torch.empty(n * n * self.layout.stride, dtype=torch.uint8, device=device)
        idx = torch.empty(max(6 * (n - 1) * (n - 1), 1), dtype=torch.int32, device=device)
        self.build(self.job(heightmap, n, vtx_out=vtx, idx_out=idx if n > 1 else None))
        vb.vertex_buffer = vtx
        vb.vertex_count = n * n
        bmin, bmax = (C.c_float * 3)(), (C.c_float * 3)()
        vc, ic = C.c_uint64(), C.c_uint64()
        self.ctx.lib.mr_terrain_describe(n, C.byref(self.params), bmin, bmax, C.byref(vc), C.byref(ic))
        return TerrainMesh(n, vb, idx, int(ic.value), tuple(bmin), tuple(bmax), self.layout)


# ---- Polygon / Triangulation -------------------------------------------------------------------
@dataclass
class PolygonBatch:
    npoly: int
    first_point: np.ndarray         # host copy, npoly+1
    first_tri: np.ndarray           # host copy, npoly+1
    vertex_buffer: object           # device bytes, 3*first_tri[-1]*stride (None for output="indices")
    bbox: object                    # device f32 [npoly,4]
    status: object                  # device u32 [npoly]
    ntri: object                    # device u32 [npoly]
    layout: VertexLayout
    index_buffer: object = None     # device u32 [3*first_tri[-1]] (output="indices" / "both"): rows of xy
    index_base: int = 0             # first_point[0]: index k is row k of the xy the batch was made from

    def draw_range(self, i: int) -> VertexBuffer:
        """VertexBuffer.new(offset, primitive_count) for polygon i inside the packed buffer."""
        prims = int(self.first_tri[i + 1] - self.first_tri[i])
        return VertexBuffer(self.vertex_buffer, prims * 3, 1, int(self.first_tri[i]) * 3, 0)

    def draw_indexed_range(self, i: int) -> MrDrawIndexedRange:
        """drawIndexed's arguments for polygon i inside index_buffer (mr_polygon_draw_indexed_range)."""
        out = MrDrawIndexedRange()
        rc = capi.load().mr_polygon_draw_indexed_range(int(self.first_tri[i]), int(self.first_tri[i + 1]),
                                                       int(self.first_tri[0]), C.byref(out))
        if rc != 0:
            raise MrError(rc, "mr_polygon_draw_indexed_range")
        return out


@dataclass
class PolygonObj:
    vertex_buffer: VertexBuffer
    bounding_box_p0: tuple
    bounding_box_p1: tuple
    status: int
    ntri: int


def polygon_offsets_host(first_point: np.ndarray) -> np.ndarray:
    n = np.diff(first_point.astype(np.int64))
    ft = np.zeros(len(first_point), dtype=np.uint64)
    ft[1:] = np.cumsum(np.maximum(n - 2, 0))
    return ft


def polygon_offsets_rings_host(first_point: np.ndarray, first_ring: np.ndarray) -> np.ndarray:
    """first_tri of mr_polygon_offsets_rings: N + 2H - 2 triangles per polygon."""
    n = np.diff(first_point.astype(np.int64))
    r = np.diff(first_ring.astype(np.int64))
    h = np.where((r >= 1) & (r <= n), r - 1, 0)
    ft = np.zeros(len(first_point), dtype=np.uint64)
    ft[1:] = np.cumsum(np.maximum(n + 2 * h - 2, 0))
    return ft


_ALGORITHMS = {"reference": "mr_triangulate_batch", "earclip": "mr_triangulate_earclip"}
_OUTPUTS = ("vertices", "indices", "both")


def _check_algorithm(algorithm, offset_prime):
    if algorithm not in _ALGORITHMS:
        raise ValueError(f"algorithm must be one of {sorted(_ALGORITHMS)}, not {algorithm!r}")
    if algorithm == "earclip" and offset_prime is not None:
        raise ValueError("ear clipping has no edge order: offset_prime applies to the reference algorithm only")


class Polygon:
    """Mirror of the Polygon module (one reusable Triangulation inside: the Context's scratch)."""

    def __init__(self, ctx: Context, layout: Optional[VertexLayout] = None):
        self.ctx = ctx
        self.layout = layout or VertexLayout.create(GPUVertex)

    def job(self, xy, first_point, npoly, *, vtx_out, first_tri, bbox_out=None, status_out=None,
            ntri_out=None, offset_prime=None, seed=0, poly_index0=0, point_base=0, tri_base=0) -> MrPolygonJob:
        j = MrPolygonJob()
        j.xy, j.first_point, j.point_base, j.npoly = _ptr(xy), _ptr(first_point), point_base, npoly
        j.offset_prime, j.seed, j.poly_index0 = _ptr(offset_prime), seed, poly_index0
        j.layout = self.layout.native
        j.vtx_out, j.first_tri, j.tri_base = _ptr(vtx_out), _ptr(first_tri), tri_base
        j.bbox_out, j.status_out, j.ntri_out = _ptr(bbox_out), _ptr(status_out), _ptr(ntri_out)
        return j

    def triangulate(self, job: MrPolygonJob, algorithm: str = "reference", rings: Optional[MrPolygonRings] = None,
                    indices: Optional[MrPolygonIndices] = None):
        """algorithm "reference": mr_triangulate_batch (the reference's triangulator, for parity); "earclip":
        mr_triangulate_earclip (correct on every simple polygon, same output format), or with `rings`
        mr_triangulate_earclip_holes (polygons with holes).  With `indices` (earclip only):
        mr_triangulate_earclip_indexed, which also writes point indices and takes a NULL vtx_out."""
        _check_algorithm(algorithm, None)
        if indices is not None:
            if algorithm != "earclip":
                raise ValueError("indexed output is written by the earclip algorithm only")
            self.ctx.check(self.ctx.lib.mr_triangulate_earclip_indexed(
                self.ctx.handle, C.byref(job), None if rings is None else C.byref(rings), C.byref(indices)),
                "mr_triangulate_earclip_indexed")
            return
        if rings is not None:
            if algorithm != "earclip":
                raise ValueError("holes are triangulated by the earclip algorithm only")
            self.ctx.check(self.ctx.lib.mr_triangulate_earclip_holes(self.ctx.handle, C.byref(job), C.byref(rings)),
                           "mr_triangulate_earclip_holes")
            return
        name = _ALGORITHMS[algorithm]
        self.ctx.check(getattr(self.ctx.lib, name)(self.ctx.handle, C.byref(job)), name)

    def create_polygons(self, xy, first_point, *, offset_prime=None, seed=0, poly_index0=0,
                        device="cuda", algorithm="reference", rings=None, output="vertices") -> PolygonBatch:
        """Batched create_polygon.  xy: [npts,2] f32 (numpy or cuda tensor); first_point: npoly+1 offsets.
        algorithm: "reference" or "earclip" (see triangulate); ear clipping takes no offset_prime.
        rings = (first_ring, ring_start): polygons with holes (earclip only), as mr_polygon_rings with ring_base
        first_ring[0]; polygon i then gets N + 2H - 2 triangles.
        output: "vertices" (vertex_buffer), "indices" (index_buffer: three u32 per triangle, rows of xy, so xy itself
        is the vertex buffer to draw them with) or "both"; anything but "vertices" needs the earclip algorithm."""
        _check_algorithm(algorithm, offset_prime)
        if rings is not None and algorithm != "earclip":
            raise ValueError("holes are triangulated by the earclip algorithm only")
        if output not in _OUTPUTS:
            raise ValueError(f"output must be one of {_OUTPUTS}, not {output!r}")
        if output != "vertices" and algorithm != "earclip":
            raise ValueError("indexed output is written by the earclip algorithm only")
        fp_host = np.ascontiguousarray(
            first_point.cpu().numpy() if _is_cuda(first_point) else first_point, dtype=np.uint64)
        npoly = len(fp_host) - 1
        rg = keep = None
        if rings is None:
            ft_host = polygon_offsets_host(fp_host)
        else:
            fr, rs = rings
            fr_host = np.ascontiguousarray(fr.cpu().numpy() if _is_cuda(fr) else fr, dtype=np.uint64)
            if len(fr_host) != npoly + 1:
                raise ValueError("first_ring must hold npoly+1 offsets")
            ft_host = polygon_offsets_rings_host(fp_host, fr_host)
            keep = (torch.from_numpy(fr_host.view(np.int64)).to(torch.device(device)),
                    rs if _is_cuda(rs) else torch.from_numpy(
                        np.ascontiguousarray(rs, dtype=np.uint64).view(np.int64)).to(torch.device(device)))
            rg = MrPolygonRings(_ptr(keep[0]), int(fr_host[0]), _ptr(keep[1]))
        dev = torch.device(device)
        xy_d = xy if _is_cuda(xy) else torch.from_numpy(np.ascontiguousarray(xy, dtype=np.float32)).to(dev)
        fp_d = torch.from_numpy(fp_host.view(np.int64)).to(dev)
        ft_d = torch.from_numpy(ft_host.view(np.int64)).to(dev)
        op_d = None
        if offset_prime is not None:
            op = np.ascontiguousarray(offset_prime, dtype=np.uint32).reshape(-1)
            if op.size != 2 * npoly:
                raise ValueError("offset_prime must hold 2*npoly values")
            op_d = torch.from_numpy(op.view(np.int32)).to(dev)
        ntri = int(ft_host[-1])
        vtx = idx = ix = None
        if output != "indices":
            vtx = torch.empty(max(ntri * 3 * self.layout.stride, 32), dtype=torch.uint8, device=dev)
        if output != "vertices":
            idx = torch.empty(max(ntri * 3, 1), dtype=torch.uint32, device=dev)
            ix = MrPolygonIndices(_ptr(idx), int(fp_host[0]))
        bbox = torch.empty((npoly, 4), dtype=torch.float32, device=dev)
        status = torch.empty(npoly, dtype=torch.int32, device=dev)
        nt = torch.empty(npoly, dtype=torch.int32, device=dev)
        self.triangulate(self.job(xy_d, fp_d, npoly, vtx_out=vtx, first_tri=ft_d, bbox_out=bbox,
                                  status_out=status, ntri_out=nt, offset_prime=op_d, seed=seed,
                                  poly_index0=poly_index0, point_base=int(fp_host[0])), algorithm, rg, ix)
        return PolygonBatch(npoly, fp_host, ft_host, None if vtx is None else vtx[: ntri * 3 * self.layout.stride],
                            bbox, status, nt, self.layout, None if idx is None else idx[: ntri * 3], int(fp_host[0]))

    def create_polygon(self, vertices, *, offset_prime=None, seed=0, index=0, algorithm="reference",
                       holes=None) -> PolygonObj:
        """Polygon.create_polygon(vertices): one polygon -> VertexBuffer of n-2 triangles + bbox.

        Like the reference (Polygon.zig:82-92: a mapped-at-creation buffer filled by the emit callback) the
        vertex range is HOST memory -- the stand-in for the mapped range -- so the call takes the library's
        small-batch path: one copy in, one kernel, one copy out.  algorithm: as for create_polygons.
        holes: a list of point arrays, one per hole (earclip only); the polygon then gets N + 2H - 2 triangles."""
        _check_algorithm(algorithm, offset_prime)
        if holes is not None and algorithm != "earclip":
            raise ValueError("holes are triangulated by the earclip algorithm only")
        v = np.ascontiguousarray(vertices, dtype=np.float32).reshape(-1, 2)
        rg = None
        if holes is not None:
            hs = [np.ascontiguousarray(h, dtype=np.float32).reshape(-1, 2) for h in holes]
            rs = np.cumsum([0, len(v)] + [len(h) for h in hs[:-1]]).astype(np.uint64) if hs else np.zeros(1, np.uint64)
            fr = np.array([0, len(hs) + 1], dtype=np.uint64)
            v = np.concatenate([v] + hs).astype(np.float32) if hs else v
            rg = MrPolygonRings(fr.ctypes.data, 0, rs.ctypes.data)
        n = len(v)
        ntri_total = n - 2 + 2 * (len(holes) if holes else 0)
        if n < 2:  # Polygon.zig:82: vertices.len - 2 underflows
            raise ValueError("a polygon needs at least 2 vertices")
        op = None if offset_prime is None else np.ascontiguousarray(offset_prime, dtype=np.uint32).reshape(2)
        fp = np.array([0, n], dtype=np.uint64)
        ft = np.array([0, ntri_total], dtype=np.uint64)
        mapped = np.zeros(max(ntri_total * 3 * self.layout.stride, 1), dtype=np.uint8)  # VertexBuffer.new: zeroed
        bb = np.zeros(4, dtype=np.float32)
        st = np.zeros(1, dtype=np.uint32)
        nt = np.zeros(1, dtype=np.uint32)
        self.triangulate(self.job(v, fp, 1, vtx_out=mapped, first_tri=ft, bbox_out=bb, status_out=st, ntri_out=nt,
                                  offset_prime=op, seed=seed, poly_index0=index), algorithm, rg)
        buf = torch.from_numpy(mapped) if torch is not None else mapped
        vb = VertexBuffer(buf, ntri_total * 3, 1, 0, 0)
        return PolygonObj(vb, (float(bb[0]), float(bb[1]), 0.0), (float(bb[2]), float(bb[3]), 0.0),
                          int(st[0]), int(nt[0]))


class Triangulation:
    """Triangulation.create_polygon(points, context, emit): the callback form of the API.

    A callback cannot cross the C ABI, so the library fills a vertex range and this wrapper
    replays it through `emit(context, point)` in the reference's emit order."""

    def __init__(self, ctx: Context):
        self._poly = Polygon(ctx, VertexLayout.create(GPUVertex))

    def create_polygon(self, points, context, emit: Callable, *, offset_prime=None, seed=0, index=0) -> int:
        obj = self._poly.create_polygon(points, offset_prime=offset_prime, seed=seed, index=index)
        raw = obj.vertex_buffer.vertex_buffer.cpu().numpy()
        stride = self._poly.layout.stride
        off_x = self._poly.layout.attributes[0][0]
        for k in range(obj.ntri * 3):
            p = raw[k * stride + off_x: k * stride + off_x + 8].view(np.float32)
            emit(context, (float(p[0]), float(p[1])))
        return obj.status
