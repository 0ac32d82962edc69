"""ctypes wrapper of the CPU parity oracle (oracle/libmr_oracle.so).

TEST INFRASTRUCTURE ONLY: imported by tests/, __graft_entry__.smoke() and bench.py's CPU-baseline
legs.  Nothing under myrenderer_b200/ imports this module.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess

import numpy as np

from myrenderer_b200._capi import (MrLayout, MrPolygonJob, MrTerrainJob, MrTerrainParams,
                                   MR_HEIGHT_F32, MR_HEIGHT_U16)

_DIR = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_DIR, "libmr_oracle.so")


class OStats(C.Structure):
    _fields_ = [(k, C.c_uint64) for k in (
        "nodes", "max_stack", "sum_stack", "descent_steps", "mountains", "max_mountain",
        "triangles", "not_acute", "point_steps", "select_steps")]

    def as_dict(self):
        return {k: int(getattr(self, k)) for k, _ in self._fields_}


class ONode(C.Structure):
    _fields_ = [(k, C.c_uint32) for k in ("type", "crumb", "child1", "child2", "point1", "point2")]


class OUnirand(C.Structure):
    _fields_ = [(k, C.c_uint32) for k in ("at", "top", "offset", "prime")]


def build(force: bool = False) -> str:
    srcs = [os.path.join(_DIR, f) for f in os.listdir(_DIR) if f.endswith((".c", ".h"))]
    srcs.append(os.path.join(_DIR, "..", "include", "myrenderer_b200.h"))
    if (force or not os.path.exists(LIB_PATH)
            or any(os.path.getmtime(s) > os.path.getmtime(LIB_PATH) for s in srcs)):
        subprocess.run(["make", "-C", _DIR, "-B"], check=True, capture_output=True)
    return LIB_PATH


_lib = None


def lib() -> C.CDLL:
    global _lib
    if _lib is None:
        build()
        L = C.CDLL(LIB_PATH)
        L.mr_o_rng_state0.restype = C.c_uint64
        L.mr_o_rng_state0.argtypes = [C.c_uint64, C.c_uint64]
        L.mr_o_rng_u32.restype = C.c_uint32
        L.mr_o_rng_u32.argtypes = [C.POINTER(C.c_uint64)]
        L.mr_o_unirand_seed.restype = None
        L.mr_o_unirand_seed.argtypes = [C.POINTER(OUnirand), C.c_uint32, C.POINTER(C.c_uint64)]
        L.mr_o_unirand_next.restype = C.c_int
        L.mr_o_unirand_next.argtypes = [C.POINTER(OUnirand), C.POINTER(C.c_uint32)]
        L.mr_o_atan2f.restype = C.c_float
        L.mr_o_atan2f.argtypes = [C.c_float, C.c_float]
        L.mr_o_atanf.restype = C.c_float
        L.mr_o_atanf.argtypes = [C.c_float]
        L.mr_o_polygon_batch.restype = C.c_int
        L.mr_o_polygon_batch.argtypes = [C.POINTER(MrPolygonJob), C.c_void_p, C.c_int,
                                         C.POINTER(OStats)]
        L.mr_o_palette.restype = None
        L.mr_o_palette.argtypes = [C.POINTER(C.c_float)]
        L.mr_o_terrain_build.restype = C.c_int
        L.mr_o_terrain_build.argtypes = [C.POINTER(MrTerrainJob), C.c_int]
        L.mr_o_heightmap_normalize.restype = None
        L.mr_o_heightmap_normalize.argtypes = [C.c_void_p, C.c_uint64, C.c_void_p]
        L.mr_o_terrain_shader_vertex.restype = C.c_int
        L.mr_o_terrain_shader_vertex.argtypes = [C.c_void_p, C.c_uint32, C.c_uint64,
                                                 C.POINTER(MrTerrainParams), C.POINTER(C.c_float)]
        L.mr_o_synth_heightmap_u16.restype = None
        L.mr_o_synth_heightmap_u16.argtypes = [C.c_uint64, C.c_uint32, C.c_uint32, C.c_uint32,
                                               C.c_void_p]
        L.mr_o_synth_polygon_sizes.restype = None
        L.mr_o_synth_polygon_sizes.argtypes = [C.c_uint64, C.c_uint64, C.c_uint32, C.c_uint32,
                                               C.c_uint32, C.c_int, C.c_void_p]
        L.mr_o_synth_polygons.restype = None
        L.mr_o_synth_polygons.argtypes = [C.c_uint64, C.c_uint64, C.c_void_p, C.c_uint32,
                                          C.c_void_p]
        L.mr_o_synth_polygons_family.restype = None
        L.mr_o_synth_polygons_family.argtypes = [C.c_int, C.c_uint64, C.c_uint64, C.c_void_p, C.c_uint32,
                                                 C.c_void_p]
        L.mr_o_test_lift_caps.restype = None
        L.mr_o_test_lift_caps.argtypes = [C.c_uint32]
        L.mr_o_test_mutant.restype = None
        L.mr_o_test_mutant.argtypes = [C.c_uint32]
        L.mr_o_terrain_tile_bounds.restype = C.c_int
        L.mr_o_terrain_tile_bounds.argtypes = [C.c_void_p, C.c_uint32, C.c_uint32, C.c_uint32, C.c_uint32,
                                               C.POINTER(MrTerrainParams), C.c_void_p]
        L.mr_o_scene_node_should_render.restype = C.c_int
        L.mr_o_scene_node_should_render.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p]
        L.mr_o_terrain_cull.restype = C.c_int
        L.mr_o_terrain_cull.argtypes = [C.c_void_p, C.c_uint32, C.c_uint32, C.c_uint32, C.c_void_p, C.c_void_p,
                                        C.c_void_p, C.c_void_p, C.c_void_p]
        L.mr_o_time_create_polygon.restype = C.c_double
        L.mr_o_time_create_polygon.argtypes = [C.c_void_p, C.c_uint32, C.c_uint32, C.c_uint32, C.c_uint32]
        L.mr_o_hardware_threads.restype = C.c_int
        L.mr_o_tri_new.restype = C.c_void_p
        L.mr_o_tri_destroy.argtypes = [C.c_void_p]
        L.mr_o_tri_create_polygon.restype = C.c_uint32
        L.mr_o_tri_create_polygon.argtypes = [C.c_void_p, C.c_void_p, C.c_uint32, OUnirand,
                                              C.c_void_p, C.c_void_p, C.POINTER(OStats)]
        L.mr_o_tri_node_count.restype = C.c_uint32
        L.mr_o_tri_node_count.argtypes = [C.c_void_p]
        L.mr_o_tri_nodes.restype = C.POINTER(ONode)
        L.mr_o_tri_nodes.argtypes = [C.c_void_p]
        _lib = L
    return _lib


def _ptr(a):
    return None if a is None else a.ctypes.data


# ---------------------------------------------------------------------------------------------
def layout_struct(stride, attrs) -> MrLayout:
    L = MrLayout()
    L.stride = stride
    L.nattr = len(attrs)
    for i, (off, ncomp) in enumerate(attrs):
        L.attr[i].offset = off
        L.attr[i].ncomp = ncomp
        L.attr[i].location = i
    return L


GPUVERTEX_DECL = (32, ((0, 2), (16, 3)))
GPUVERTEX_ZIGAUTO = (32, ((16, 2), (0, 3)))
TERRAINVERTEX = (32, ((0, 3), (16, 3)))


def hardware_threads() -> int:
    return int(lib().mr_o_hardware_threads())


def unirand_seed(top: int, seed: int, index: int):
    """(offset, prime) the documented stream yields for polygon `index` of size `top`."""
    st = C.c_uint64(lib().mr_o_rng_state0(seed, index))
    r = OUnirand()
    lib().mr_o_unirand_seed(C.byref(r), top, C.byref(st))
    return int(r.offset), int(r.prime)


def unirand_sequence(top: int, offset: int, prime: int):
    r = OUnirand(0, top, offset, prime)
    out, v = [], C.c_uint32()
    while lib().mr_o_unirand_next(C.byref(r), C.byref(v)):
        out.append(int(v.value))
    return out


def polygon_offsets(first_point: np.ndarray) -> np.ndarray:
    n = np.diff(first_point.astype(np.int64))
    ft = np.zeros(len(first_point), dtype=np.uint64)
    ft[1:] = np.cumsum(np.maximum(n - 2, 0))
    return ft


def polygon_batch(xy, first_point, *, offset_prime=None, seed=0, poly_index0=0,
                  layout=GPUVERTEX_DECL, nthreads=1, want_ids=True, want_stats=False):
    """Run the oracle on a packed batch.  Returns dict(vtx, bbox, status, ntri, ids, stats)."""
    xy = np.ascontiguousarray(xy, dtype=np.float32).reshape(-1)
    first_point = np.ascontiguousarray(first_point, dtype=np.uint64)
    npoly = len(first_point) - 1
    first_tri = polygon_offsets(first_point)
    ntri_total = int(first_tri[-1])
    stride = layout[0]
    vtx = np.zeros(max(ntri_total * 3 * stride, 1), dtype=np.uint8)
    bbox = np.zeros((npoly, 4), dtype=np.float32)
    status = np.zeros(npoly, dtype=np.uint32)
    ntri = np.zeros(npoly, dtype=np.uint32)
    ids = np.full(max(ntri_total * 3, 1), 0xFFFFFFFF, dtype=np.uint32) if want_ids else None
    op = None
    if offset_prime is not None:
        op = np.ascontiguousarray(offset_prime, dtype=np.uint32).reshape(-1)
        assert op.size == 2 * npoly
    job = MrPolygonJob()
    job.xy = _ptr(xy)
    job.first_point = _ptr(first_point)
    job.point_base = int(first_point[0])
    job.npoly = npoly
    job.offset_prime = _ptr(op)
    job.seed = seed
    job.poly_index0 = poly_index0
    job.layout = layout_struct(*layout)
    job.vtx_out = _ptr(vtx)
    job.first_tri = _ptr(first_tri)
    job.tri_base = 0
    job.bbox_out = _ptr(bbox)
    job.status_out = _ptr(status)
    job.ntri_out = _ptr(ntri)
    stats = OStats()
    rc = lib().mr_o_polygon_batch(C.byref(job), _ptr(ids), nthreads,
                                  C.byref(stats) if want_stats else None)
    if rc != 0:
        raise RuntimeError(f"oracle polygon_batch rc={rc}")
    return dict(vtx=vtx[: ntri_total * 3 * stride], bbox=bbox, status=status, ntri=ntri,
                ids=None if ids is None else ids[: ntri_total * 3], first_tri=first_tri,
                stats=stats.as_dict() if want_stats else None)


def terrain_build(height, n, *, layout=TERRAINVERTEX, params=(0.2, 0.1, 5.0), rows=None,
                  qrows=None, height_row0=0, want_vtx=True, want_idx=True, nthreads=1):
    """Oracle mesh of rows [rows) / quad rows [qrows) of an n x n terrain.
    `height` is u16 or f32, holding rows height_row0.. of the heightmap."""
    height = np.ascontiguousarray(height)
    fmt = MR_HEIGHT_U16 if height.dtype == np.uint16 else MR_HEIGHT_F32
    if fmt == MR_HEIGHT_F32:
        height = height.astype(np.float32, copy=False)
    rows = (0, n) if rows is None else rows
    qrows = (0, max(n - 1, 0)) if qrows is None else qrows
    stride = layout[0]
    vtx = np.zeros((rows[1] - rows[0]) * n * stride, dtype=np.uint8) if want_vtx else None
    idx = np.zeros((qrows[1] - qrows[0]) * 6 * max(n - 1, 0), dtype=np.uint32) if want_idx else None
    job = MrTerrainJob()
    job.n = n
    job.height_fmt = fmt
    job.height = _ptr(height)
    job.height_row0 = height_row0
    job.height_rows = height.size // n
    job.row_begin, job.row_end = rows
    job.vtx_out = _ptr(vtx) if want_vtx and vtx.size else None
    job.vtx_row0 = rows[0]
    job.qrow_begin, job.qrow_end = qrows
    job.idx_out = _ptr(idx) if want_idx and idx.size else None
    job.idx_qrow0 = qrows[0]
    job.layout = layout_struct(*layout)
    job.params = MrTerrainParams(*params)
    rc = lib().mr_o_terrain_build(C.byref(job), nthreads)
    if rc != 0:
        raise RuntimeError(f"oracle terrain_build rc={rc}")
    return vtx, idx


def tile_count(n, tile_rows, tile_cols):
    return (n - 1 + tile_rows - 1) // tile_rows, (n - 1 + tile_cols - 1) // tile_cols


def terrain_tile_bounds(height, n, tile_rows, tile_cols, params=(0.2, 0.1, 5.0)) -> np.ndarray:
    """[tiles, 8] f32: p0.xyzw, p1.xyzw per tile (tile t = tr * tiles_c + tc)."""
    height = np.ascontiguousarray(height)
    fmt = MR_HEIGHT_U16 if height.dtype == np.uint16 else MR_HEIGHT_F32
    tr, tc = tile_count(n, tile_rows, tile_cols)
    out = np.zeros((tr * tc, 8), dtype=np.float32)
    p = MrTerrainParams(*params)
    rc = lib().mr_o_terrain_tile_bounds(_ptr(height), fmt, n, tile_rows, tile_cols, C.byref(p), _ptr(out))
    if rc != 0:
        raise RuntimeError(f"oracle tile_bounds rc={rc}")
    return out


def scene_node_should_render(xform, p0, p1) -> bool:
    """SceneNode.zig:96-110 for one bounding box; xform = 16 floats, memory image of mach.math.Mat4x4 (columns)."""
    m = np.ascontiguousarray(xform, dtype=np.float32).reshape(16)
    a = np.ascontiguousarray(p0, dtype=np.float32).reshape(4)
    b = np.ascontiguousarray(p1, dtype=np.float32).reshape(4)
    return bool(lib().mr_o_scene_node_should_render(_ptr(m), _ptr(a), _ptr(b)))


def terrain_cull(bbox, n, tile_rows, tile_cols, xform, want_idx=True):
    bbox = np.ascontiguousarray(bbox, dtype=np.float32)
    m = np.ascontiguousarray(xform, dtype=np.float32).reshape(16)
    ntiles = bbox.shape[0]
    vis = np.zeros(ntiles, dtype=np.uint32)
    ids = np.zeros(ntiles, dtype=np.uint32)
    idx = np.zeros(6 * (n - 1) * (n - 1), dtype=np.uint32) if want_idx else None
    counts = np.zeros(2, dtype=np.uint64)
    rc = lib().mr_o_terrain_cull(_ptr(bbox), n, tile_rows, tile_cols, _ptr(m), _ptr(vis), _ptr(ids), _ptr(idx), _ptr(counts))
    if rc != 0:
        raise RuntimeError(f"oracle terrain_cull rc={rc}")
    return dict(visible=vis, ids=ids[: int(counts[0])], idx=None if idx is None else idx[: int(counts[1])], counts=counts)


def heightmap_normalize(u16: np.ndarray) -> np.ndarray:
    u16 = np.ascontiguousarray(u16, dtype=np.uint16)
    out = np.empty(u16.shape, dtype=np.float32)
    lib().mr_o_heightmap_normalize(_ptr(u16), u16.size, _ptr(out))
    return out


def terrain_shader_vertex(h: np.ndarray, n: int, vi: int, params=(0.2, 0.1, 5.0)):
    h = np.ascontiguousarray(h, dtype=np.float32)
    out = (C.c_float * 4)()
    p = MrTerrainParams(*params)
    ok = lib().mr_o_terrain_shader_vertex(_ptr(h), n, vi, C.byref(p), out)
    return np.array(out[:], dtype=np.float32) if ok else None


def synth_heightmap_u16(seed, n, row0=0, rows=None) -> np.ndarray:
    rows = n if rows is None else rows
    out = np.empty((rows, n), dtype=np.uint16)
    lib().mr_o_synth_heightmap_u16(seed, n, row0, rows, _ptr(out))
    return out


def synth_polygon_sizes(seed, npoly, nmin, nmax, dist=0, poly_index0=0) -> np.ndarray:
    fp = np.zeros(npoly + 1, dtype=np.uint64)
    lib().mr_o_synth_polygon_sizes(seed, poly_index0, npoly, nmin, nmax, dist, _ptr(fp))
    return fp


FAMILY_STAR, FAMILY_ELLIPSE, FAMILY_ZIPPER = 0, 1, 2


def synth_polygons(seed, first_point, poly_index0=0, family=FAMILY_STAR) -> np.ndarray:
    first_point = np.ascontiguousarray(first_point, dtype=np.uint64)
    npts = int(first_point[-1] - first_point[0])
    xy = np.empty((npts, 2), dtype=np.float32)
    lib().mr_o_synth_polygons_family(family, seed, poly_index0, _ptr(first_point), len(first_point) - 1, _ptr(xy))
    return xy


def time_create_polygon(xy, offset, prime, reps=20000) -> float:
    """Mean seconds per single-polygon call of the CPU port (timed inside C)."""
    xy = np.ascontiguousarray(xy, dtype=np.float32).reshape(-1, 2)
    return float(lib().mr_o_time_create_polygon(_ptr(xy), len(xy), offset, prime, reps))


def lift_caps(multiplier: int):
    """Test-only: multiply the contract caps of the oracle (1 restores them)."""
    lib().mr_o_test_lift_caps(multiplier)


# Test-only mutants of the float rules (mr_oracle.h, MR_O_MUT_*): name -> (id, rule).  Same order as the C enum.
MUTANTS = {name: (i + 1, rule) for i, (name, rule) in enumerate((
    ("fma", "side"), ("f64", "side"), ("exactdiff", "side"), ("reform", "side"), ("ftz", "side"), ("ge", "side"),
    ("rawzero", "order"), ("signflip", "order"), ("daz", "order"), ("tie_le", "order"),
    ("cr_atan2", "acute"), ("pi_down", "acute"), ("le", "acute"), ("always", "acute"), ("daz_atan2", "acute"),
    ("tie_replaces", "bbox"), ("own_y", "bbox"),
    ("x_only", "nonfinite"), ("nan_only", "nonfinite")))}


class mutant:
    """Test-only: `with mutant("ftz"): ...` runs the oracle with one float rule replaced (None = the reference)."""

    def __init__(self, name):
        self.id = 0 if name is None else MUTANTS[name][0]

    def __enter__(self):
        lib().mr_o_test_mutant(self.id)
        return self

    def __exit__(self, *exc):
        lib().mr_o_test_mutant(0)


def atan2f(y, x) -> float:
    return float(lib().mr_o_atan2f(y, x))
