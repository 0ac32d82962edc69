"""ctypes view of include/myrenderer_b200.h and the loader for libmyrenderer_b200.so.

The library is the product: there is no Python or CPU fallback.  `load()` raises if the shared
object is missing (run `python -c "import __graft_entry__ as g; g.build()"` or `make -C
myrenderer_b200/csrc`), and every compute call raises `MrError` if CUDA is unavailable.
"""
from __future__ import annotations

import ctypes as C
import os

MR_MAX_ATTR = 4
MR_OK = 0
MR_HEIGHT_U16 = 0
MR_HEIGHT_F32 = 1
MR_LAYOUT_GPUVERTEX_DECL = 0
MR_LAYOUT_GPUVERTEX_ZIGAUTO = 1
MR_LAYOUT_TERRAINVERTEX = 2
MR_SIZES_UNIFORM = 0
MR_SIZES_LOGUNIFORM = 1
MR_IPC_HANDLE_BYTES = 64
MR_MAX_POLYGON_POINTS = 4096

MR_POLY_OK = 0
MR_POLY_DEGENERATE = 1
MR_POLY_NONFINITE = 2
MR_POLY_NULL_UNWRAP = 4
MR_POLY_OVERFLOW = 8
MR_POLY_STUCK = 16
MR_POLY_TOO_LARGE = 32
MR_POLY_ARENA = 64
MR_POLY_UNDERFILL = 128
MR_POLY_NO_EAR = 256
MR_POLY_BAD_HOLE = 512

ERROR_NAMES = {-1: "MR_E_BADARG", -2: "MR_E_CUDA", -3: "MR_E_NOMEM", -4: "MR_E_ARENA"}


class MrAttr(C.Structure):
    _fields_ = [("offset", C.c_uint32), ("ncomp", C.c_uint32), ("location", C.c_uint32)]


class MrLayout(C.Structure):
    _fields_ = [("stride", C.c_uint32), ("nattr", C.c_uint32), ("attr", MrAttr * MR_MAX_ATTR)]


class MrDrawRange(C.Structure):
    _fields_ = [
        ("vertex_count", C.c_uint32),
        ("instance_count", C.c_uint32),
        ("first_vertex", C.c_uint32),
        ("first_instance", C.c_uint32),
    ]


class MrTerrainParams(C.Structure):
    _fields_ = [("grid_step", C.c_float), ("origin_scale", C.c_float), ("height_scale", C.c_float)]


class MrTerrainJob(C.Structure):
    _fields_ = [
        ("n", C.c_uint32),
        ("height_fmt", C.c_uint32),
        ("height", C.c_void_p),
        ("height_row0", C.c_uint32),
        ("height_rows", C.c_uint32),
        ("row_begin", C.c_uint32),
        ("row_end", C.c_uint32),
        ("vtx_out", C.c_void_p),
        ("vtx_row0", C.c_uint32),
        ("qrow_begin", C.c_uint32),
        ("qrow_end", C.c_uint32),
        ("idx_out", C.c_void_p),
        ("idx_qrow0", C.c_uint32),
        ("layout", MrLayout),
        ("params", MrTerrainParams),
    ]


class MrPolygonJob(C.Structure):
    _fields_ = [
        ("xy", C.c_void_p),
        ("first_point", C.c_void_p),
        ("point_base", C.c_uint64),
        ("npoly", C.c_uint32),
        ("offset_prime", C.c_void_p),
        ("seed", C.c_uint64),
        ("poly_index0", C.c_uint64),
        ("layout", MrLayout),
        ("vtx_out", C.c_void_p),
        ("first_tri", C.c_void_p),
        ("tri_base", C.c_uint64),
        ("bbox_out", C.c_void_p),
        ("status_out", C.c_void_p),
        ("ntri_out", C.c_void_p),
    ]


class MrPolygonRings(C.Structure):
    _fields_ = [("first_ring", C.c_void_p), ("ring_base", C.c_uint64), ("ring_start", C.c_void_p)]


class MrPolygonIndices(C.Structure):
    _fields_ = [("idx_out", C.c_void_p), ("index_base", C.c_uint64)]


class MrDrawIndexedRange(C.Structure):
    _fields_ = [
        ("index_count", C.c_uint32),
        ("instance_count", C.c_uint32),
        ("first_index", C.c_uint32),
        ("base_vertex", C.c_int32),
        ("first_instance", C.c_uint32),
    ]


class MrError(RuntimeError):
    def __init__(self, code: int, where: str, detail: str = ""):
        self.code = code
        name = ERROR_NAMES.get(code, str(code))
        super().__init__(f"{where} failed with {name}" + (f": {detail}" if detail else ""))


_PKG_DIR = os.path.dirname(os.path.abspath(__file__))
# MR_B200_LIB selects another build of the same library (the bounds-checked one: make -C myrenderer_b200/csrc checked)
LIB_PATH = os.environ.get("MR_B200_LIB") or os.path.join(_PKG_DIR, "lib", "libmyrenderer_b200.so")

# name -> (restype, argtypes); also the list tests use to check that every declared symbol exports
SIGNATURES = {
    "mr_abi_version": (C.c_int, []),
    "mr_device_count": (C.c_int, [C.POINTER(C.c_int)]),
    "mr_context_create": (C.c_int, [C.c_int, C.POINTER(C.c_void_p)]),
    "mr_context_destroy": (C.c_int, [C.c_void_p]),
    "mr_context_set_stream": (C.c_int, [C.c_void_p, C.c_void_p]),
    "mr_context_stream": (C.c_int, [C.c_void_p, C.POINTER(C.c_void_p)]),
    "mr_sync": (C.c_int, [C.c_void_p]),
    "mr_last_error": (C.c_char_p, [C.c_void_p]),
    "mr_launch_count": (C.c_uint64, [C.c_void_p]),
    "mr_device_alloc": (C.c_int, [C.c_void_p, C.c_size_t, C.POINTER(C.c_void_p)]),
    "mr_device_free": (C.c_int, [C.c_void_p, C.c_void_p]),
    "mr_pinned_alloc": (C.c_int, [C.c_void_p, C.c_size_t, C.POINTER(C.c_void_p)]),
    "mr_pinned_free": (C.c_int, [C.c_void_p, C.c_void_p]),
    "mr_copy": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t]),
    "mr_fill_zero": (C.c_int, [C.c_void_p, C.c_void_p, C.c_size_t]),
    "mr_layout_preset": (C.c_int, [C.c_int, C.POINTER(MrLayout)]),
    "mr_terrain_params_default": (C.c_int, [C.POINTER(MrTerrainParams)]),
    "mr_terrain_build": (C.c_int, [C.c_void_p, C.POINTER(MrTerrainJob)]),
    "mr_terrain_build_full": (
        C.c_int,
        [C.c_void_p, C.c_void_p, C.c_uint32, C.c_uint32, C.POINTER(MrLayout),
         C.POINTER(MrTerrainParams), C.c_void_p, C.c_void_p],
    ),
    "mr_terrain_describe": (
        C.c_int,
        [C.c_uint32, C.POINTER(MrTerrainParams), C.POINTER(C.c_float), C.POINTER(C.c_float),
         C.POINTER(C.c_uint64), C.POINTER(C.c_uint64)],
    ),
    "mr_heightmap_normalize": (C.c_int, [C.c_void_p, C.c_void_p, C.c_uint64, C.c_void_p]),
    "mr_selftest_fastdiv": (C.c_int, [C.c_void_p, C.c_float, C.c_int, C.POINTER(C.c_uint64)]),
    "mr_triangulate_batch": (C.c_int, [C.c_void_p, C.POINTER(MrPolygonJob)]),
    "mr_triangulate_earclip": (C.c_int, [C.c_void_p, C.POINTER(MrPolygonJob)]),
    "mr_selftest_orient": (C.c_int, [C.c_void_p, C.c_void_p, C.c_uint64, C.c_void_p]),
    "mr_triangulate_earclip_holes": (C.c_int, [C.c_void_p, C.POINTER(MrPolygonJob), C.POINTER(MrPolygonRings)]),
    "mr_triangulate_earclip_indexed": (
        C.c_int, [C.c_void_p, C.POINTER(MrPolygonJob), C.POINTER(MrPolygonRings), C.POINTER(MrPolygonIndices)]),
    "mr_polygon_draw_indexed_range": (
        C.c_int, [C.c_uint64, C.c_uint64, C.c_uint64, C.POINTER(MrDrawIndexedRange)]),
    "mr_selftest_crossing": (C.c_int, [C.c_void_p, C.c_void_p, C.c_uint64, C.c_void_p]),
    "mr_polygon_offsets_rings": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint32, C.c_void_p]),
    "mr_polygon_offsets": (C.c_int, [C.c_void_p, C.c_void_p, C.c_uint32, C.c_void_p]),
    "mr_triangulate_tier_counts": (C.c_int, [C.c_void_p, C.POINTER(C.c_uint32)]),
    "mr_polygon_draw_range": (
        C.c_int, [C.c_uint64, C.c_uint64, C.c_uint64, C.POINTER(MrDrawRange)]),
    "mr_rng_u32": (C.c_uint32, [C.POINTER(C.c_uint64)]),
    "mr_rng_state0": (C.c_uint64, [C.c_uint64, C.c_uint64]),
    "mr_unirand_seed_host": (
        C.c_int, [C.c_uint32, C.c_uint64, C.c_uint64, C.POINTER(C.c_uint32), C.POINTER(C.c_uint32)]),
    "mr_unirand_seed_batch": (
        C.c_int, [C.c_void_p, C.c_void_p, C.c_uint32, C.c_uint64, C.c_uint64, C.c_void_p]),
    "mr_synth_heightmap_u16": (
        C.c_int, [C.c_void_p, C.c_uint64, C.c_uint32, C.c_uint32, C.c_uint32, C.c_void_p]),
    "mr_synth_polygon_sizes": (
        C.c_int,
        [C.c_uint64, C.c_uint64, C.c_uint32, C.c_uint32, C.c_uint32, C.c_int, C.c_void_p]),
    "mr_synth_polygons": (
        C.c_int, [C.c_void_p, C.c_uint64, C.c_uint64, C.c_void_p, C.c_uint32, C.c_void_p]),
    "mr_terrain_tile_count": (C.c_int, [C.c_uint32, C.c_uint32, C.c_uint32, C.POINTER(C.c_uint32), C.POINTER(C.c_uint32)]),
    "mr_terrain_tile_bounds": (
        C.c_int, [C.c_void_p, C.c_void_p, C.c_uint32, C.c_uint32, C.c_uint32, C.c_uint32, C.c_void_p, C.c_void_p]),
    "mr_terrain_cull": (
        C.c_int, [C.c_void_p, C.c_void_p, C.c_uint32, C.c_uint32, C.c_uint32, C.c_void_p, C.c_void_p, C.c_void_p,
                  C.c_void_p, C.c_void_p]),
    "mr_terrain_cull_frustum": (
        C.c_int, [C.c_void_p, C.c_void_p, C.c_uint32, C.c_uint32, C.c_uint32, C.c_void_p, C.c_void_p, C.c_void_p,
                  C.c_void_p, C.c_void_p]),
    "mr_build_flags": (C.c_int, []),
    "mr_context_trim": (C.c_int, [C.c_void_p]),
    "mr_context_scratch_bytes": (C.c_int, [C.c_void_p, C.POINTER(C.c_uint64)]),
    "mr_synth_polygons_family": (
        C.c_int, [C.c_void_p, C.c_int, C.c_uint64, C.c_uint64, C.c_void_p, C.c_uint32, C.c_void_p]),
    "mr_ipc_export": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p]),
    "mr_ipc_open": (C.c_int, [C.c_void_p, C.c_void_p, C.POINTER(C.c_void_p)]),
    "mr_ipc_close": (C.c_int, [C.c_void_p, C.c_void_p]),
    "mr_polygon_partition": (C.c_int, [C.c_void_p, C.c_uint32, C.c_uint32, C.c_void_p]),
    "mr_terrain_partition": (C.c_int, [C.c_uint32, C.c_uint32, C.c_void_p, C.c_void_p]),
}

_lib = None


def load() -> C.CDLL:
    """Load libmyrenderer_b200.so (once).  Raises if it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            f"{LIB_PATH} is missing: build the CUDA library first "
            "(python -c 'import __graft_entry__ as g; g.build()'). There is no CPU fallback."
        )
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)  # AttributeError here means the .so is stale
        fn.restype = res
        fn.argtypes = args
    if lib.mr_abi_version() != 1:
        raise ImportError("libmyrenderer_b200.so ABI version mismatch; rebuild")
    _lib = lib
    return lib
