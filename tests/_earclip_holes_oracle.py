"""ctypes view of tests/earclip_holes_oracle/libmr_oracle_earclip_holes.so, the CPU checker of
mr_triangulate_earclip_holes: crossing_sign() is the exact crossing predicate, triangulate_earclip_holes() a whole batch in
the outputs of _earclip_oracle.triangulate_earclip.  The library is built by __graft_entry__.build() (or
`make -C tests/earclip_holes_oracle`)."""
import ctypes as C
import os

import numpy as np

import _earclip_oracle as EO
from oracle import oracle as O


class MrPolygonRings(C.Structure):
    _fields_ = [("first_ring", C.c_void_p), ("ring_base", C.c_uint64), ("ring_start", C.c_void_p)]


LIB_PATH = os.path.join(os.path.dirname(os.path.abspath(__file__)), "earclip_holes_oracle", "libmr_oracle_earclip_holes.so")
_lib = None


def lib():
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise ImportError(f"{LIB_PATH} is missing: run `make -C tests/earclip_holes_oracle` (build() does)")
        L = C.CDLL(LIB_PATH)
        L.mr_o_crossing_sign.restype = C.c_int
        L.mr_o_crossing_sign.argtypes = [C.c_void_p]
        L.mr_o_triangulate_earclip_holes.restype = C.c_int
        L.mr_o_triangulate_earclip_holes.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p]
        _lib = L
    return _lib


def crossing_sign(q) -> int:
    t = np.ascontiguousarray(q, dtype=np.float32).reshape(9)
    return int(lib().mr_o_crossing_sign(t.ctypes.data))


def offsets_rings(first_point, first_ring):
    """first_tri of mr_polygon_offsets_rings."""
    fp = np.asarray(first_point, np.uint64)
    fr = np.asarray(first_ring, np.uint64)
    n = (fp[1:] - fp[:-1]).astype(np.uint64)
    r = (fr[1:] - fr[:-1]).astype(np.uint64)
    h = np.where((r >= 1) & (r <= n), r.astype(np.int64) - 1, 0)
    cnt = np.maximum(n.astype(np.int64) + 2 * h - 2, 0)
    ft = np.zeros(len(fp), np.uint64)
    ft[1:] = np.cumsum(cnt)
    return ft


def triangulate_earclip_holes(xy, first_point, first_ring, ring_start, *, layout=O.GPUVERTEX_DECL, first_tri=None,
                              ring_base=0):
    """Oracle of a packed batch: dict(vtx, bbox, status, ntri, ids, first_tri); ids are point ids relative to each
    polygon's first point (0xFFFFFFFF where nothing was emitted)."""
    xy = np.ascontiguousarray(xy, dtype=np.float32).reshape(-1)
    first_point = np.ascontiguousarray(first_point, dtype=np.uint64)
    first_ring = np.ascontiguousarray(first_ring, dtype=np.uint64)
    ring_start = np.ascontiguousarray(ring_start, dtype=np.uint64)
    if ring_start.size == 0:
        ring_start = np.zeros(1, np.uint64)
    npoly = len(first_point) - 1
    first_tri = offsets_rings(first_point, first_ring) if first_tri is None else np.ascontiguousarray(first_tri, np.uint64)
    total = int(first_tri[-1] - first_tri[0])
    vtx = np.zeros(max(total * 3 * layout[0], 1), dtype=np.uint8)
    bbox = np.zeros((npoly, 4), dtype=np.float32)
    status = np.zeros(npoly, dtype=np.uint32)
    ntri = np.zeros(npoly, dtype=np.uint32)
    ids = np.full(max(total * 3, 1), 0xFFFFFFFF, dtype=np.uint32)
    job = EO._job(xy, first_point, first_tri, layout, vtx, bbox, status, ntri)
    rg = MrPolygonRings(first_ring.ctypes.data, ring_base, ring_start.ctypes.data)
    rc = lib().mr_o_triangulate_earclip_holes(C.byref(job), C.byref(rg), ids.ctypes.data)
    if rc != 0:
        raise RuntimeError(f"oracle triangulate_earclip_holes rc={rc}")
    return dict(vtx=vtx[: total * 3 * layout[0]], bbox=bbox, status=status, ntri=ntri, ids=ids[: total * 3],
                first_tri=first_tri)
