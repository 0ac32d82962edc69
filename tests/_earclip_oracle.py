"""ctypes view of tests/earclip_oracle/libmr_oracle_earclip.so: the CPU checker of mr_triangulate_earclip.

orient_sign() is the exact predicate, triangulate_earclip() a whole batch in the outputs of oracle.polygon_batch plus
the triangle corner ids, emit_ids() the restated sink alone.  The library is built by __graft_entry__.build() (or
`make -C tests/earclip_oracle`)."""
import ctypes as C
import os

import numpy as np

from oracle import oracle as O

LIB_PATH = os.path.join(os.path.dirname(os.path.abspath(__file__)), "earclip_oracle", "libmr_oracle_earclip.so")
_lib = None


def lib():
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise ImportError(f"{LIB_PATH} is missing: run `make -C tests/earclip_oracle` (build() does)")
        L = C.CDLL(LIB_PATH)
        L.mr_o_orient_sign.restype = C.c_int
        L.mr_o_orient_sign.argtypes = [C.c_void_p]
        L.mr_o_triangulate_earclip.restype = C.c_int
        L.mr_o_triangulate_earclip.argtypes = [C.c_void_p, C.c_void_p]
        L.mr_o_emit_ids.restype = C.c_int
        L.mr_o_emit_ids.argtypes = [C.c_void_p, C.c_void_p]
        _lib = L
    return _lib


def _ptr(a):
    return None if a is None else a.ctypes.data


def orient_sign(abc) -> int:
    t = np.ascontiguousarray(abc, dtype=np.float32).reshape(6)
    return int(lib().mr_o_orient_sign(_ptr(t)))


def _job(xy, first_point, first_tri, layout, vtx, bbox, status, ntri):
    job = O.MrPolygonJob()
    job.xy = _ptr(xy)
    job.first_point = _ptr(first_point)
    job.point_base = int(first_point[0])
    job.npoly = len(first_point) - 1
    job.layout = O.layout_struct(*layout)
    job.vtx_out = _ptr(vtx)
    job.first_tri = _ptr(first_tri)
    job.tri_base = int(first_tri[0])
    job.bbox_out = _ptr(bbox)
    job.status_out = _ptr(status)
    job.ntri_out = _ptr(ntri)
    return job


def triangulate_earclip(xy, first_point, *, layout=O.GPUVERTEX_DECL, first_tri=None):
    """Oracle ear clipping of a packed batch: dict(vtx, bbox, status, ntri, ids, first_tri) like oracle.polygon_batch;
    ids holds the corner ids of every triangle of the first_tri ranges (0xFFFFFFFF where nothing was emitted)."""
    xy = np.ascontiguousarray(xy, dtype=np.float32).reshape(-1)
    first_point = np.ascontiguousarray(first_point, dtype=np.uint64)
    npoly = len(first_point) - 1
    first_tri = O.polygon_offsets(first_point) if first_tri is None else np.ascontiguousarray(first_tri, dtype=np.uint64)
    total = int(first_tri[-1] - first_tri[0])
    vtx = np.zeros(max(total * 3 * layout[0], 1), dtype=np.uint8)
    bbox = np.zeros((npoly, 4), dtype=np.float32)
    status = np.zeros(npoly, dtype=np.uint32)
    ntri = np.zeros(npoly, dtype=np.uint32)
    ids = np.full(max(total * 3, 1), 0xFFFFFFFF, dtype=np.uint32)
    job = _job(xy, first_point, first_tri, layout, vtx, bbox, status, ntri)
    rc = lib().mr_o_triangulate_earclip(C.byref(job), _ptr(ids))
    if rc != 0:
        raise RuntimeError(f"oracle triangulate_earclip rc={rc}")
    return dict(vtx=vtx[: total * 3 * layout[0]], bbox=bbox, status=status, ntri=ntri, ids=ids[: total * 3],
                first_tri=first_tri)


def emit_ids(xy, first_point, ids, *, layout=O.GPUVERTEX_DECL):
    """The restated sink fed with given corner ids: (vtx, bbox)."""
    xy = np.ascontiguousarray(xy, dtype=np.float32).reshape(-1)
    first_point = np.ascontiguousarray(first_point, dtype=np.uint64)
    first_tri = O.polygon_offsets(first_point)
    total = int(first_tri[-1])
    vtx = np.zeros(max(total * 3 * layout[0], 1), dtype=np.uint8)
    bbox = np.zeros((len(first_point) - 1, 4), dtype=np.float32)
    ids = np.ascontiguousarray(ids, dtype=np.uint32)
    job = _job(xy, first_point, first_tri, layout, vtx, bbox, None, None)
    lib().mr_o_emit_ids(C.byref(job), _ptr(ids))
    return vtx[: total * 3 * layout[0]], bbox
