"""ctypes view of tests/frustum_oracle/libmr_oracle_frustum.so: the CPU checker of mr_terrain_cull_frustum.

frustum_visible() is the per-box test and terrain_cull_frustum() the whole cull, with the outputs and the idx_capacity
rule of oracle.terrain_cull.  The library is built by __graft_entry__.build() (or `make -C tests/frustum_oracle`).
"""
import ctypes as C
import os

import numpy as np

LIB_PATH = os.path.join(os.path.dirname(os.path.abspath(__file__)), "frustum_oracle", "libmr_oracle_frustum.so")
_lib = None


def lib():
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise ImportError(f"{LIB_PATH} is missing: run `make -C tests/frustum_oracle` (build() does)")
        L = C.CDLL(LIB_PATH)
        L.mr_o_frustum_visible.restype = C.c_int
        L.mr_o_frustum_visible.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p]
        L.mr_o_terrain_cull_frustum.restype = C.c_int
        L.mr_o_terrain_cull_frustum.argtypes = [C.c_void_p, C.c_uint32, C.c_uint32, C.c_uint32, C.c_void_p, C.c_void_p,
                                                C.c_void_p, C.c_void_p, C.c_void_p]
        _lib = L
    return _lib


def _ptr(a):
    return None if a is None else a.ctypes.data


def frustum_visible(view_proj, p0, p1) -> bool:
    """The six-plane frustum test of mr_terrain_cull_frustum for one box; view_proj as xform of oracle.terrain_cull."""
    m = np.ascontiguousarray(view_proj, dtype=np.float32).reshape(16)
    a = np.ascontiguousarray(p0, dtype=np.float32).reshape(4)
    b = np.ascontiguousarray(p1, dtype=np.float32).reshape(4)
    return bool(lib().mr_o_frustum_visible(_ptr(m), _ptr(a), _ptr(b)))


def terrain_cull_frustum(bbox, n, tile_rows, tile_cols, view_proj, want_idx=True, idx_capacity=None):
    """Oracle frustum cull: dict(visible, ids, idx, counts) as oracle.terrain_cull returns them.  The index buffer holds
    6 (n-1)^2 words unless idx_capacity is given: then a first pass counts the visible indices and the buffer holds
    exactly that many (at most idx_capacity words)."""
    bbox = np.ascontiguousarray(bbox, dtype=np.float32)
    m = np.ascontiguousarray(view_proj, dtype=np.float32).reshape(16)
    ntiles = bbox.shape[0]
    vis = np.zeros(ntiles, dtype=np.uint32)
    ids = np.zeros(ntiles, dtype=np.uint32)
    counts = np.zeros(2, dtype=np.uint64)
    words = 6 * (n - 1) * (n - 1)
    fn = lib().mr_o_terrain_cull_frustum
    if want_idx and idx_capacity is not None:
        rc = fn(_ptr(bbox), n, tile_rows, tile_cols, _ptr(m), _ptr(vis), _ptr(ids), None, _ptr(counts))
        if rc != 0:
            raise RuntimeError(f"oracle terrain_cull_frustum rc={rc}")
        words = int(counts[1])
        if words > idx_capacity:
            raise ValueError(f"oracle terrain_cull_frustum: {words} visible indices exceed idx_capacity {idx_capacity}")
    idx = np.zeros(words, dtype=np.uint32) if want_idx else None
    rc = fn(_ptr(bbox), n, tile_rows, tile_cols, _ptr(m), _ptr(vis), _ptr(ids), _ptr(idx), _ptr(counts))
    if rc != 0:
        raise RuntimeError(f"oracle terrain_cull_frustum rc={rc}")
    return dict(visible=vis, ids=ids[: int(counts[0])], idx=None if idx is None else idx[: int(counts[1])], counts=counts)
