"""The expected output of mr_triangulate_earclip_indexed, built from the ear-clipping oracles' corner ids by the header's
rule, and its replay through the oracle's sink (mr_o_emit_ids)."""
import ctypes as C

import numpy as np

import _earclip_oracle as EO
from oracle import oracle as O

NONE = 0xFFFFFFFF
M32 = np.uint64(0xFFFFFFFF)


def _poly_of_entry(first_tri):
    ft = np.asarray(first_tri, np.uint64).astype(np.int64)
    return np.repeat(np.arange(len(ft) - 1), 3 * np.diff(ft))


def expected_indices(ids, first_point, first_tri, index_base):
    """idx_out over the job's range [3*first_tri[0], 3*first_tri[npoly]) from the oracle's polygon-local corner ids: id k
    of polygon i becomes the low 32 bits of first_point[i] + k - index_base, and an entry the oracle left at 0xFFFFFFFF
    (nothing emitted there) becomes 0."""
    fp = np.asarray(first_point, np.uint64)
    ids = np.asarray(ids, np.uint32)
    poly = _poly_of_entry(first_tri)
    v = (fp[:-1][poly] + ids.astype(np.uint64) - np.uint64(index_base)) & M32
    return np.where(ids == NONE, 0, v).astype(np.uint32)


def local_ids(idx, first_point, first_tri, index_base, ntri):
    """The inverse for a replay: polygon-local corner ids of each polygon's first ntri[i] triangles, 0xFFFFFFFF after."""
    fp = np.asarray(first_point, np.uint64)
    ft = np.asarray(first_tri, np.uint64).astype(np.int64)
    poly = _poly_of_entry(first_tri)
    k = (np.asarray(idx, np.uint32).astype(np.uint64) + np.uint64(index_base) - fp[:-1][poly]) & M32
    pos = np.arange(len(poly)) - 3 * (ft[:-1][poly] - ft[0])
    return np.where(pos < 3 * np.asarray(ntri, np.int64)[poly], k, NONE).astype(np.uint32)


def replay(xy, first_point, first_tri, ids, *, layout=O.GPUVERTEX_DECL):
    """The oracle's sink fed with polygon-local corner ids over the given first_tri ranges: (vtx, bbox).  xy holds the
    points from first_point[0] on."""
    xy = np.ascontiguousarray(xy, dtype=np.float32).reshape(-1)
    fp = np.ascontiguousarray(first_point, dtype=np.uint64)
    ft = np.ascontiguousarray(first_tri, dtype=np.uint64)
    total = int(ft[-1] - ft[0])
    vtx = np.zeros(max(total * 3 * layout[0], 1), dtype=np.uint8)
    bbox = np.zeros((len(fp) - 1, 4), dtype=np.float32)
    ids = np.ascontiguousarray(np.concatenate([np.asarray(ids, np.uint32), [NONE]]), dtype=np.uint32)
    job = EO._job(xy, fp, ft, layout, vtx, bbox, None, None)
    EO.lib().mr_o_emit_ids(C.byref(job), ids.ctypes.data)
    return vtx[: total * 3 * layout[0]], bbox


def check_replay(ref, idx, xy, first_point, index_base, *, layout=O.GPUVERTEX_DECL):
    """Gathering xy through idx and replaying the sink gives the oracle's vertex bytes, and its bbox wherever no triangle
    was dropped (an OVERFLOW bbox also counts the dropped ones)."""
    ft = ref["first_tri"]
    ids = local_ids(idx, first_point, ft, index_base, ref["ntri"])
    vtx, bbox = replay(xy, first_point, ft, ids, layout=layout)
    assert np.array_equal(vtx, ref["vtx"]), "replayed vertex bytes differ"
    keep = (ref["status"] & 8) == 0
    assert np.array_equal(bbox[keep].view(np.uint32), ref["bbox"][keep].view(np.uint32)), "replayed bbox differs"
