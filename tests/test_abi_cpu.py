"""CPU tests of the C-ABI library: it loads, exports every symbol the header declares, its structs
match the ctypes mirror, and its host-side helpers agree with the oracle.  No compute calls."""
import ctypes as C
import os
import re
import subprocess
import sys
import tempfile

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HEADER = os.path.join(ROOT, "include", "myrenderer_b200.h")


@pytest.fixture(scope="module")
def lib():
    from myrenderer_b200 import _capi

    return _capi.load()


def _declared_functions():
    text = open(HEADER).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(mr_[a-z0-9_]+)\s*\(", text)))


def test_every_declared_symbol_is_exported(lib):
    from myrenderer_b200 import _capi

    names = _declared_functions()
    assert len(names) >= 35
    for n in names:
        assert hasattr(lib, n), f"{n} is declared in the header but not exported by the .so"
    assert sorted(_capi.SIGNATURES) == names, "ctypes signature table and header disagree"
    assert os.path.exists(os.path.join(ROOT, "myrenderer_b200", "lib", "libmyrenderer_b200.a"))


def test_struct_layouts_match_the_header():
    from myrenderer_b200 import _capi

    src = r'''
#include <stdio.h>
#include <stddef.h>
#include "myrenderer_b200.h"
int main(void){
 printf("%zu %zu %zu %zu %zu %zu\n", sizeof(mr_layout), sizeof(mr_terrain_job), sizeof(mr_polygon_job),
        sizeof(mr_terrain_params), sizeof(mr_draw_range), sizeof(mr_attr));
 printf("%zu %zu %zu %zu\n", offsetof(mr_terrain_job, vtx_out), offsetof(mr_terrain_job, layout),
        offsetof(mr_polygon_job, layout), offsetof(mr_polygon_job, ntri_out));
 printf("%u %u\n", MR_NODE_CAP(64), MR_STACK_CAP(64));
 return 0; }'''
    with tempfile.TemporaryDirectory() as d:
        open(os.path.join(d, "t.c"), "w").write(src)
        subprocess.run(["gcc", "-std=c11", "-I", os.path.join(ROOT, "include"), "-o", os.path.join(d, "t"), os.path.join(d, "t.c")], check=True)
        out = subprocess.run([os.path.join(d, "t")], capture_output=True, text=True, check=True).stdout.split()
    vals = [int(x) for x in out]
    assert vals[:6] == [C.sizeof(_capi.MrLayout), C.sizeof(_capi.MrTerrainJob), C.sizeof(_capi.MrPolygonJob),
                        C.sizeof(_capi.MrTerrainParams), C.sizeof(_capi.MrDrawRange), C.sizeof(_capi.MrAttr)]
    assert vals[6:10] == [_capi.MrTerrainJob.vtx_out.offset, _capi.MrTerrainJob.layout.offset,
                          _capi.MrPolygonJob.layout.offset, _capi.MrPolygonJob.ntri_out.offset]
    assert vals[10:] == [8 * 64 + 64, 16 * 64 + 64]


_NO_DEVICE_CHECKS = r'''
import ctypes as C
import sys

sys.path.insert(0, sys.argv[1])
import myrenderer_b200 as mr
from myrenderer_b200._capi import MrTerrainJob

lib = mr.load()
h = C.c_void_p()
assert lib.mr_context_create(0, C.byref(h)) == -2 and not h.value  # MR_E_CUDA
try:
    mr.Context(0)
    raise SystemExit("mr.Context(0) did not raise MrError")
except mr.MrError:
    pass
n = C.c_int(-1)
assert lib.mr_device_count(C.byref(n)) in (0, -2) and n.value == 0
# null context is rejected, not dereferenced
assert lib.mr_terrain_build(None, C.byref(MrTerrainJob())) == -1
print("no-device checks ok")
'''


def test_no_cpu_fallback():
    """No device visible (none installed, or all hidden through CUDA_VISIBLE_DEVICES): every entry point fails with an
    error code, nothing computes on the CPU.  Runs in a child process so that the devices can be hidden from it."""
    r = subprocess.run([sys.executable, "-c", _NO_DEVICE_CHECKS, ROOT], capture_output=True, text=True, timeout=300,
                       env=dict(os.environ, CUDA_VISIBLE_DEVICES=""))
    assert r.returncode == 0 and "no-device checks ok" in r.stdout, r.stdout[-2000:] + r.stderr[-2000:]


def test_layout_presets_and_describe(lib):
    from myrenderer_b200._capi import MrLayout, MrTerrainParams, MrDrawRange

    L = MrLayout()
    assert lib.mr_layout_preset(0, C.byref(L)) == 0
    assert (L.stride, L.nattr, L.attr[0].offset, L.attr[0].ncomp, L.attr[1].offset, L.attr[1].ncomp) == (32, 2, 0, 2, 16, 3)
    assert lib.mr_layout_preset(1, C.byref(L)) == 0 and (L.attr[0].offset, L.attr[1].offset) == (16, 0)
    assert lib.mr_layout_preset(2, C.byref(L)) == 0 and (L.attr[0].ncomp, L.attr[1].ncomp) == (3, 3)
    assert lib.mr_layout_preset(9, C.byref(L)) == -1
    p = MrTerrainParams()
    lib.mr_terrain_params_default(C.byref(p))
    assert (p.grid_step, p.origin_scale, p.height_scale) == (np.float32(0.2), np.float32(0.1), 5.0)
    bmin, bmax, vc, ic = (C.c_float * 3)(), (C.c_float * 3)(), C.c_uint64(), C.c_uint64()
    assert lib.mr_terrain_describe(100, None, bmin, bmax, C.byref(vc), C.byref(ic)) == 0
    assert list(bmin) == [-10.0, 0.0, -10.0] and list(bmax) == [10.0, 5.0, 10.0]  # Terrain.zig:103-110
    assert vc.value == 10000 and ic.value == 58806
    lib.mr_terrain_describe(16384, None, None, None, C.byref(vc), C.byref(ic))
    assert ic.value == 1610416134  # SURVEY 8-a3
    d = MrDrawRange()
    assert lib.mr_polygon_draw_range(10, 15, 4, C.byref(d)) == 0
    assert (d.vertex_count, d.instance_count, d.first_vertex, d.first_instance) == (15, 1, 18, 0)  # VertexBuffer.zig:20-24


def test_unirand_host_matches_oracle(lib, oracle):
    off, prime = C.c_uint32(), C.c_uint32()
    for top in list(range(1, 100)) + [1024, 1723, 4096]:
        assert lib.mr_unirand_seed_host(top, 0xFEED, 3, C.byref(off), C.byref(prime)) == 0
        if top == 1:
            assert prime.value == 1
            continue
        assert (off.value, prime.value) == oracle.unirand_seed(top, 0xFEED, 3)
    st = C.c_uint64(lib.mr_rng_state0(5, 9))
    so = C.c_uint64(oracle.lib().mr_o_rng_state0(5, 9))
    assert st.value == so.value
    for _ in range(20):
        assert lib.mr_rng_u32(C.byref(st)) == oracle.lib().mr_o_rng_u32(C.byref(so))


def test_synth_sizes_and_partitions(lib, oracle):
    for dist in (0, 1):
        fp = np.zeros(5001, dtype=np.uint64)
        assert lib.mr_synth_polygon_sizes(0x5EED0005, 17, 5000, 8, 1024, dist, fp.ctypes.data) == 0
        assert np.array_equal(fp, oracle.synth_polygon_sizes(0x5EED0005, 5000, 8, 1024, dist, poly_index0=17))
    for world in (1, 2, 3, 8):
        r = (C.c_uint32 * (world + 1))()
        assert lib.mr_polygon_partition(fp.ctypes.data, 5000, world, r) == 0
        r = list(r)
        assert r[0] == 0 and r[-1] == 5000 and r == sorted(r)
        n = np.diff(fp.astype(np.int64)).astype(np.float64)
        w = n * np.log2(n) + n
        loads = [w[r[i]:r[i + 1]].sum() for i in range(world)]
        assert max(loads) <= 1.05 * (sum(loads) / world) + w.max()
        rows, qrows = (C.c_uint32 * (world + 1))(), (C.c_uint32 * (world + 1))()
        assert lib.mr_terrain_partition(16384, world, rows, qrows) == 0
        assert rows[0] == 0 and rows[world] == 16384 and qrows[world] == 16383
        assert all(rows[i] <= rows[i + 1] for i in range(world))
