"""The C++ mirror of the Zig interface, linked against the STATIC library (the build.zig route),
running the reference App's scene construction (App.zig:54-91)."""
import json
import os
import re
import subprocess

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
EXE = os.path.join(ROOT, "examples", "app_scene")
GOLDEN = os.path.join(os.path.dirname(__file__), "golden")


def _fnv1a(b: bytes) -> int:
    h = 1469598103934665603
    for x in b:
        h = ((h ^ x) * 1099511628211) & 0xFFFFFFFFFFFFFFFF
    return h


def _run(tmp_path, *extra, env=None):
    h = np.load(os.path.join(GOLDEN, "heightmap_100.npy"))
    raw = tmp_path / "heightmap.u16"
    h.astype("<u2").tofile(raw)
    return subprocess.run([EXE, str(raw), "100", *extra], capture_output=True, text=True, timeout=120, env=env)


def test_example_fails_loudly_without_gpu(tmp_path):
    """No device visible (none installed, or all hidden through CUDA_VISIBLE_DEVICES): the example says so and exits 1."""
    assert os.path.exists(EXE), "build() must produce examples/app_scene"
    r = _run(tmp_path, env=dict(os.environ, CUDA_VISIBLE_DEVICES=""))
    assert r.returncode == 1 and "no usable CUDA device" in r.stderr


@pytest.mark.gpu
def test_example_matches_oracle(tmp_path, oracle):
    r = _run(tmp_path, "1", "1")
    assert r.returncode == 0, r.stderr
    out = r.stdout
    h = np.load(os.path.join(GOLDEN, "heightmap_100.npy"))
    vtx, idx = oracle.terrain_build(h, 100)
    m = re.search(r"terrain n=100 vertices=10000 indices=58806 bbox=\(-10,0,-10\)-\(10,5,10\) vtx_hash=(\w+) idx_hash=(\w+)", out)
    assert m, out
    assert int(m.group(1), 16) == _fnv1a(vtx.tobytes()) and int(m.group(2), 16) == _fnv1a(idx.tobytes())
    app = json.load(open(os.path.join(GOLDEN, "app_polygons.json")))
    for k, name in ((1, "polygon1"), (2, "polygon2")):
        P = np.array(app[name], dtype=np.float32)
        ref = oracle.polygon_batch(P, np.array([0, len(P)]), offset_prime=[1, 1])
        m = re.search(rf"polygon{k} n={len(P)} status=0 ntri={len(P) - 2} vertex_count={3 * (len(P) - 2)} bbox=\S+ vtx_hash=(\w+)", out)
        assert m, out
        assert int(m.group(1), 16) == _fnv1a(ref["vtx"].tobytes())
    # SURVEY 8-a known answer through the emit-callback form
    assert "emit: (40,40) (10,40) (40,10) (10,40) (10,10) (40,10)" in out
