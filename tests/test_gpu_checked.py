"""The polygon parity and float-edge cases once more against the BOUNDS-CHECKED build of the library (-DMR_CHECKED: every workspace
array of the fast path carries its length and traps on an index out of range).  compute-sanitizer is not available on
the GPU pool; this is the memory-safety evidence for the shared-memory overlays of triangulate_fast.cuh."""
import os
import subprocess
import sys

import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CHECKED = os.path.join(ROOT, "myrenderer_b200", "lib", "libmyrenderer_b200_checked.so")
CASES = ("xl_class or app_polygons or known_answer or star_polygons or zigauto or generic_vertex or convex_and_large or size_class or skewed "
         "or edge_cases or acute or too_large or host_pointers_and_subrange or sound_families or zipper or small_batch or repeat_edges")


def test_polygon_parity_under_the_checked_build():
    if not os.path.exists(CHECKED):
        pytest.skip("checked library not built (make -C myrenderer_b200/csrc checked)")
    env = dict(os.environ, MR_B200_LIB=CHECKED)
    probe = subprocess.run([sys.executable, "-c", "import myrenderer_b200 as m; print('flags', m.load().mr_build_flags())"],
                           capture_output=True, text=True, cwd=ROOT, env=env)
    assert "flags 1" in probe.stdout, probe.stdout + probe.stderr  # the checked build is the one that gets loaded
    for args in (["test_gpu_parity.py", "-k", CASES], ["test_gpu_poly_float_edges.py"]):
        r = subprocess.run([sys.executable, "-m", "pytest", os.path.join(ROOT, "tests", args[0]), "-x", "-q"] + args[1:],
                           capture_output=True, text=True, timeout=1700, cwd=ROOT, env=env)
        tail = r.stdout[-3000:] + r.stderr[-2000:]
        assert r.returncode == 0, tail
        assert "MR_CHECKED" not in r.stdout + r.stderr, tail
        assert " passed" in r.stdout and "skipped" not in r.stdout.splitlines()[-1], tail
