"""Regenerates tests/golden/*.  Run in the build container only (reads /root/reference).

  heightmap_100.npy       u16[100][100] decoded from the reference's App/HEIGHTMAP.png
                          (sha256 of the PNG checked against SURVEY 4); a data fixture, not source
  heightmap_100.png       the same pixels as a 16-bit grayscale PNG written by write_png_u16 below (not by the
                          loader's library), the input of the PNG loader's test; `make_golden.py png` rewrites it
                          from the committed heightmap_100.npy alone
  app_polygons.json       the two literal polygons of App/App.zig:68-83 (f32 values)
  kat.json                oracle outputs (known-answer vectors):
      polygon2 / linear order  -> the hand-derived answer of SURVEY 8-a
      polygon1, polygon2 for every (offset, prime) unirand_seed can produce -> emitted ids
      terrain: sha256 of the oracle's vertex and index bytes for HEIGHTMAP.png
"""
import hashlib
import json
import os
import struct
import sys
import zlib

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))
from oracle import oracle as O  # noqa: E402

REF = "/root/reference"
PNG_SHA = "8bea44e35bb0ef2fcb40f24bd38ad4000bf435c3ea7a6e2d48858058c9d2f646"

POLYGON1 = [[62.742857, 106.97143], [93.085712, 65.828571], [147.08571, 85.628572], [122.14285, 144.77143],
            [102.34286, 93.857142], [79.199998, 130.37143], [81.00000, 105.17143]]
POLYGON2 = [[10.0, 10.0], [40.0, 10.0], [40.0, 40.0], [10.0, 40.0]]


def write_png_u16(path, a):
    """Minimal PNG writer: 16-bit grayscale, no interlace, filter type 0 on every row, one IDAT chunk."""
    h, w = a.shape
    raw = b"".join(b"\x00" + np.ascontiguousarray(a[r], dtype=">u2").tobytes() for r in range(h))

    def chunk(tag, data):
        return struct.pack(">I", len(data)) + tag + data + struct.pack(">I", zlib.crc32(tag + data))

    with open(path, "wb") as f:
        f.write(b"\x89PNG\r\n\x1a\n" + chunk(b"IHDR", struct.pack(">IIBBBBB", w, h, 16, 0, 0, 0, 0))
                + chunk(b"IDAT", zlib.compress(raw, 9)) + chunk(b"IEND", b""))


def write_heightmap_png():
    write_png_u16(os.path.join(HERE, "heightmap_100.png"), np.load(os.path.join(HERE, "heightmap_100.npy")))


def main():
    from PIL import Image

    png = os.path.join(REF, "App", "HEIGHTMAP.png")
    assert hashlib.sha256(open(png, "rb").read()).hexdigest() == PNG_SHA
    h = np.ascontiguousarray(np.asarray(Image.open(png)).astype(np.uint16))
    assert h.shape == (100, 100)
    np.save(os.path.join(HERE, "heightmap_100.npy"), h)
    write_heightmap_png()
    json.dump({"polygon1": POLYGON1, "polygon2": POLYGON2}, open(os.path.join(HERE, "app_polygons.json"), "w"))

    kat = {}
    vtx, idx = O.terrain_build(h, 100)
    kat["terrain_100"] = {
        "vtx_sha256": hashlib.sha256(vtx.tobytes()).hexdigest(),
        "idx_sha256": hashlib.sha256(idx.tobytes()).hexdigest(),
        "first_vertex_words": vtx[:32].view(np.uint32).tolist(),
        "vertex_5050_words": vtx[32 * 5050: 32 * 5051].view(np.uint32).tolist(),
        "first_indices": idx[:12].tolist(),
    }
    primes = [1, 2, 3, 5]
    for name, pts in (("polygon1", POLYGON1), ("polygon2", POLYGON2)):
        p = np.array(pts, dtype=np.float32)
        n = len(p)
        out = {}
        for off in range(0, n):
            for prime in primes:
                if prime != 1 and (prime >= n or n % prime == 0):
                    continue
                r = O.polygon_batch(p, np.array([0, n]), offset_prime=[off, prime], want_stats=True)
                out[f"{off},{prime}"] = {
                    "ids": r["ids"].tolist(), "status": int(r["status"][0]),
                    "bbox_bits": r["bbox"].view(np.uint32)[0].tolist(), "nodes": r["stats"]["nodes"],
                    "vtx_sha256": hashlib.sha256(r["vtx"].tobytes()).hexdigest(),
                }
        kat[name] = out
    json.dump(kat, open(os.path.join(HERE, "kat.json"), "w"), indent=1)
    print("golden written")


if __name__ == "__main__":
    write_heightmap_png() if sys.argv[1:] == ["png"] else main()
