#!/usr/bin/env python3
"""Writes tests/golden/opencl_test_crop.octree2 and opencl_test_camera.json from the reference's benchmark scene.

  python scripts/make_octree2_fixture.py <reference checkout> [out dir]

The scene file (benchmark/OpenCL_test/OpenCL_test.octree2, 1.3 MB) is too large to keep in the repository, so the
fixture keeps what the loader has to parse - the header and all 3091 block-palette NBT compounds, byte for byte - and
crops the world and water octrees to the 128^3 cell in which most of the benchmark camera's first hits lie
(x 512..639, y 0..127, z 384..511): every subtree outside that cell becomes one air leaf, the tree keeps its depth of 10.
The scene description is cut down to the fields camera_from_json reads.
"""
import gzip
import json
import os
import struct
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from chunkyclplugin_b200 import octree2  # noqa: E402

KEEP_LO, KEEP_HI = (512, 0, 384), (640, 128, 512)


def crop(tree: np.ndarray, depth: int, air: int):
    """Pre-order stream of ``tree`` with every node outside the kept box replaced by an air leaf."""
    out = []
    todo = [(0, 0, 0, 0, 1 << depth)]
    while todo:
        at, x, y, z, size = todo.pop()
        inside = all(lo < c + size and c < hi for c, lo, hi in zip((x, y, z), KEEP_LO, KEEP_HI))
        w = int(tree[at])
        if not inside:
            out.append(air)
        elif w > 0:
            out.append(octree2.BRANCH)
            h = size // 2
            for i in range(7, -1, -1):            # child i = x<<2 | y<<1 | z, child 0 read first
                todo.append((w + i, x + h * (i >> 2), y + h * ((i >> 1) & 1), z + h * (i & 1), h))
        else:
            out.append(-w)
    return out


def main() -> int:
    ref = sys.argv[1]
    out_dir = sys.argv[2] if len(sys.argv) > 2 else os.path.join(ROOT, "tests", "golden")
    src = os.path.join(ref, "benchmark", "OpenCL_test")
    path = os.path.join(src, "OpenCL_test.octree2")
    o = octree2.load(path)
    raw = octree2._read_stream(path)
    pos = 12
    for _ in range(len(o.blocks)):
        _, pos = octree2._nbt_compound_body(raw, pos)
    air = next(i for i, b in enumerate(o.blocks) if b.get("Name") == "minecraft:air")
    body = bytearray(raw[:pos])
    for depth, tree in ((o.world_depth, o.world), (o.water_depth, o.water)):
        body += struct.pack(">i", depth) + np.asarray(crop(tree, depth, air), dtype=">i4").tobytes()
    with gzip.GzipFile(os.path.join(out_dir, "opencl_test_crop.octree2"), "wb", compresslevel=9, mtime=0) as f:
        f.write(bytes(body))
    d = json.loads(open(os.path.join(src, "OpenCL_test.json"), "rb").read().decode("latin-1"))
    with open(os.path.join(out_dir, "opencl_test_camera.json"), "w") as f:
        json.dump({"chunkList": d["chunkList"], "yMin": d.get("yMin", 0), "camera": d["camera"]}, f)
    print({k: v for k, v in octree2.load(os.path.join(out_dir, "opencl_test_crop.octree2")).stats().items()})
    return 0


if __name__ == "__main__":
    sys.exit(main())
