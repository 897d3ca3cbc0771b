#!/usr/bin/env python3
"""Writes tests/golden/opencl_test_crop.octree2 and opencl_test_camera.json from the reference's benchmark scene.

  python scripts/make_octree2_fixture.py <reference checkout> [out dir]
  python scripts/make_octree2_fixture.py --biomes <reference checkout> [out dir]

The scene file (benchmark/OpenCL_test/OpenCL_test.octree2, 1.3 MB) is too large to keep in the repository, so the
fixture keeps what the loader has to parse - the header and all 3091 block-palette NBT compounds, byte for byte - and
crops the world and water octrees to the 128^3 cell in which most of the benchmark camera's first hits lie
(x 512..639, y 0..127, z 384..511): every subtree outside that cell becomes one air leaf, the tree keeps its depth of 10.
The scene description is cut down to the fields camera_from_json reads.

--biomes writes tests/golden/opencl_test_crop_biomes.bin.gz instead: the file's biome colour section (grass, foliage and water
textures in that order, octree2.read_biomes) restricted to the chunks of the same cell, cx 32..39 and cz 24..31, byte for byte
in the file's format.  The scene's chunk list ends at cz = 30, so chunk row cz = 31 has no tiles.  Texel order: across the x
seam of two neighbouring tiles the colours step by 0 on average (all three textures) when texel = (z & 15) * 16 + (x & 15), and
by 1.4e-4 (grass) when texel = (x & 15) * 16 + (z & 15); the script checks the first.  The scene is nearly one biome, so
this is weak evidence, but it agrees with Chunky's BiomeStructure layout.
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


def seam_step(chunks: np.ndarray, rgb: np.ndarray) -> float:
    """Mean |colour step| across the x seams of neighbouring tiles, reading texel (z & 15) * 16 + (x & 15)."""
    at = {(int(c[0]), int(c[1])): i for i, c in enumerate(chunks)}
    steps = [np.abs(rgb[j].reshape(16, 16, 3)[:, 0] - rgb[i].reshape(16, 16, 3)[:, 15]).mean()
             for (cx, cz), i in at.items() if (j := at.get((cx + 1, cz))) is not None]
    return float(np.mean(steps))


def biomes_main(ref: str, out_dir: str) -> int:
    o = octree2.load(os.path.join(ref, "benchmark", "OpenCL_test", "OpenCL_test.octree2"))
    lo, hi = (KEEP_LO[0] >> 4, KEEP_LO[2] >> 4), (KEEP_HI[0] >> 4, KEEP_HI[2] >> 4)
    kept = {}
    for name, (chunks, rgb) in o.biomes.items():
        assert seam_step(chunks, rgb) == 0.0, name
        sel = (chunks[:, 0] >= lo[0]) & (chunks[:, 0] < hi[0]) & (chunks[:, 1] >= lo[1]) & (chunks[:, 1] < hi[1])
        kept[name] = (chunks[sel], rgb[sel])
    with gzip.GzipFile(os.path.join(out_dir, "opencl_test_crop_biomes.bin.gz"), "wb", compresslevel=9, mtime=0) as f:
        f.write(octree2.write_biomes(kept))
    print({k: int(v[0].shape[0]) for k, v in kept.items()})
    return 0


def main() -> int:
    if sys.argv[1] == "--biomes":
        return biomes_main(sys.argv[2], sys.argv[3] if len(sys.argv) > 3 else os.path.join(ROOT, "tests", "golden"))
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
