"""`.octree2` loader (SURVEY 8f #4): round trip on a synthetic file, a crop of the reference's benchmark scene."""
import os

import numpy as np
import pytest

from chunkyclplugin_b200 import native, octree2
from chunkyclplugin_b200.javarandom import pass_seeds

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def _synthetic_file(tmp_path, scenes):
    """A terrain octree written as an .octree2 file: palette indices instead of block pointers (pointer = 2 * index)."""
    p = scenes("terrain64")
    tree = np.asarray(p.octree, dtype=np.int64).copy()
    leaf = tree <= 0
    tree[leaf] = -((-tree[leaf]) // 2)
    names = ["minecraft:air", "minecraft:stone", "minecraft:dirt", "minecraft:grass_block", "minecraft:sand", "minecraft:glowstone",
             "minecraft:glass", "minecraft:cave_air", "minecraft:oak_log"]
    blocks = [{"Name": n} for n in names]
    blocks[8] = {"Name": "minecraft:oak_log", "Properties": {"axis": "y"}}
    path = str(tmp_path / "synthetic.octree2")
    octree2.save(path, blocks, p.octree_depth, tree)
    return path, p, tree, blocks


def test_round_trip(tmp_path, scenes):
    path, p, tree, blocks = _synthetic_file(tmp_path, scenes)
    o = octree2.load(path)
    assert (o.version, o.palette_version, o.world_depth) == (6, 4, p.octree_depth)
    assert o.blocks == blocks
    # the packed arrays differ in child-block order only: compare through the pre-order stream and leaf lookups
    assert octree2.write_preorder(o.world) == octree2.write_preorder(tree)
    rng = np.random.default_rng(1)
    xyz = rng.integers(0, 1 << p.octree_depth, size=(20000, 3))
    a = native.layout_lookup(np.where(o.world <= 0, o.world * 2, o.world).astype(np.int32), p.octree_depth, xyz)
    b = native.layout_lookup(np.asarray(p.octree, dtype=np.int32), p.octree_depth, xyz)
    assert np.array_equal(a["wide_value"], b["wide_value"]) and np.array_equal(a["wide_level"], b["wide_level"])
    assert o.stats()["nodes"] == tree.size


def test_scene_from_file_renders_like_the_source_scene_geometry(tmp_path, scenes):
    """Same voxels, flat-colour palette: the first-hit geometry (distance, normal) equals the source scene's."""
    import oracle
    path, p, _, _ = _synthetic_file(tmp_path, scenes)
    s = octree2.to_scene(octree2.load(path), p.width, p.height, camera=p.camera)
    assert s.octree_depth == p.octree_depth and s.block_palette[0] == 0
    seed = pass_seeds(1)[0]
    a, b = oracle.Oracle(s).first_hit(seed), oracle.Oracle(p).first_hit(seed)
    # glass (alpha-tested in the source scene) is opaque here; everywhere else the geometry agrees
    same = a["kind"] == b["kind"]
    assert same.mean() > 0.95
    assert np.array_equal(a["t"][same & (b["kind"] > 0)].view(np.uint32), b["t"][same & (b["kind"] > 0)].view(np.uint32))


def test_bad_files(tmp_path):
    bad = tmp_path / "bad.octree2"
    bad.write_bytes(b"\x00\x00\x00\x03\x00\x00\x00\x01\x00\x00\x00\x00")
    with pytest.raises(ValueError):
        octree2.load(str(bad))
    with pytest.raises(ValueError):
        octree2.pack_preorder(np.array([-1, 0, 0], dtype=np.int32))     # branch with missing children


def test_reference_benchmark_scene():
    """The reference's own fixture (benchmark/OpenCL_test), cropped by scripts/make_octree2_fixture.py to one 128^3 cell:
    its header and 3091 palette NBT compounds verbatim, world and water trees of depth 10 with air outside the cell."""
    import oracle
    path = os.path.join(GOLD, "opencl_test_crop.octree2")
    o = octree2.load(path)
    st = o.stats()
    assert (o.version, o.palette_version, len(o.blocks)) == (6, 4, 3091)
    assert st == {"nodes": 255249, "branches": 31906, "any_type_leaves": 23887, "leaf_types": 817, "depth": 10,
                  "water_nodes": 6177, "water_depth": 10}
    assert 1 + 8 * st["branches"] == st["nodes"]
    s = octree2.load_scene(path, os.path.join(GOLD, "opencl_test_camera.json"), 160, 90)
    # commit-time layouts against the root descent on the real scene (depth 10, ANY_TYPE leaves), in and around the cell
    from test_layouts import root_descent
    rng = np.random.default_rng(2)
    xyz = np.stack([rng.integers(448, 704, 100000), rng.integers(0, 192, 100000), rng.integers(320, 576, 100000)], -1)
    tree = np.asarray(s.octree, dtype=np.int32)
    want_value, want_level = root_descent(tree, 10, xyz)
    got = native.layout_lookup(tree, 10, xyz)
    assert np.array_equal(got["wide_value"], want_value) and np.array_equal(got["wide_level"], want_level)
    assert np.array_equal(got["air_solid"] == 0, want_value == 0)
    fh = oracle.Oracle(s).first_hit(1)
    assert (fh["kind"] > 0).mean() > 0.3


@pytest.mark.gpu
def test_cuda_renders_a_loaded_file(tmp_path, scenes, cuda_ctx):
    import oracle
    from conftest import load_scene
    path, p, _, _ = _synthetic_file(tmp_path, scenes)
    s = octree2.to_scene(octree2.load(path), p.width, p.height, camera=p.camera)
    load_scene(cuda_ctx, s)
    seeds = pass_seeds(3)
    cuda_ctx.render_passes(seeds)
    got, _ = cuda_ctx.render_read()
    assert np.array_equal(got.view(np.uint32), oracle.Oracle(s).render(seeds).view(np.uint32))
