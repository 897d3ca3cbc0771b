"""CCU_RENDER_BIOME_TINT on the CPU (DESIGN.md §13): the .octree2 biome section, the commit-time layout against a numpy
restatement, and the CPU restatement (specular_oracle.FlagsOracle) against the flag-off image and against closed-form pixels."""
import dataclasses
import gzip
import os

import numpy as np
import pytest

from chunkyclplugin_b200 import native, octree2
from chunkyclplugin_b200 import scenes as S
import specular_oracle as SO

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
BIOME = 512
FIXED = (0xFF71A74D, 0xFF8EB971, 0xFF3F76E4)   # the fixed tints of tint types 1, 2, 3 (material.h:61-72)


def crop_with_biomes():
    o = octree2.load(os.path.join(GOLDEN, "opencl_test_crop.octree2"))
    o.biomes = octree2.read_biomes(gzip.decompress(open(os.path.join(GOLDEN, "opencl_test_crop_biomes.bin.gz"), "rb").read()), 0)
    return o


def argb_floats(argb):
    return np.array([(argb >> 16) & 0xFF, (argb >> 8) & 0xFF, argb & 0xFF], np.float32) / np.float32(256)


def fixed_tint_biome(p, holes=0.0):
    """Biome colours whose every texel of plane k holds the fixed tint of tint type k + 1."""
    chunks, _ = S.with_biomes(p, holes=holes).biome
    rgb = np.empty((chunks.shape[0], 3, 256, 3), np.float32)
    for k in range(3):
        rgb[:, k] = argb_floats(FIXED[k])
    return chunks, rgb


# ------------------------------------------------------------------------------------------------------------------------
# loader
# ------------------------------------------------------------------------------------------------------------------------
def test_crop_fixture_has_no_biomes():
    assert octree2.load(os.path.join(GOLDEN, "opencl_test_crop.octree2")).biomes is None


def test_crop_biome_section():
    o = crop_with_biomes()
    assert list(o.biomes) == ["grass", "foliage", "water"]
    means = {"grass": (0.19, 0.54, 0.10), "foliage": (0.10, 0.43, 0.03), "water": (0.05, 0.18, 0.78)}
    for name, (chunks, rgb) in o.biomes.items():
        # the crop's chunks x 32..39, z 24..31; the scene has no chunk row z = 31
        assert chunks.shape == (56, 2) and rgb.shape == (56, 256, 3)
        assert set(map(tuple, chunks)) == {(x, z) for x in range(32, 40) for z in range(24, 31)}
        np.testing.assert_allclose(rgb.reshape(-1, 3).mean(0), means[name], atol=0.03)


def test_biome_save_load_round_trip(tmp_path):
    o = crop_with_biomes()
    path = str(tmp_path / "b.octree2")
    octree2.save(path, o.blocks, o.world_depth, o.world, o.water_depth, o.water, biomes=o.biomes)
    r = octree2.load(path)
    np.testing.assert_array_equal(r.world, o.world)
    for name in octree2.BIOME_TEXTURES:
        np.testing.assert_array_equal(r.biomes[name][0], o.biomes[name][0])
        np.testing.assert_array_equal(r.biomes[name][1], o.biomes[name][1])


@pytest.mark.parametrize("cut", [1, 4, 9, 8 + 3072 + 5, 4 + 3 * (8 + 3072) - 1])
def test_truncated_biome_section_raises(tmp_path, cut):
    o = crop_with_biomes()
    section = octree2.write_biomes({k: (v[0][:1], v[1][:1]) for k, v in o.biomes.items()})
    assert octree2.read_biomes(section, 0) is not None
    with pytest.raises(ValueError):
        octree2.read_biomes(section[:len(section) - cut], 0)


def test_biome_tints_assign_tint_types():
    o = crop_with_biomes()
    plain = octree2.to_scene(o, 32, 18)
    tinted = octree2.to_scene(o, 32, 18, biome_tints=True)
    assert plain.biome is None
    np.testing.assert_array_equal(plain.mat_palette, octree2.to_scene(crop_with_biomes(), 32, 18).mat_palette)
    want = {"grass_block": 2, "short_grass": 2, "grass": 2, "tall_grass": 2, "fern": 2, "large_fern": 2, "sugar_cane": 2,
            "oak_leaves": 1, "jungle_leaves": 1, "acacia_leaves": 1, "dark_oak_leaves": 1, "mangrove_leaves": 1, "vine": 1,
            "water": 3}
    seen = set()
    for i, blk in enumerate(o.blocks):
        name = str(blk.get("Name", "")).split(":", 1)[-1]
        if str(blk.get("Name")) in octree2._INVISIBLE:
            continue
        bp = tinted.block_palette
        # palette entries are added in block order: the i-th visible block's material
        ptr = [bp[b + 1] for b in range(2, bp.size, 2)][sum(1 for b in o.blocks[:i] if str(b.get("Name")) not in octree2._INVISIBLE)]
        tt = (int(tinted.mat_palette[ptr + 1]) & 0xFFFFFFFF) >> 24
        assert tt == want.get(name, 0), name
        if tt:
            seen.add(tt)
            assert int(tinted.mat_palette[ptr + 3]) & 0xFFFFFF == 0xC8C8C8
    assert seen == {1, 2, 3}
    chunks, rgb = tinted.biome
    assert rgb.shape == (56, 3, 256, 3)
    for k, name in enumerate(("foliage", "grass", "water")):
        np.testing.assert_array_equal(rgb[:, k], o.biomes[name][1])


# ------------------------------------------------------------------------------------------------------------------------
# commit-time layout
# ------------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("depth", [3, 8, 11])
@pytest.mark.parametrize("holes", [0.0, 0.4])
def test_debug_biome_layout_matches_numpy(depth, holes):
    n = max(1, (1 << depth) // 16)
    chunks = np.stack(np.meshgrid(np.arange(n), np.arange(n), indexing="ij"), -1).reshape(-1, 2)
    chunks = chunks[S.hash_u32(chunks[:, 0], chunks[:, 1], depth) / 2.0 ** 32 >= holes]
    if depth == 11:
        chunks = chunks[::97]                       # a spread of the 16384 chunks
    chunks = chunks.astype(np.int32)
    rgb = S.biome_field(chunks, seed=depth)
    got = native.debug_biome_layout(chunks, rgb, depth)
    want = SO.biome_layout(chunks, rgb, depth)
    assert (got["x0"], got["z0"]) == (want["x0"], want["z0"]) == tuple(int(v) for v in chunks.min(0))
    assert got["grid"].shape == tuple(int(v) for v in chunks.max(0) - chunks.min(0) + 1)
    np.testing.assert_array_equal(got["grid"], want["grid"])
    np.testing.assert_array_equal(got["tiles"].view(np.uint32), want["tiles"].view(np.uint32))
    assert (got["grid"] >= 0).sum() == chunks.shape[0]


def test_debug_biome_layout_rejects():
    rgb = np.ones((1, 3, 256, 3), np.float32)
    for chunk, depth in (((1, 0), 3), ((0, 16), 8), ((128, 3), 11)):
        with pytest.raises(native.ChunkyCuError, match="outside"):
            native.debug_biome_layout([chunk], rgb, depth)
        with pytest.raises(ValueError):
            SO.biome_layout([chunk], rgb, depth)
    with pytest.raises(native.ChunkyCuError, match="negative coordinate"):
        native.debug_biome_layout([(-1, 0)], rgb, 8)
    with pytest.raises(native.ChunkyCuError, match="twice"):
        native.debug_biome_layout([(2, 3), (2, 3)], np.ones((2, 3, 256, 3), np.float32), 8)
    for bad in (np.nan, np.inf, -1e-30):
        r = rgb.copy()
        r[0, 2, 17, 1] = bad
        with pytest.raises(native.ChunkyCuError, match="component"):
            native.debug_biome_layout([(0, 0)], r, 8)
    b = native.debug_biome_layout(np.zeros((0, 2), np.int32), np.zeros((0, 3, 256, 3), np.float32), 8)
    assert b["grid"].size == 0 and b["tiles"].shape[0] == 0


def test_deep_sparse_biome_layout():
    """The grid covers the chunks' bounding box, not the octree: a few chunks of a depth-30 octree lay out in a small grid, and
    chunks spread wider than 2^24 chunks are refused with an error (not an abort)."""
    rgb = S.biome_field(np.array([[0, 0], [1, 1]], np.int32))
    top = (1 << 26) - 1
    for chunks in ([[top, top], [top - 3, top - 1]], [[5, 1 << 20], [7, (1 << 20) + 9]]):
        got = native.debug_biome_layout(np.array(chunks, np.int32), rgb, 30)
        want = SO.biome_layout(chunks, rgb, 30)
        assert got["grid"].shape == want["grid"].shape and got["grid"].size <= 40
        np.testing.assert_array_equal(got["grid"], want["grid"])
        assert (got["x0"], got["z0"]) == (want["x0"], want["z0"])
    for chunks in ([[0, 0], [top, top]], [[0, 0], [4096, 4096]]):
        with pytest.raises(native.ChunkyCuError, match="span more than") as e:
            native.debug_biome_layout(np.array(chunks, np.int32), rgb, 30)
        assert e.value.code == native.CCU_EINVAL
        with pytest.raises(ValueError):
            SO.biome_layout(chunks, rgb, 30)
    native.debug_biome_layout(np.array([[0, 0], [4095, 4095]], np.int32), rgb, 30)   # 2^24 cells: the largest grid


def test_biome_planes_with_different_chunk_sets():
    """A chunk that one texture lacks gets that plane filled with the fixed tint's floats."""
    o = crop_with_biomes()
    keep = {"grass": slice(0, 40), "foliage": slice(10, 56), "water": slice(0, 0)}
    part = {k: (c[keep[k]], t[keep[k]]) for k, (c, t) in o.biomes.items()}
    chunks, rgb = octree2.biome_planes(part)
    assert chunks.shape == (56, 2) and len({tuple(c) for c in chunks}) == 56
    at = {tuple(c): i for i, c in enumerate(chunks)}
    for k, (name, fixed) in enumerate((("foliage", FIXED[0]), ("grass", FIXED[1]), ("water", FIXED[2]))):
        c, t = part[name]
        have = {tuple(x) for x in c}
        for i, x in enumerate(c):
            np.testing.assert_array_equal(rgb[at[tuple(x)], k], t[i])
        for x, i in at.items():
            if x not in have:
                assert (rgb[i, k] == argb_floats(fixed)).all()


# ------------------------------------------------------------------------------------------------------------------------
# CPU restatement
# ------------------------------------------------------------------------------------------------------------------------
def _render(p, flags, seeds=(11, 22), **kw):
    return SO.FlagsOracle(p, flags, **kw).render(list(seeds))


@pytest.fixture(scope="module")
def lit_decorated():
    """Decorated terrain (foliage quads, grass cubes) with a water tint and emitting grass, small canvas."""
    p = S.water_tinted(S.terrain_scene(64, 48, 27, seed=11, decorate=True))
    mp = p.mat_palette.copy()
    for i in range(mp.size // 6):
        if (int(mp[6 * i + 1]) >> 24) == 2:
            mp[6 * i + 4] = 200          # grass emits: the NEE samplers evaluate a tinted material
    return dataclasses.replace(p, mat_palette=mp)


def test_flag_without_biomes_is_flag_off(lit_decorated):
    assert lit_decorated.biome is None
    for extra in (0, 8):
        a = _render(lit_decorated, extra)
        b = _render(lit_decorated, extra | BIOME)
        np.testing.assert_array_equal(a.view(np.uint32), b.view(np.uint32))


@pytest.mark.parametrize("extra", [0, 4, 8, 8 | 128, 8 | 256 | 128])
def test_fixed_tint_colours_render_as_flag_off(lit_decorated, extra):
    p = dataclasses.replace(lit_decorated, biome=fixed_tint_biome(lit_decorated, holes=0.3))
    p = S.glossy(p) if extra & 4 else p
    a = _render(p, extra)
    b = _render(p, extra | BIOME)
    np.testing.assert_array_equal(a.view(np.uint32), b.view(np.uint32))
    # real colours change the image
    q = S.with_biomes(p, holes=0.3)
    assert not np.array_equal(_render(q, extra | BIOME), a)


def floor_scene(width=64, height=48):
    """A 64^3 world whose only blocks are a floor (y = 0) of flat, emissive, grass-tinted cubes, seen from above; no sun, a
    black sky."""
    pal = S.Palettes()
    m = pal.put_material(S.pack_material(0, 0, emittance=1.0, tint=2 << 24, textured=False, argb=S._s32(0xFFC0C0C0)))
    pal.blocks += [1, m]
    types = np.zeros((64, 64, 64), np.int32)
    types[:, 0, :] = 1
    tree, depth = S.build_octree(types, np.array([0, len(pal.blocks) - 2]))
    cam = S.pinhole_camera((30.3, 7.7, 33.2), 30.0, -90.0, 70.0)
    p = S._finish("floor", tree, depth, pal, cam, width, height, sun_draw=False)
    return dataclasses.replace(S.with_biomes(p, seed=5, holes=0.25), sky=np.zeros_like(p.sky))


def floor_expected(p):
    """Per pixel: the closed-form value (col * em * scale) * col of the one column the pixel's footprint lies in, or NaN where
    the footprint straddles columns."""
    cam = np.asarray(p.camera, np.float64)
    o, M = cam[0:3], cam[3:12].reshape(3, 3)
    hw, ih = p.width / (2.0 * p.height), 1.0 / p.height
    px, py = np.meshgrid(np.arange(p.width), np.arange(p.height))
    cols = []
    for jx, jy in ((0, 0), (1, 0), (0, 1), (1, 1)):
        x = -hw + (px + jx) * ih
        y = -0.5 + (py + jy) * ih
        d = np.stack([cam[14] * x, cam[14] * y, np.ones_like(x)], -1) @ M.T
        assert (d[..., 1] < 0).all()
        t = (1.0 - o[1]) / d[..., 1]
        cols.append((o[0] + t * d[..., 0], o[2] + t * d[..., 2]))
    cx = np.floor(np.stack([c[0] for c in cols]))
    cz = np.floor(np.stack([c[1] for c in cols]))
    one = (cx.min(0) == cx.max(0)) & (cz.min(0) == cz.max(0)) & (cx[0] >= 0) & (cx[0] < 64) & (cz[0] >= 0) & (cz[0] < 64)
    chunks, rgb = p.biome
    tile = {(int(a), int(b)): i for i, (a, b) in enumerate(chunks)}
    base = np.float32(192) / np.float32(256)
    out = np.full((p.height, p.width, 3), np.nan, np.float32)
    for j, i in zip(*np.nonzero(one)):
        x, z = int(cx[0, j, i]), int(cz[0, j, i])
        k = tile.get((x >> 4, z >> 4))
        c = rgb[k, 1, (z & 15) * 16 + (x & 15)] if k is not None else argb_floats(FIXED[1])
        col = base * c.astype(np.float32)
        out[j, i] = (col * (np.float32(1.0) * np.float32(13.0))) * col
    return out.reshape(-1)


def test_floor_matches_closed_form():
    p = floor_scene()
    want = floor_expected(p)
    got = SO.FlagsOracle(p, BIOME, max_depth=1).render([5])
    ok = ~np.isnan(want)
    assert ok.sum() > 0.4 * want.size
    np.testing.assert_array_equal(got[ok].view(np.uint32), want[ok].view(np.uint32))
    # the hole chunks keep the fixed tint, and the field varies along both axes
    assert len(np.unique(want[ok])) > 100
