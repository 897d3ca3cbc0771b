"""CCU_RENDER_BIOME_TINT on the device: both render kernels against the CPU restatement (FlagsOracle) bit for bit, alone and
with the specular and emitter-sampling flags; kernel selection; the fixed-tint equivalence at 1080p; the closed-form floor;
the setter and commit checks; one group case; the loaded .octree2 crop with its biome section."""
import dataclasses
import os

import numpy as np
import pytest

from chunkyclplugin_b200 import native, octree2
from chunkyclplugin_b200 import scenes as S
from chunkyclplugin_b200.javarandom import pass_seeds
from chunkyclplugin_b200.renderer import upload_scene
from oracle import edge_rays as E
from test_biome_tint import crop_with_biomes, fixed_tint_biome, floor_expected, floor_scene
from test_gpu_specular import assert_bits
from test_oracle_edge_rays import E_PASSES, EDGE

import specular_oracle as SO

pytestmark = pytest.mark.gpu
BIOME, SPEC, NEE, NEAR, MODELS = 512, 4, 8, 128, 256
FLAGS = [BIOME, BIOME | SPEC, BIOME | NEE, BIOME | NEE | NEAR, BIOME | NEE | MODELS, BIOME | NEE | MODELS | NEAR]


def load_biome_scene(ctx, p):
    """Upload a PackedScene with its biome colours (set before commit), camera and canvas."""
    upload_scene(ctx, p)
    ctx.camera_set(p.projector_type, p.camera)
    ctx.render_begin(p.width, p.height)


def _render(ctx, p, seeds, kernel, flags, max_depth=5):
    ctx.render_set_params(kernel=kernel, flags=flags, max_depth=max_depth)
    try:
        ctx.render_begin(p.width, p.height)
        ctx.render_passes(np.asarray(seeds, np.int32))
        return ctx.render_read()[0]
    finally:
        ctx.render_set_params()


def emitting_tints(p):
    """p with its grass-tinted materials emitting (a tinted full-cube emitter) and its model materials emissive (the foliage-
    tinted CROSS quads of decorated terrain become tinted model emitters)."""
    p = S.emissive_models(p)
    mp = p.mat_palette.copy()
    for i in range(mp.size // 6):
        if (int(mp[6 * i + 1]) >> 24) == 2:
            mp[6 * i + 4] = 180
    return dataclasses.replace(p, mat_palette=mp)


def _scene(scenes, name):
    if name == "terrain64":
        return S.with_biomes(scenes("terrain64"), seed=1)
    if name == "decorated":
        return S.with_biomes(emitting_tints(scenes("decorated")), seed=2)
    if name == "water":
        return S.with_biomes(S.water_tinted(scenes("terrain64")), seed=3)
    if name == "tiny8":
        return S.with_biomes(S.water_tinted(scenes("tiny8")), seed=4, holes=0.0)
    if name == "large2048":
        return S.with_biomes(S.water_tinted(scenes("large2048")), seed=5, holes=0.9)
    if name == "entities":
        return S.with_biomes(S.water_tinted(scenes("entities")), seed=6)
    raise KeyError(name)


SCENES = ["terrain64", "decorated", "water", "tiny8", "large2048", "entities"]


@pytest.mark.parametrize("flags", FLAGS)
@pytest.mark.parametrize("name", SCENES)
def test_kernels_match_the_oracle(scenes, cuda_ctx, name, flags):
    p = _scene(scenes, name)
    if flags & SPEC:
        p = S.glossy(p)
    seeds = pass_seeds(3)
    want = SO.FlagsOracle(p, flags).render(seeds)
    load_biome_scene(cuda_ctx, p)
    for kernel in (4, 1):
        assert_bits(_render(cuda_ctx, p, seeds, kernel, flags), want)


@pytest.mark.parametrize("flags", [BIOME, BIOME | NEE | MODELS | NEAR])
@pytest.mark.parametrize("name", EDGE)
def test_edge_rays(cuda_ctx, name, flags):
    p = S.with_biomes(S.water_tinted(E.scenes()[name]), seed=9)
    seeds = pass_seeds(E_PASSES)
    want = SO.FlagsOracle(p, flags).render(seeds)
    load_biome_scene(cuda_ctx, p)
    for kernel in (4, 1):
        assert_bits(_render(cuda_ctx, p, seeds, kernel, flags), want)


def test_biomes_change_the_image(scenes, cuda_ctx):
    p = _scene(scenes, "decorated")
    seeds = pass_seeds(2)
    load_biome_scene(cuda_ctx, p)
    for kernel in (4, 1):
        assert not np.array_equal(_render(cuda_ctx, p, seeds, kernel, BIOME), _render(cuda_ctx, p, seeds, kernel, 0))


def test_flag_on_without_biomes_is_flag_off(scenes, cuda_ctx):
    p = emitting_tints(scenes("decorated"))
    seeds = pass_seeds(3)
    load_biome_scene(cuda_ctx, p)
    for kernel in (4, 1, 0):
        for extra in (0, NEE | NEAR):
            assert_bits(_render(cuda_ctx, p, seeds, kernel, BIOME | extra), _render(cuda_ctx, p, seeds, kernel, extra))


def test_flag_off_with_biomes_is_flag_off(scenes, cuda_ctx):
    """Biome colours change nothing while the flag is off."""
    p = emitting_tints(scenes("decorated"))
    seeds = pass_seeds(3)
    load_biome_scene(cuda_ctx, p)
    off = {(k, f): _render(cuda_ctx, p, seeds, k, f) for k in (4, 1) for f in (0, NEE)}
    load_biome_scene(cuda_ctx, S.with_biomes(p, seed=2))
    for (k, f), want in off.items():
        assert_bits(_render(cuda_ctx, p, seeds, k, f), want)


def test_fixed_tint_colours_at_1080p(cuda_ctx):
    """Config 1 at 1920 x 1080, 16 passes: biome colours equal to the fixed tints render as flag off on both kernels."""
    p = S.water_tinted(S.terrain_scene(256, 1920, 1080))
    p = dataclasses.replace(p, biome=fixed_tint_biome(p, holes=0.2))
    seeds = pass_seeds(16)
    load_biome_scene(cuda_ctx, p)
    for kernel in (4, 1):
        assert_bits(_render(cuda_ctx, p, seeds, kernel, BIOME), _render(cuda_ctx, p, seeds, kernel, 0))


def test_floor_matches_closed_form(cuda_ctx):
    p = floor_scene()
    want = floor_expected(p)
    ok = ~np.isnan(want)
    load_biome_scene(cuda_ctx, p)
    for kernel in (4, 1):
        got = _render(cuda_ctx, p, [5], kernel, BIOME, max_depth=1)
        np.testing.assert_array_equal(got[ok].view(np.uint32), want[ok].view(np.uint32))


def test_loaded_crop_with_biomes(cuda_ctx):
    p = octree2.to_scene(crop_with_biomes(), 96, 54, camera=octree2.camera_from_json(
        os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "opencl_test_camera.json")), biome_tints=True)
    assert p.biome is not None
    seeds = pass_seeds(2)
    want = SO.FlagsOracle(p, BIOME).render(seeds)
    load_biome_scene(cuda_ctx, p)
    for kernel in (4, 1):
        assert_bits(_render(cuda_ctx, p, seeds, kernel, BIOME), want)


# ------------------------------------------------------------------------------------------------------------------------
# ABI
# ------------------------------------------------------------------------------------------------------------------------
def test_setter_rejections(cuda_ctx):
    lib, h = native.load(), cuda_ctx._h
    rgb = np.ones((2, 3, 256, 3), np.float32)
    assert lib.ccu_scene_set_biome_colors(h, None, None, -1) == native.CCU_EINVAL
    assert lib.ccu_scene_set_biome_colors(h, None, native._ptr(rgb), 1) == native.CCU_EINVAL
    assert lib.ccu_scene_set_biome_colors(h, native._ptr(np.zeros(2, np.int32)), None, 1) == native.CCU_EINVAL
    for chunks in ([(0, -1), (1, 1)], [(3, 4), (3, 4)]):
        with pytest.raises(native.ChunkyCuError) as e:
            cuda_ctx.set_biome_colors(chunks, rgb)
        assert e.value.code == native.CCU_EINVAL
    for bad in (np.nan, -np.inf, -0.5):
        r = rgb.copy()
        r[1, 0, 255, 2] = bad
        with pytest.raises(native.ChunkyCuError):
            cuda_ctx.set_biome_colors([(0, 0), (1, 0)], r)
    cuda_ctx.set_biome_colors(np.zeros((0, 2), np.int32), np.zeros((0, 3, 256, 3), np.float32))


def test_commit_rejects_a_chunk_outside_the_octree(scenes, cuda_ctx):
    p = scenes("terrain64")                           # depth 6: 4 x 4 chunks
    q = dataclasses.replace(p, biome=(np.array([[0, 0], [1, 4]], np.int32), np.ones((2, 3, 256, 3), np.float32)))
    with pytest.raises(native.ChunkyCuError, match=r"chunk 1 \(1, 4\)") as e:
        load_biome_scene(cuda_ctx, q)
    assert e.value.code == native.CCU_EINVAL
    load_biome_scene(cuda_ctx, p)


def test_scene_begin_clears_the_colours_and_device_bytes_grow(scenes, cuda_ctx):
    p = emitting_tints(scenes("decorated"))
    q = S.with_biomes(p, seed=2)
    seeds = pass_seeds(2)
    load_biome_scene(cuda_ctx, p)
    plain = cuda_ctx.scene_device_bytes()
    off = _render(cuda_ctx, p, seeds, 4, BIOME)
    load_biome_scene(cuda_ctx, q)
    b = native.debug_biome_layout(*q.biome, q.octree_depth)
    assert cuda_ctx.scene_device_bytes() == plain + max(b["grid"].size, 16) * 4 + b["tiles"].shape[0] * 3 * 256 * 16
    assert not np.array_equal(_render(cuda_ctx, q, seeds, 4, BIOME), off)
    load_biome_scene(cuda_ctx, p)                     # scene_begin drops the colours; p sets none
    assert cuda_ctx.scene_device_bytes() == plain
    assert_bits(_render(cuda_ctx, p, seeds, 4, BIOME), off)


def test_group_replicates_the_colours(scenes, cuda_ctx):
    if native.device_count() < 2:
        pytest.skip("needs two GPUs")
    p = _scene(scenes, "decorated")
    seeds = pass_seeds(4)
    flags = BIOME | NEE
    load_biome_scene(cuda_ctx, p)
    want = _render(cuda_ctx, p, seeds, 0, flags).astype(np.float64)
    group = native.Group(devices=[0, 1])
    try:
        m0 = group.member(0)
        load_biome_scene(m0, p)
        m0.render_end()
        group.replicate_scene()
        group.camera_set(p.projector_type, p.camera)
        group.render_set_params(flags=flags)
        group.render_begin(p.width, p.height)
        sb = np.zeros(p.width * p.height * 3, dtype=np.float64)
        group.render_passes(seeds)
        assert group.render_merge(sb, 0) == len(seeds)
        group.render_end()
        assert np.array_equal(sb, want)
    finally:
        group.close()
