"""CCU_RENDER_SPECULAR on the device: both render kernels against the CPU oracle bit for bit on glossy scenes (every
octree layout, with and without entity BVHs, sun on and off, DoF and pre-generated rays, ray depths 2 and 5, partial tiles),
on the edge-ray catalogue, at the BASELINE canvas, through the analytic mirror, and through the group API.  The launch picks
the specular kernels only when the flag is on and the scene has a specular word; the selection tests pin that."""
import dataclasses

import numpy as np
import pytest

from chunkyclplugin_b200 import scenes as S
from chunkyclplugin_b200.javarandom import pass_seeds
from conftest import load_scene
from oracle import edge_rays as E
from test_oracle_edge_rays import E_PASSES, EDGE
from test_specular import EMITTER_SCALE, assert_mirror, mirror_expectation, mirror_scene

pytestmark = pytest.mark.gpu


def _render(ctx, p, seeds, kernel, flags, max_depth=5, emitter_scale=13.0):
    ctx.render_set_params(kernel=kernel, flags=flags, max_depth=max_depth, emitter_scale=emitter_scale)
    try:
        ctx.render_begin(p.width, p.height)
        ctx.render_passes(np.asarray(seeds, np.int32))
        return ctx.render_read()[0]
    finally:
        ctx.render_set_params()


def _oracle(p, max_depth=5, specular=False):
    import oracle
    from specular_oracle import SpecularOracle
    return (SpecularOracle if specular else oracle.Oracle)(p, max_depth=max_depth)


def assert_bits(got, want):
    ok = E.same_bits_or_nan(got, want)
    assert ok.all(), np.unique(np.nonzero(~ok)[0] // 3)[:8]


def _pregenerated(p):
    """the scene's pinhole camera as pre-generated rays through the pixel centres"""
    return dataclasses.replace(p, projector_type=-1, camera=S.pregenerated_rays(p.camera, p.width, p.height))


# name -> (base scene, what it covers)
CASES = {
    "terrain64": ("terrain64", "full cubes, top table in shared memory"),
    "decorated": ("decorated", "AABB / quad models, alpha tests"),
    "mixed": ("mixed", "entity BVHs, DoF, emitters on triangles"),
    "mixed_odd": ("mixed", "partial tiles (97 x 55)"),
    "indoor": ("indoor", "sun flag off, emissive-specular ceilings"),
    "entities": ("entities", "larger BVHs"),
    "terrain128": ("terrain128", "odd octree depth"),
    "large512": ("large512", "depth 9: top table in global memory"),
    "large2048": ("large2048", "depth 11: deep-world layout"),
    "terrain64_rays": ("terrain64", "pre-generated rays"),
}


def _case(scenes, name):
    p = S.glossy(scenes(CASES[name][0]))
    if name == "mixed_odd":
        p = p.with_resolution(97, 55)
    if name == "terrain64_rays":
        p = _pregenerated(p)
    return p


@pytest.mark.parametrize("max_depth", [2, 5])
@pytest.mark.parametrize("sun", ["sun", "nosun"])
@pytest.mark.parametrize("name", list(CASES))
def test_kernels_match_the_oracle(scenes, cuda_ctx, name, sun, max_depth):
    p = _case(scenes, name)
    if sun == "nosun":
        p = E.without_sun(p)
    assert (p.mat_palette[5::6] != 0).any()
    seeds = pass_seeds(3)
    want = _oracle(p, max_depth=max_depth, specular=True).render(seeds)
    load_scene(cuda_ctx, p)
    for kernel in (4, 1):
        assert_bits(_render(cuda_ctx, p, seeds, kernel, 4, max_depth=max_depth), want)


@pytest.mark.parametrize("name", EDGE)
def test_edge_rays(cuda_ctx, name):
    p = S.glossy(E.scenes()[name])
    seeds = pass_seeds(E_PASSES)
    want = _oracle(p, specular=True).render(seeds)
    load_scene(cuda_ctx, p)
    assert_bits(_render(cuda_ctx, p, seeds, 4, 4), want)
    assert_bits(_render(cuda_ctx, p, seeds, 1, 4), want)


@pytest.mark.parametrize("name", ["terrain64", "mixed"])
def test_unused_specular_word_changes_nothing(scenes, cuda_ctx, name):
    """The only specular word sits on a material no surface uses: the flag launches the specular kernels (the scene has a
    word), and their paths never meet an event."""
    p = scenes(name)
    p = dataclasses.replace(p, mat_palette=np.concatenate([p.mat_palette, S._i32(S.pack_material(0, 0, specular=0.9, metalness=0.5))]))
    seeds = pass_seeds(3)
    load_scene(cuda_ctx, p)
    for kernel in (4, 1):
        off = _render(cuda_ctx, p, seeds, kernel, 0)
        assert_bits(_render(cuda_ctx, p, seeds, kernel, 4), off)
    assert_bits(off, _oracle(p).render(seeds))


@pytest.mark.parametrize("name", ["decorated", "mixed"])
def test_flag_off_ignores_the_words(scenes, cuda_ctx, name):
    g = S.glossy(scenes(name))
    seeds = pass_seeds(3)
    load_scene(cuda_ctx, g)
    got = {k: _render(cuda_ctx, g, seeds, k, 0) for k in (4, 1)}
    load_scene(cuda_ctx, scenes(name))
    for k in (4, 1):
        assert_bits(got[k], _render(cuda_ctx, scenes(name), seeds, k, 0))


def test_baseline_canvas(cuda_ctx):
    """BASELINE config 1 geometry with glossy materials at 1920 x 1080, checked on every 64th pixel."""
    p = S.glossy(S.terrain_scene(256, 1920, 1080))
    seeds = pass_seeds(2)
    gids = np.arange(0, p.width * p.height, 64, dtype=np.int32)
    want = _oracle(p, specular=True).render(seeds, gids=gids).reshape(-1, 3)[gids]
    load_scene(cuda_ctx, p)
    for kernel in (4, 1):
        got = _render(cuda_ctx, p, seeds, kernel, 4).reshape(-1, 3)[gids]
        assert_bits(got, want)


@pytest.mark.parametrize("metal", [False, True], ids=["white_mirror", "metal_mirror"])
def test_analytic_mirror(cuda_ctx, metal):
    p = mirror_scene(metal)
    want, _, _ = mirror_expectation(p, metal)
    load_scene(cuda_ctx, p)
    for kernel in (4, 1):
        assert_mirror(_render(cuda_ctx, p, pass_seeds(1), kernel, 4, max_depth=2, emitter_scale=EMITTER_SCALE), want)


def _group_render(group, p, seeds):
    m0 = group.member(0)
    load_scene(m0, p)
    m0.render_end()
    group.replicate_scene()
    group.camera_set(p.projector_type, p.camera)
    group.render_set_params(flags=4)
    group.render_begin(p.width, p.height)
    sb = np.zeros(p.width * p.height * 3, dtype=np.float64)
    group.render_passes(seeds)
    assert group.render_merge(sb, 0) == len(seeds)
    group.render_end()
    return sb


def test_group_of_one_matches_a_context(scenes, cuda_ctx):
    from chunkyclplugin_b200 import native
    p = S.glossy(scenes("mixed"))
    seeds = pass_seeds(4)
    load_scene(cuda_ctx, p)
    want = _render(cuda_ctx, p, seeds, 0, 4).astype(np.float64)
    group = native.Group(devices=[0])
    try:
        assert np.array_equal(_group_render(group, p, seeds), want)
    finally:
        group.close()


def test_two_gpu_group_matches_one_gpu(scenes, cuda_ctx):
    from chunkyclplugin_b200 import native
    if native.device_count() < 2:
        pytest.skip("NEEDS 2 GPUs - the 2-GPU group path is not exercised on this box")
    p = S.glossy(scenes("mixed"))
    seeds = pass_seeds(6)
    load_scene(cuda_ctx, p)
    want = _render(cuda_ctx, p, seeds, 0, 4).astype(np.float64)
    group = native.Group(devices=[0, 1])
    try:
        assert np.allclose(_group_render(group, p, seeds), want, rtol=2e-6, atol=1e-7)
    finally:
        group.close()
