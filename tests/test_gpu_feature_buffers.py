"""The denoiser's feature buffers on the GPU (DESIGN.md §16): the 24 k_features instances against the CPU restatement
(FlagsOracle.features) bit for bit, with the instance each launch reports; the one-pass anchor to ccu_first_hit at 1080p;
pre-generated rays; CCU_RENDER_NO_ENTITIES and the flags that do not act; isolation from a render window; the argument and
state checks; renderer.render_features against the C ABI, one and two calls; and a group member's context."""
import ctypes as C
import dataclasses

import numpy as np
import pytest

from chunkyclplugin_b200 import native
from chunkyclplugin_b200 import scenes as S
from chunkyclplugin_b200.javarandom import pass_seeds
from chunkyclplugin_b200.renderer import (CudaPathTracingRenderer, CudaSceneLoader, DefaultRenderManager, RendererInstance, Scene,
                                          upload_scene)
from test_gpu_clouds import cloud_scene
from test_gpu_variants import SEEDS, ctx_no_wide, deep, loader  # noqa: F401

import specular_oracle as SO

BIOME, CLOUDS = native.CCU_RENDER_BIOME_TINT, native.CCU_RENDER_CLOUDS
F = np.float32


def bits(a):
    return np.ascontiguousarray(a, F).view(np.uint32)


def assert_bits(got, want):
    np.testing.assert_array_equal(bits(got), bits(want))


def canonical(a):
    """float32 bits with -0 read as +0: the running mean folds the first pass as (0 * 0 + v) / 1, which maps -0 to +0."""
    return (np.ascontiguousarray(a, F) + F(0)).view(np.uint32)


def features(ctx, p, seeds, flags=0, **params):
    ctx.render_set_params(flags=flags, **params)
    try:
        ctx.render_begin(p.width, p.height)
        return ctx.render_features(np.asarray(seeds, np.int32))
    finally:
        ctx.render_set_params()


# MODE x HAS_BVH x biome x clouds: every instance, on the variant fixture with its biome colours and cloud layer
CASES = [(mode, bvh, biome, clouds) for mode in (0, 1, 2) for bvh in (1, 0) for biome in (0, 1) for clouds in (0, 1)]
_oracle = {}


def oracle_features(bvh, flags, in_deep):
    key = (bvh, flags, in_deep)
    if key not in _oracle:
        p = cloud_scene(0, bool(bvh))
        _oracle[key] = SO.FlagsOracle(deep(p) if in_deep else p, flags).features(SEEDS)
    return _oracle[key]


def test_the_cases_cover_every_instance():
    assert len(set(CASES)) == 24


@pytest.mark.gpu
@pytest.mark.parametrize("case", CASES, ids=lambda c: "mode%d-%s%s%s" % (c[0], "bvh" if c[1] else "nobvh", "-biome" * c[2],
                                                                            "-clouds" * c[3]))
def test_feature_instance(cuda_ctx, ctx_no_wide, loader, monkeypatch, case):  # noqa: F811
    mode, bvh, biome, clouds = case
    flags = (BIOME if biome else 0) | (CLOUDS if clouds else 0)
    p = cloud_scene(0, bool(bvh))
    ctx = cuda_ctx
    if mode == 2:
        p = deep(p)
    if mode == 0:
        monkeypatch.setenv("CCU_NO_WIDE", "1")          # read at commit
        ctx = ctx_no_wide
    loader(ctx, p, (p.name, mode == 0))
    albedo, normal = features(ctx, p, SEEDS, flags)
    assert ctx.last_features() == (mode, bvh, biome, clouds)
    want_a, want_n = oracle_features(bvh, flags, mode == 2)
    assert_bits(albedo, want_a)
    assert_bits(normal, want_n)


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["config1", "entities"])
def test_one_pass_is_the_first_hit_1080p(cuda_ctx, name):
    p = S.terrain_scene(256, 1920, 1080) if name == "config1" else S.entity_scene(256, 1920, 1080)
    upload_scene(cuda_ctx, p)
    cuda_ctx.camera_set(p.projector_type, p.camera)
    cuda_ctx.render_begin(p.width, p.height)
    seed = pass_seeds(1)[0]
    fh = cuda_ctx.first_hit(seed)
    albedo, normal = cuda_ctx.render_features([seed])
    assert cuda_ctx.last_kernel_ms() > 0
    hit = fh["kind"] != 0
    assert hit.mean() > 0.3
    np.testing.assert_array_equal(bits(albedo).reshape(-1, 3)[hit], canonical(fh["color"].reshape(-1, 4)[hit, :3]))
    np.testing.assert_array_equal(bits(normal).reshape(-1, 3)[hit], canonical(fh["normal"].reshape(-1, 3)[hit]))
    assert not normal.reshape(-1, 3)[~hit].any()
    # either output alone is the same buffer
    a_only, none = cuda_ctx.render_features([seed], normal=False)
    assert none is None
    assert_bits(a_only, albedo)
    none, n_only = cuda_ctx.render_features([seed], albedo=False)
    assert none is None
    assert_bits(n_only, normal)
    cuda_ctx.render_end()


@pytest.mark.gpu
def test_pregenerated_rays(cuda_ctx):
    p = S.mixed_test_scene()
    rays = S.pregenerated_rays(p.camera[:15], p.width, p.height, jitter=np.random.default_rng(2))
    upload_scene(cuda_ctx, p)
    cuda_ctx.camera_set(-1, rays)
    seeds = pass_seeds(4)
    albedo, normal = features(cuda_ctx, p, seeds)
    want_a, want_n = SO.FlagsOracle(p, 0).features(seeds, rays=rays)
    assert_bits(albedo, want_a)
    assert_bits(normal, want_n)
    assert not np.array_equal(want_a, SO.FlagsOracle(p, 0).features(seeds)[0])


@pytest.mark.gpu
def test_no_entities_and_the_flags_that_do_not_act(cuda_ctx):
    """CCU_RENDER_NO_ENTITIES gives the features of the scene without BVHs; specular, emitter sampling, fog, no-sun, max_depth and
    emitter_scale change nothing."""
    p = dataclasses.replace(S.entity_scene(128, 160, 90, n_world=96, n_actor=8, subdiv=1), fog=(0.02, 0.5, (0.5, 0.6, 0.7), 0))
    upload_scene(cuda_ctx, p)
    cuda_ctx.camera_set(p.projector_type, p.camera)
    seeds = pass_seeds(3)
    base = features(cuda_ctx, p, seeds)
    assert cuda_ctx.last_features()[1] == 1
    want = SO.FlagsOracle(p, 0).features(seeds)
    assert_bits(base[0], want[0])
    assert_bits(base[1], want[1])
    bare = dataclasses.replace(p, world_bvh=S.EMPTY_BVH.copy(), actor_bvh=S.EMPTY_BVH.copy())
    want_bare = SO.FlagsOracle(bare, 0).features(seeds)
    got = features(cuda_ctx, p, seeds, native.CCU_RENDER_NO_ENTITIES)
    assert cuda_ctx.last_features()[1] == 0
    assert_bits(got[0], want_bare[0])
    assert_bits(got[1], want_bare[1])
    assert not np.array_equal(want_bare[0], want[0])
    ignored = (native.CCU_RENDER_SPECULAR | native.CCU_RENDER_EMITTER_SAMPLING | native.CCU_RENDER_EMITTER_NEAR_FIELD
               | native.CCU_RENDER_EMITTER_MODELS | native.CCU_RENDER_FOG | native.CCU_RENDER_NO_SUN)
    for flags, params in ((native.CCU_RENDER_NO_SUN, {}), (ignored, {}), (0, {"max_depth": 1, "emitter_scale": 2.0})):
        got = features(cuda_ctx, p, seeds, flags, **params)
        assert_bits(got[0], base[0])
        assert_bits(got[1], base[1])


@pytest.mark.gpu
@pytest.mark.parametrize("kernel", [1, 4])
def test_a_feature_call_leaves_the_render_window_alone(cuda_ctx, kernel):
    p = cloud_scene(0)
    upload_scene(cuda_ctx, p)
    cuda_ctx.camera_set(p.projector_type, p.camera)
    seeds = np.asarray(pass_seeds(4), np.int32)
    flags = BIOME | CLOUDS

    def window(with_features):
        cuda_ctx.render_set_params(kernel=kernel, flags=flags)
        try:
            cuda_ctx.render_begin(p.width, p.height)
            cuda_ctx.render_passes(seeds[:2])
            feats = cuda_ctx.render_features(seeds) if with_features else None
            cuda_ctx.render_passes(seeds[2:], block=False)
            img, spp = cuda_ctx.render_read()
            return img, spp, cuda_ctx.last_render_n(9), feats
        finally:
            cuda_ctx.render_set_params()

    img0, spp0, rep0, _ = window(False)
    img1, spp1, rep1, feats = window(True)
    assert spp0 == spp1 == 4
    assert rep0 == rep1
    assert_bits(img1, img0)
    want = SO.FlagsOracle(p, flags).features(seeds)
    assert_bits(feats[0], want[0])
    assert_bits(feats[1], want[1])


@pytest.mark.gpu
def test_argument_and_state_checks(cuda_ctx):
    lib = native.load()
    p = S.mixed_test_scene()
    n = p.width * p.height * 3
    out = np.zeros(n, F)
    seeds = np.asarray(pass_seeds(1025), np.int32)
    vp = lambda a: a.ctypes.data_as(C.c_void_p)      # noqa: E731
    # before ccu_render_begin (a fresh context with a committed scene and a camera)
    fresh = native.Context(0)
    try:
        assert lib.ccu_render_features(fresh._h, vp(seeds), 1, vp(out), None) == native.CCU_ESTATE
        upload_scene(fresh, p)
        fresh.camera_set(p.projector_type, p.camera)
        assert lib.ccu_render_features(fresh._h, vp(seeds), 1, vp(out), None) == native.CCU_ESTATE
        fresh.render_begin(p.width, p.height)
        assert lib.ccu_render_features(fresh._h, vp(seeds), 1, vp(out), None) == native.CCU_OK
        fresh.render_end()
        assert lib.ccu_render_features(fresh._h, vp(seeds), 1, vp(out), None) == native.CCU_ESTATE
        with pytest.raises(native.ChunkyCuError) as e:      # the binding finds no render target and does not call
            fresh.render_features(seeds[:1])
        assert e.value.code == native.CCU_ESTATE
    finally:
        fresh.close()
    upload_scene(cuda_ctx, p)
    cuda_ctx.camera_set(p.projector_type, p.camera)
    cuda_ctx.render_begin(p.width, p.height)
    launches = cuda_ctx.launch_count()
    bad = [(None, vp(seeds), 1, vp(out), vp(out)), (cuda_ctx._h, None, 1, vp(out), vp(out)), (cuda_ctx._h, vp(seeds), 0, vp(out), None),
           (cuda_ctx._h, vp(seeds), -1, vp(out), None), (cuda_ctx._h, vp(seeds), 1025, vp(out), None),
           (cuda_ctx._h, vp(seeds), 1, None, None)]
    for args in bad:
        assert lib.ccu_render_features(*args) == native.CCU_EINVAL
    assert cuda_ctx.launch_count() == launches
    with pytest.raises(native.ChunkyCuError):
        cuda_ctx.render_features([])
    # the largest call: 1024 passes
    a, _ = cuda_ctx.render_features(seeds[:1024], normal=False)
    assert np.isfinite(a).all()
    assert lib.ccu_debug_last_features(None, vp(np.zeros(4, np.int32))) == native.CCU_EINVAL
    cuda_ctx.render_end()


@pytest.mark.gpu
@pytest.mark.parametrize("spp", [5, 1025])
def test_renderer_render_features_matches_the_c_abi(spp):
    """renderer.render_features against direct calls on render()'s seeds; 1025 passes take two calls (1024 + 1) whose means
    the renderer combines in double."""
    p = cloud_scene(0)
    inst = RendererInstance.get(0)
    scene = Scene(p, target_spp=spp)
    renderer = CudaPathTracingRenderer(CudaSceneLoader(inst))
    albedo, normal = renderer.render_features(DefaultRenderManager(scene), spp)
    assert albedo.dtype == np.float64 and albedo.shape == (p.width * p.height * 3,)
    ctx = inst.context
    ctx.camera_set(p.projector_type, p.camera)
    ctx.render_begin(p.width, p.height)
    seeds = np.asarray(pass_seeds(spp), np.int32)
    parts = [seeds[i:i + native.CCU_FEATURES_MAX_PASSES] for i in range(0, spp, native.CCU_FEATURES_MAX_PASSES)]
    outs = [ctx.render_features(part) for part in parts]
    ctx.render_end()
    want_a, want_n = outs[0][0].astype(np.float64), outs[0][1].astype(np.float64)
    done = parts[0].size
    for part, (a, n) in zip(parts[1:], outs[1:]):
        want_a = (want_a * done + a.astype(np.float64) * part.size) / (done + part.size)
        want_n = (want_n * done + n.astype(np.float64) * part.size) / (done + part.size)
        done += part.size
    np.testing.assert_array_equal(albedo, want_a)
    np.testing.assert_array_equal(normal, want_n)
    if spp == 5:
        # the flags default to off: the restatement without biome colours or clouds
        want = SO.FlagsOracle(p, 0).features(seeds)
        assert_bits(outs[0][0], want[0])
        assert_bits(outs[0][1], want[1])


@pytest.mark.gpu
def test_group_member_renders_features():
    """A group member's context gets its canvas from ccu_group_render_begin: render_features on it returns full buffers, the
    restatement's bits."""
    p = cloud_scene(0)
    flags = BIOME | CLOUDS
    want = SO.FlagsOracle(p, flags).features(SEEDS)
    group = native.Group(devices=[0])
    try:
        upload_scene(group.member(0), p)
        group.replicate_scene()
        group.camera_set(p.projector_type, p.camera)
        group.render_set_params(flags=flags)
        group.render_begin(p.width, p.height)
        albedo, normal = group.member(0).render_features(SEEDS)
        assert albedo.shape == normal.shape == (p.width * p.height * 3,)
        assert_bits(albedo, want[0])
        assert_bits(normal, want[1])
        group.render_end()
    finally:
        group.close()
