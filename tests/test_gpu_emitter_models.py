"""CCU_RENDER_EMITTER_MODELS on the device: both render kernels (wavefront and thread-per-pixel) with flags 8 | 256 and
8 | 256 | 128 against the CPU restatement (FlagsOracle) bit for bit, on the case matrix of the CCU_RENDER_EMITTER_SAMPLING
tests with model emitters (quad and AABB models made emissive), on the torch contact scene, the edge-ray catalogue and config
3 lit by models at 1920 x 1080.  Kernel selection: without a model emitter 256 changes nothing.  One group-API case."""
import dataclasses

import numpy as np
import pytest

from chunkyclplugin_b200 import native
from chunkyclplugin_b200 import scenes as S
from chunkyclplugin_b200.javarandom import pass_seeds
from conftest import load_scene
from oracle import edge_rays as E
from test_emitter_models import analytic_quad_scene, contact_scene, deep_models, lantern_scene
from test_emitter_sampling import SCALE
from test_gpu_emitter_sampling import CASES, _render
from test_gpu_specular import _case, assert_bits
from test_oracle_edge_rays import E_PASSES, EDGE

import specular_oracle as SO

pytestmark = pytest.mark.gpu
NEE, NEAR, MODELS, SPEC, NO_ENTITIES = 8, 128, 256, 4, 1


def lit_models(p):
    """p with its quad and AABB model materials made emissive when it has models; otherwise p with its sand, grass, dirt or
    stone (the first that gives a model table) turned into torches and lanterns appended to its palettes."""
    q = S.emissive_models(p)
    if SO.emitter_grid(q, models=True)["has_emitters"]:
        return q
    bp, mp = list(p.block_palette), list(p.mat_palette)
    quads, aabbs = list(p.quad_models), list(p.aabb_models)
    mat0 = len(mp)
    # flat-coloured materials (the scene's atlas is left as it is): an emitting one, and the lantern's cap
    mp += S.pack_material(0, 0, textured=False, argb=S._s32(0xFFFFD070), emittance=1.0)
    mp += S.pack_material(0, 0, textured=False, argb=S._s32(0xFF404048))
    tq, ta = len(quads), len(aabbs)
    quads += S._torch_quads(mat0)
    aabbs += S._lantern_boxes(mat0, mat0 + 6)
    pos_t, pos_l = len(bp), len(bp) + 2
    bp += [3, tq, 2, ta]
    for block, new in ((8, pos_t), (6, pos_l), (4, pos_t), (2, pos_l)):
        tree = np.where(p.octree == -block, -new, p.octree).astype(np.int32)
        r = dataclasses.replace(p, octree=tree, block_palette=S._i32(bp), mat_palette=S._i32(mp), quad_models=S._i32(quads),
                                aabb_models=S._i32(aabbs), name=p.name + "_torches")
        if SO.emitter_grid(r, models=True)["has_emitters"]:
            return r
    raise AssertionError(f"{p.name}: no model table")


def _oracle(p, flags, max_depth=5, **kw):
    if flags & NO_ENTITIES:
        p = dataclasses.replace(p, world_bvh=S.EMPTY_BVH.copy(), actor_bvh=S.EMPTY_BVH.copy())
    return SO.FlagsOracle(p, flags=flags & (NEE | NEAR | MODELS | SPEC), max_depth=max_depth, **kw)


EXTRA = {"deep13": deep_models, "lanterns": lantern_scene, "indoor_models": lambda: S.indoor_models_scene(64, 48, 27)}


@pytest.mark.parametrize("near", [0, NEAR], ids=["area", "near"])
@pytest.mark.parametrize("max_depth", [2, 5])
@pytest.mark.parametrize("spec", [0, SPEC], ids=["diffuse", "specular"])
@pytest.mark.parametrize("sun", ["sun", "nosun"])
@pytest.mark.parametrize("name", list(CASES) + list(EXTRA))
def test_kernel_matches_the_oracle(scenes, cuda_ctx, name, sun, spec, max_depth, near):
    p = EXTRA[name]() if name in EXTRA else lit_models(_case(scenes, name))
    if sun == "nosun":
        p = E.without_sun(p)
    assert SO.emitter_grid(p, models=True)["has_emitters"]
    seeds = pass_seeds(3)
    flags = NEE | MODELS | near | spec
    want = _oracle(p, flags, max_depth).render(seeds)
    load_scene(cuda_ctx, p)
    for kernel in (4, 1):
        assert_bits(_render(cuda_ctx, p, seeds, kernel, flags, max_depth), want)


@pytest.mark.parametrize("near", [0, NEAR], ids=["area", "near"])
@pytest.mark.parametrize("name", ["mixed", "entities"])
def test_no_entities(scenes, cuda_ctx, name, near):
    p = lit_models(_case(scenes, name))
    seeds = pass_seeds(3)
    flags = NEE | MODELS | near | NO_ENTITIES
    want = _oracle(p, flags).render(seeds)
    load_scene(cuda_ctx, p)
    for kernel in (4, 1):
        assert_bits(_render(cuda_ctx, p, seeds, kernel, flags), want)


@pytest.mark.parametrize("near", [0, NEAR], ids=["area", "near"])
@pytest.mark.parametrize("name", EDGE)
def test_edge_rays(cuda_ctx, name, near):
    p = lit_models(E.scenes()[name])
    seeds = pass_seeds(E_PASSES)
    want = _oracle(p, NEE | MODELS | near).render(seeds)
    load_scene(cuda_ctx, p)
    for kernel in (4, 1):
        assert_bits(_render(cuda_ctx, p, seeds, kernel, NEE | MODELS | near), want)


@pytest.mark.parametrize("near", [0, NEAR], ids=["area", "near"])
@pytest.mark.parametrize("name", ["contact", "analytic"])
@pytest.mark.parametrize("max_depth", [2, 5])
def test_contact_and_analytic_scenes(cuda_ctx, name, max_depth, near):
    """The torch contact scene (floor points down to 1e-3 from the stick) and the quad over the analytic floor."""
    p = contact_scene() if name == "contact" else analytic_quad_scene(1024)
    seeds = pass_seeds(4)
    flags = NEE | MODELS | near
    want = _oracle(p, flags, max_depth, emitter_scale=SCALE).render(seeds)
    load_scene(cuda_ctx, p)
    try:
        for kernel in (4, 1):
            cuda_ctx.render_set_params(kernel=kernel, flags=flags, max_depth=max_depth, emitter_scale=SCALE)
            cuda_ctx.render_begin(p.width, p.height)
            cuda_ctx.render_passes(np.asarray(seeds, np.int32))
            assert_bits(cuda_ctx.render_read()[0], want)
    finally:
        cuda_ctx.render_set_params()


@pytest.mark.parametrize("near", [0, NEAR], ids=["area", "near"])
def test_baseline_canvas_config3_models(cuda_ctx, near):
    """Config 3 lit by model blocks (indoor_models_scene(256)) at 1920 x 1080, every 64th pixel."""
    p = S.indoor_models_scene(256, 1920, 1080)
    seeds = pass_seeds(2)
    gids = np.arange(0, p.width * p.height, 64, dtype=np.int32)
    flags = NEE | MODELS | near
    want = _oracle(p, flags).render(seeds, gids=gids).reshape(-1, 3)[gids]
    load_scene(cuda_ctx, p)
    for kernel in (4, 1):
        assert_bits(_render(cuda_ctx, p, seeds, kernel, flags).reshape(-1, 3)[gids], want)


def test_cube_only_scene_renders_as_bit_8(scenes, cuda_ctx):
    """Without a model emitter, 256 selects the kernels of bit 8 alone: the same bits."""
    p = scenes("indoor")
    assert not SO.emitter_grid(p, models=True)["has_emitters"]
    seeds = pass_seeds(3)
    load_scene(cuda_ctx, p)
    for kernel in (4, 1, 0):
        for near in (0, NEAR):
            assert_bits(_render(cuda_ctx, p, seeds, kernel, NEE | MODELS | near), _render(cuda_ctx, p, seeds, kernel, NEE | near))


@pytest.mark.parametrize("name", ["terrain64", "entities"])
def test_no_emitters_renders_as_flag_off(scenes, cuda_ctx, name):
    p = scenes(name)
    assert not SO.emitter_grid(p)["has_emitters"] and not SO.emitter_grid(p, models=True)["has_emitters"]
    seeds = pass_seeds(3)
    load_scene(cuda_ctx, p)
    for kernel in (4, 1, 0):
        assert_bits(_render(cuda_ctx, p, seeds, kernel, NEE | MODELS | NEAR), _render(cuda_ctx, p, seeds, kernel, 0))


def test_models_only_scene_runs_the_nee_kernels(cuda_ctx):
    """A scene lit by model blocks only: with 256 the NEE kernels run and render differently from flags 0 and from bit 8 alone
    (which has no table there)."""
    p = S.indoor_models_scene(64, 48, 27)
    assert not SO.emitter_grid(p)["has_emitters"]
    seeds = pass_seeds(2)
    load_scene(cuda_ctx, p)
    off = _render(cuda_ctx, p, seeds, 4, 0)
    assert_bits(_render(cuda_ctx, p, seeds, 4, NEE), off)
    for kernel in (4, 1, 0):
        assert not np.array_equal(_render(cuda_ctx, p, seeds, kernel, NEE | MODELS), off)


def _group_render(group, p, seeds, flags):
    m0 = group.member(0)
    load_scene(m0, p)
    m0.render_end()
    group.replicate_scene()
    group.camera_set(p.projector_type, p.camera)
    group.render_set_params(flags=flags)
    group.render_begin(p.width, p.height)
    sb = np.zeros(p.width * p.height * 3, dtype=np.float64)
    group.render_passes(seeds)
    assert group.render_merge(sb, 0) == len(seeds)
    group.render_end()
    return sb


def test_group_of_one_matches_a_context(cuda_ctx):
    p = S.indoor_models_scene(64, 48, 27)
    seeds = pass_seeds(4)
    flags = NEE | MODELS | NEAR
    load_scene(cuda_ctx, p)
    want = _render(cuda_ctx, p, seeds, 0, flags).astype(np.float64)
    group = native.Group(devices=[0])
    try:
        assert np.array_equal(_group_render(group, p, seeds, flags), want)
    finally:
        group.close()
