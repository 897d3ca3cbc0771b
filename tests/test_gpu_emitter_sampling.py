"""CCU_RENDER_EMITTER_SAMPLING on the device: both render kernels (wavefront and thread-per-pixel) against the CPU
restatement (FlagsOracle) bit for bit on scenes with full-cube emitters (every octree layout including the deep-world one,
entity BVHs, sun on and off, the specular flag on and off, ray depths 2 and 5, CCU_RENDER_NO_ENTITIES, pre-generated rays),
on the edge-ray catalogue, at config 3's BASELINE canvas, and through the group API.  Kernel selection: the flag picks the
NEE kernels only on a scene with emitters."""
import dataclasses

import numpy as np
import pytest

from chunkyclplugin_b200 import native
from chunkyclplugin_b200 import scenes as S
from chunkyclplugin_b200.javarandom import pass_seeds
from conftest import load_scene
from oracle import edge_rays as E
from test_emitter_sampling import cluster_scene, deep_indoor
from test_gpu_specular import CASES, _case, assert_bits
from test_oracle_edge_rays import E_PASSES, EDGE

import specular_oracle as SO

pytestmark = pytest.mark.gpu
NEE, SPEC, NO_ENTITIES = 8, 4, 1


def _render(ctx, p, seeds, kernel, flags, max_depth=5):
    ctx.render_set_params(kernel=kernel, flags=flags, max_depth=max_depth)
    try:
        ctx.render_begin(p.width, p.height)
        ctx.render_passes(np.asarray(seeds, np.int32))
        return ctx.render_read()[0]
    finally:
        ctx.render_set_params()


def _oracle(p, flags, max_depth=5):
    if flags & NO_ENTITIES:
        p = dataclasses.replace(p, world_bvh=S.EMPTY_BVH.copy(), actor_bvh=S.EMPTY_BVH.copy())
    return SO.FlagsOracle(p, flags=flags & (NEE | SPEC), max_depth=max_depth)


def lit(p):
    """p itself when it has full-cube emitters, else p with its sand, grass, dirt or stone (the first that gives a table)
    turned into glowstone"""
    for block in (0, 8, 6, 4, 2):
        q = dataclasses.replace(p, octree=np.where(p.octree == -block, -10, p.octree).astype(np.int32)) if block else p
        if SO.emitter_grid(q)["has_emitters"]:
            return q
    raise AssertionError(f"{p.name}: no emitter table")


def _with_emitters(scenes, name):
    return lit(_case(scenes, name))


EXTRA = {"deep13": deep_indoor, "cluster": cluster_scene}


@pytest.mark.parametrize("max_depth", [2, 5])
@pytest.mark.parametrize("spec", [0, SPEC], ids=["diffuse", "specular"])
@pytest.mark.parametrize("sun", ["sun", "nosun"])
@pytest.mark.parametrize("name", list(CASES) + list(EXTRA))
def test_kernel_matches_the_oracle(scenes, cuda_ctx, name, sun, spec, max_depth):
    p = EXTRA[name]() if name in EXTRA else _with_emitters(scenes, name)
    if sun == "nosun":
        p = E.without_sun(p)
    assert SO.emitter_grid(p)["has_emitters"]
    seeds = pass_seeds(3)
    flags = NEE | spec
    want = _oracle(p, flags, max_depth).render(seeds)
    load_scene(cuda_ctx, p)
    for kernel in (4, 1):
        assert_bits(_render(cuda_ctx, p, seeds, kernel, flags, max_depth), want)


@pytest.mark.parametrize("name", ["mixed", "entities"])
def test_no_entities(scenes, cuda_ctx, name):
    p = _with_emitters(scenes, name)
    seeds = pass_seeds(3)
    want = _oracle(p, NEE | NO_ENTITIES).render(seeds)
    load_scene(cuda_ctx, p)
    for kernel in (4, 1):
        assert_bits(_render(cuda_ctx, p, seeds, kernel, NEE | NO_ENTITIES), want)


@pytest.mark.parametrize("name", EDGE)
def test_edge_rays(cuda_ctx, name):
    p = lit(E.scenes()[name])
    seeds = pass_seeds(E_PASSES)
    want = _oracle(p, NEE).render(seeds)
    load_scene(cuda_ctx, p)
    for kernel in (4, 1):
        assert_bits(_render(cuda_ctx, p, seeds, kernel, NEE), want)


def test_baseline_canvas_config3(cuda_ctx):
    """BASELINE config 3 (indoor256, sun off) at 1920 x 1080, every 64th pixel."""
    p = S.indoor_scene(256, 1920, 1080)
    seeds = pass_seeds(2)
    gids = np.arange(0, p.width * p.height, 64, dtype=np.int32)
    want = _oracle(p, NEE).render(seeds, gids=gids).reshape(-1, 3)[gids]
    load_scene(cuda_ctx, p)
    for kernel in (4, 1):
        assert_bits(_render(cuda_ctx, p, seeds, kernel, NEE).reshape(-1, 3)[gids], want)


@pytest.mark.parametrize("name", ["terrain64", "entities"])
def test_no_emitters_changes_nothing(scenes, cuda_ctx, name):
    """Without full-cube emitters the flag selects the old kernels and renders the same bits."""
    p = scenes(name)
    assert not SO.emitter_grid(p)["has_emitters"]
    seeds = pass_seeds(3)
    load_scene(cuda_ctx, p)
    for kernel in (4, 1, 0):
        assert_bits(_render(cuda_ctx, p, seeds, kernel, NEE), _render(cuda_ctx, p, seeds, kernel, 0))


def test_kernel_selection(scenes, cuda_ctx):
    p = scenes("indoor")
    seeds = pass_seeds(2)
    load_scene(cuda_ctx, p)
    on4 = _render(cuda_ctx, p, seeds, 4, NEE)
    assert_bits(_render(cuda_ctx, p, seeds, 0, NEE), on4)
    assert_bits(_render(cuda_ctx, p, seeds, 1, NEE), on4)
    assert not np.array_equal(on4, _render(cuda_ctx, p, seeds, 4, 0))


def _group_render(group, p, seeds):
    m0 = group.member(0)
    load_scene(m0, p)
    m0.render_end()
    group.replicate_scene()
    group.camera_set(p.projector_type, p.camera)
    group.render_set_params(flags=NEE)
    group.render_begin(p.width, p.height)
    sb = np.zeros(p.width * p.height * 3, dtype=np.float64)
    group.render_passes(seeds)
    assert group.render_merge(sb, 0) == len(seeds)
    group.render_end()
    return sb


def test_group_of_one_matches_a_context(scenes, cuda_ctx):
    p = scenes("indoor")
    seeds = pass_seeds(4)
    load_scene(cuda_ctx, p)
    want = _render(cuda_ctx, p, seeds, 0, NEE).astype(np.float64)
    group = native.Group(devices=[0])
    try:
        assert np.array_equal(_group_render(group, p, seeds), want)
    finally:
        group.close()


def test_two_gpu_group_matches_one_gpu(scenes, cuda_ctx):
    if native.device_count() < 2:
        pytest.skip("NEEDS 2 GPUs - the 2-GPU group path is not exercised on this box")
    p = scenes("indoor")
    seeds = pass_seeds(6)
    load_scene(cuda_ctx, p)
    want = _render(cuda_ctx, p, seeds, 0, NEE).astype(np.float64)
    group = native.Group(devices=[0, 1])
    try:
        assert np.allclose(_group_render(group, p, seeds), want, rtol=2e-6, atol=1e-7)
    finally:
        group.close()
