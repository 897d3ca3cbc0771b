"""CCU_RENDER_EMITTER_NEAR_FIELD on the device: both render kernels (wavefront and thread-per-pixel) with flags 8 | 128 against
the CPU restatement (FlagsOracle) bit for bit, on the case matrix of the CCU_RENDER_EMITTER_SAMPLING tests, on the contact
scene where every sample is near, and on the edge-ray catalogue.  Kernel selection: without an emitter table the flags pick
the plain kernels.  One group-API case."""
import dataclasses

import numpy as np
import pytest

from chunkyclplugin_b200 import native
from chunkyclplugin_b200 import scenes as S
from chunkyclplugin_b200.javarandom import pass_seeds
from conftest import load_scene
from oracle import edge_rays as E
from test_emitter_near_field import contact_scene
from test_emitter_sampling import SCALE
from test_gpu_emitter_sampling import CASES, EXTRA, _render, _with_emitters, lit
from test_gpu_specular import assert_bits
from test_oracle_edge_rays import E_PASSES, EDGE

import specular_oracle as SO

pytestmark = pytest.mark.gpu
NEE, NEAR, SPEC, NO_ENTITIES = 8, 128, 4, 1


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
    flags = NEE | NEAR | spec
    want = SO.FlagsOracle(p, flags=flags, max_depth=max_depth).render(seeds)
    load_scene(cuda_ctx, p)
    for kernel in (4, 1):
        assert_bits(_render(cuda_ctx, p, seeds, kernel, flags, max_depth), want)


def _oracle(p, flags, max_depth=5):
    if flags & NO_ENTITIES:
        p = dataclasses.replace(p, world_bvh=S.EMPTY_BVH.copy(), actor_bvh=S.EMPTY_BVH.copy())
    return SO.FlagsOracle(p, flags=flags & (NEE | NEAR | SPEC), max_depth=max_depth)


@pytest.mark.parametrize("name", ["mixed", "entities"])
def test_no_entities(scenes, cuda_ctx, name):
    p = _with_emitters(scenes, name)
    seeds = pass_seeds(3)
    want = _oracle(p, NEE | NEAR | NO_ENTITIES).render(seeds)
    load_scene(cuda_ctx, p)
    for kernel in (4, 1):
        assert_bits(_render(cuda_ctx, p, seeds, kernel, NEE | NEAR | NO_ENTITIES), want)


@pytest.mark.parametrize("name", EDGE)
def test_edge_rays(cuda_ctx, name):
    p = lit(E.scenes()[name])
    seeds = pass_seeds(E_PASSES)
    want = SO.FlagsOracle(p, flags=NEE | NEAR).render(seeds)
    load_scene(cuda_ctx, p)
    for kernel in (4, 1):
        assert_bits(_render(cuda_ctx, p, seeds, kernel, NEE | NEAR), want)


@pytest.mark.parametrize("max_depth", [2, 5])
def test_contact_scene(cuda_ctx, max_depth):
    """Floor points down to 1e-3 from the emitter's side faces: nearly every sample takes the near branch."""
    p = contact_scene()
    seeds = pass_seeds(4)
    want = SO.FlagsOracle(p, flags=NEE | NEAR, max_depth=max_depth, emitter_scale=SCALE).render(seeds)
    load_scene(cuda_ctx, p)
    try:
        for kernel in (4, 1):
            cuda_ctx.render_set_params(kernel=kernel, flags=NEE | NEAR, max_depth=max_depth, emitter_scale=SCALE)
            cuda_ctx.render_begin(p.width, p.height)
            cuda_ctx.render_passes(np.asarray(seeds, np.int32))
            assert_bits(cuda_ctx.render_read()[0], want)
    finally:
        cuda_ctx.render_set_params()


@pytest.mark.parametrize("name", ["terrain64", "entities"])
def test_no_emitters_runs_the_plain_kernels(scenes, cuda_ctx, name):
    """Without full-cube emitters the flags select the kernels without a sampler and render the same bits as flags off."""
    p = scenes(name)
    assert not SO.emitter_grid(p)["has_emitters"]
    seeds = pass_seeds(3)
    load_scene(cuda_ctx, p)
    for kernel in (4, 1, 0):
        assert_bits(_render(cuda_ctx, p, seeds, kernel, NEE | NEAR), _render(cuda_ctx, p, seeds, kernel, 0))


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
    """On the contact scene, where the near branch decides most samples."""
    p = contact_scene()
    seeds = pass_seeds(4)
    load_scene(cuda_ctx, p)
    want = _render(cuda_ctx, p, seeds, 0, NEE | NEAR).astype(np.float64)
    assert not np.array_equal(want, _render(cuda_ctx, p, seeds, 0, NEE).astype(np.float64))
    group = native.Group(devices=[0])
    try:
        assert np.array_equal(_group_render(group, p, seeds, NEE | NEAR), want)
    finally:
        group.close()
