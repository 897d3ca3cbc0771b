"""CCU_RENDER_CLOUDS on the GPU (DESIGN.md §15): the 360 cloud instances of both render kernels against the CPU restatement
(FlagsOracle) bit for bit, with the instance each launch reports, the selection rule for flag and scene, the setter's checks and
the scene lifecycle (ccu_scene_begin, device bytes, group replication), and the flag-off identities at 1080p on both kernels."""
import dataclasses
import functools

import numpy as np
import pytest

from chunkyclplugin_b200 import native
from chunkyclplugin_b200 import scenes as S
from chunkyclplugin_b200.javarandom import pass_seeds
from chunkyclplugin_b200.renderer import upload_scene
from test_clouds import fixture_clouds
from test_gpu_fog import FOG_FAST, FOG_SLOW, fog_lay, fog_staged
from test_gpu_specular import assert_bits
from test_gpu_variants import (SEEDS, SHADES, _render, ctx_no_wide, deep, loader, shade_flags, shade_id,  # noqa: F401
                               staged_texels, variant_scene)

import specular_oracle as SO

CLOUDS = native.CCU_RENDER_CLOUDS
FOG = native.CCU_RENDER_FOG
MASK_BYTES = 256 * 256 // 8     # the bit-packed mask the committed scene holds


@functools.lru_cache(maxsize=None)
def cloud_scene(fog: int, bvh: bool = True) -> S.PackedScene:
    """The variant fixture (every Shade switch acts on it, the sun is on) with the cloud layer of test_clouds.fixture_clouds;
    fog: 0 none, 1 slow fog, 2 fast fog."""
    p = fixture_clouds(variant_scene(bvh))
    if fog:
        p = dataclasses.replace(p, fog=FOG_FAST if fog == 2 else FOG_SLOW, name=p.name + ("_fogfast" if fog == 2 else "_fog"))
    return p


_images = {}


def cloud_image(fog: int, flags: int, bvh: bool = True, in_deep: bool = False) -> np.ndarray:
    """FlagsOracle's image of cloud_scene, or of its copy embedded in a depth-13 world.  Unlike the fixture without clouds the
    two differ: a bounce off a cloud beyond the 64^3 world starts outside the shallow octree (which it enters through its
    bounding box) but inside the deep one (which it marches through from its origin), so its hit distances round differently."""
    key = (fog, flags, bool(bvh), in_deep)
    if key not in _images:
        p = cloud_scene(fog, bvh)
        _images[key] = SO.FlagsOracle(deep(p) if in_deep else p, flags).render(SEEDS)
    return _images[key]


# kernel 4 x HAS_BVH x LAY x 20 Shades x fog and kernel 1 x MODE x 20 x fog, all with clouds; the fog instances take fast fog on
# LAY / MODE 1 and slow fog on 0 and 2, as in test_gpu_fog
CASES = ([(4, bvh, lay, i, fog) for bvh in (1, 0) for lay in (0, 1, 2) for i in range(20) for fog in (0, 1)]
         + [(1, 1, mode, i, fog) for mode in (0, 1, 2) for i in range(20) for fog in (0, 1)])


def _case_id(c):
    kernel, bvh, lay, i, fog = c
    return ((f"k4-{'bvh' if bvh else 'nobvh'}-lay{lay}" if kernel == 4 else f"k1-mode{lay}") + "-" + shade_id(i)
            + ("-fog" if fog else ""))


def test_the_cases_cover_every_cloud_instance():
    assert len(CASES) == 360 and len(set(CASES)) == 360


@pytest.mark.gpu
@pytest.mark.parametrize("case", CASES, ids=_case_id)
def test_cloud_instance(cuda_ctx, ctx_no_wide, loader, monkeypatch, case):  # noqa: F811
    kernel, bvh, lay, i, fog = case
    spec, nee, biome = SHADES[i]
    flags = shade_flags(spec, nee, biome) | CLOUDS | (FOG if fog else 0)
    fog_kind = (2 if lay == 1 else 1) if fog else 0
    p = cloud_scene(fog_kind, bvh)
    ctx = cuda_ctx
    if lay == 2:
        p = deep(p)
    if kernel == 4 and lay == 1:
        monkeypatch.setenv("CCU_NO_TOPS", "1")          # read at every launch
    if kernel == 1 and lay == 0:
        monkeypatch.setenv("CCU_NO_WIDE", "1")          # read at commit
        ctx = ctx_no_wide
    loader(ctx, p, (p.name, lay == 0 and kernel == 1))
    got = _render(ctx, p, SEEDS, kernel, flags)
    if kernel == 4:
        # the clouds add no slot field: the LAY rule and the sky staging are those of the same launch without clouds
        ran = fog_lay(bvh, lay, spec, nee != 0) if fog else lay
        sky = (fog_staged(bvh, ran, spec, nee != 0, p.sky.shape[0]) if fog
               else staged_texels(bvh, ran == 0, spec, nee != 0, p.sky.shape[0]))
    else:
        ran, sky = lay, 0
    assert ctx.last_render_n(9) == (kernel, bvh, ran, spec, nee, biome, sky, fog, 1)
    assert ctx.last_render_n(8) == (kernel, bvh, ran, spec, nee, biome, sky, fog)
    assert ctx.last_render() == (kernel, bvh, ran, spec, nee, biome, sky)
    assert_bits(got, cloud_image(fog_kind, flags, bvh, lay == 2))


@pytest.mark.gpu
@pytest.mark.parametrize("kernel", [0, 1, 4])
def test_selection(cuda_ctx, kernel):
    """The clouds switch is on exactly when the flag is set and the scene has a mask with a set cell; otherwise the launch runs
    the kernel and bits it runs without the flag."""
    base = cloud_scene(0)
    empty = (np.zeros((256, 256), np.uint8),) + base.clouds[1:]
    for clouds in (None, empty, base.clouds):
        p = dataclasses.replace(base, clouds=clouds)
        upload_scene(cuda_ctx, p)
        cuda_ctx.camera_set(p.projector_type, p.camera)
        off = _render(cuda_ctx, p, SEEDS, kernel, 0)
        rep_off = cuda_ctx.last_render_n(9)
        assert rep_off[8] == 0
        on = _render(cuda_ctx, p, SEEDS, kernel, CLOUDS)
        if clouds is base.clouds:
            assert cuda_ctx.last_render_n(9) == rep_off[:8] + (1,)
            assert_bits(on, cloud_image(0, CLOUDS))
        else:
            assert cuda_ctx.last_render_n(9) == rep_off
            assert_bits(on, off)


@pytest.mark.gpu
def test_setter_checks_and_scene_lifecycle(cuda_ctx):
    p = cloud_scene(0)
    upload_scene(cuda_ctx, dataclasses.replace(p, clouds=None))
    without = cuda_ctx.scene_device_bytes()
    mask = p.clouds[0]
    nan, inf = float("nan"), float("inf")
    bad = [(0.0, 1, 2, 0, 0), (-1.0, 1, 2, 0, 0), (nan, 1, 2, 0, 0), (inf, 1, 2, 0, 0), (4.0, nan, 2, 0, 0), (4.0, 1, inf, 0, 0),
           (4.0, -inf, 2, 0, 0), (4.0, 1, 2, nan, 0), (4.0, 1, 2, 0, inf), (4.0, 2, 2, 0, 0), (4.0, 3, 2, 0, 0)]
    for args in bad:
        with pytest.raises(native.ChunkyCuError) as e:
            cuda_ctx.set_clouds(mask, *args)
        assert e.value.code == native.CCU_EINVAL, args
    cuda_ctx.set_clouds(None, nan, nan, nan, nan, nan)       # removal ignores the other arguments
    # the clouds take effect at commit and the committed scene holds the bit-packed mask
    upload_scene(cuda_ctx, p)
    assert cuda_ctx.scene_device_bytes() == without + MASK_BYTES
    cuda_ctx.camera_set(p.projector_type, p.camera)
    assert_bits(_render(cuda_ctx, p, SEEDS, 1, CLOUDS), cloud_image(0, CLOUDS))
    # ccu_scene_begin removes them: the same scene uploaded without clouds renders flag-on as flag-off
    q = dataclasses.replace(p, clouds=None)
    upload_scene(cuda_ctx, q)
    assert cuda_ctx.scene_device_bytes() == without
    cuda_ctx.camera_set(q.projector_type, q.camera)
    on = _render(cuda_ctx, q, SEEDS, 1, CLOUDS)
    assert cuda_ctx.last_render_n(9)[8] == 0
    assert_bits(on, _render(cuda_ctx, q, SEEDS, 1, 0))


@pytest.mark.gpu
def test_group_replicates_clouds():
    """Every member of a group of one (and of two where there are two GPUs) renders the cloud image after replicate_scene."""
    p = cloud_scene(0)
    want = cloud_image(0, CLOUDS)
    n = min(native.device_count(), 2)
    for k in sorted({1, n}):
        group = native.Group(devices=list(range(k)))
        try:
            upload_scene(group.member(0), p)
            group.replicate_scene()
            for i in range(k):
                m = group.member(i)
                m.camera_set(p.projector_type, p.camera)
                assert_bits(_render(m, p, SEEDS, 4, CLOUDS), want)
                assert m.last_render_n(9)[8] == 1
                assert m.scene_device_bytes() == group.member(0).scene_device_bytes()
        finally:
            group.close()


SEEDS2 = pass_seeds(2)


@pytest.mark.gpu
@pytest.mark.parametrize("kernel", [0, 1])
def test_flag_off_identities_1080p(cuda_ctx, kernel):
    """DESIGN §15.5 at 1080p: the flag on a scene without clouds, and clouds without the flag, render the flag-off bits."""
    base = S.mixed_test_scene(64, 1920, 1080)
    clouded = S.with_clouds(base, S.cloud_mask(seed=4), size=3.0, y0=40.0, y1=44.0)

    def render(p, flags):
        upload_scene(cuda_ctx, p)
        cuda_ctx.camera_set(p.projector_type, p.camera)
        return _render(cuda_ctx, p, SEEDS2, kernel, flags)

    ref = render(base, 0)
    assert_bits(render(base, CLOUDS), ref)
    assert cuda_ctx.last_render_n(9)[8] == 0 and cuda_ctx.last_render_n(9)[0] == (4 if kernel == 0 else 1)
    assert_bits(render(clouded, 0), ref)
    assert cuda_ctx.last_render_n(9)[8] == 0
