"""CCU_RENDER_FOG on the GPU (DESIGN.md §14): the 180 fog instances of both render kernels against the CPU restatement
(FlagsOracle) bit for bit, the instance each launch reports (with the LAY rule of DESIGN §5), the selection rule for flag and
scene, the sky-staging boundary of every fog footprint, the setter's checks, replication to a group, and the bit-identities
of §14.5 at 1080p on both kernels."""
import dataclasses
import functools
import math

import numpy as np
import pytest

from chunkyclplugin_b200 import native
from chunkyclplugin_b200 import scenes as S
from chunkyclplugin_b200.javarandom import pass_seeds
from chunkyclplugin_b200.renderer import upload_scene
from oracle import edge_rays as E
from test_gpu_specular import assert_bits
from test_gpu_input_edges import noise_sky
from test_gpu_variants import (BIOME, NEE, Q_SMEM_LIMIT, SEEDS, SHADES, SKY_SMEM_DEFAULT, SPEC, FOOTPRINTS, _render,  # noqa: F401
                               ctx_no_wide, loader, q_smem_bytes, shade_flags, shade_id, variant_scene)

import specular_oracle as SO

FOG = native.CCU_RENDER_FOG
FOG_SLOW = (0.03, 0.6, (0.55, 0.65, 0.9), False)
FOG_FAST = (0.03, 0.6, (0.55, 0.65, 0.9), True)


FOG_FIELDS = 8          # slot fields the fog adds to k_render_queue (ccu_queue.cuh, q_fields)


def q_smem_fog(bvh, tops, spec, nee):
    return q_smem_bytes(bvh, tops, spec, nee) + FOG_FIELDS * 1024 * 4


def fog_lay(bvh, lay, spec, nee):
    """DESIGN §5: a fog launch whose footprint does not fit beside the staged top table runs on LAY 1."""
    return 1 if lay == 0 and q_smem_fog(bvh, 1, spec, nee) > Q_SMEM_LIMIT else lay


def fog_staged(bvh, lay, spec, nee, sky_res, sky_max=SKY_SMEM_DEFAULT):
    n = sky_res * sky_res
    return n if n * 4 <= sky_max and q_smem_fog(bvh, lay == 0, spec, nee) + n * 4 <= Q_SMEM_LIMIT else 0


@functools.lru_cache(maxsize=None)
def fog_scene(fast: bool, bvh: bool = True) -> S.PackedScene:
    """The variant fixture (every Shade switch acts on it, the sun is on) with fog."""
    p = variant_scene(bvh)
    return dataclasses.replace(p, fog=FOG_FAST if fast else FOG_SLOW, name=p.name + ("_fogfast" if fast else "_fog"))


def deep(p):
    return dataclasses.replace(p, octree=E.embed_octree(p.octree, 13 - p.octree_depth), octree_depth=13, name=p.name + "_deep13")


_images = {}


def fog_image(fast: bool, flags: int, bvh: bool = True) -> np.ndarray:
    key = (fast, flags, bool(bvh))
    if key not in _images:
        _images[key] = SO.FlagsOracle(fog_scene(fast, bvh), flags).render(SEEDS)
    return _images[key]


def test_fog_changes_the_fixture():
    """CPU: fog changes most pixels of the fixture, and the two fog kinds differ."""
    off = SO.FlagsOracle(fog_scene(False), 0).render(SEEDS)
    for fast in (False, True):
        on = fog_image(fast, FOG)
        assert np.mean(~E.same_bits_or_nan(on, off).reshape(-1, 3).all(1)) > 0.5
    assert not E.same_bits_or_nan(fog_image(False, FOG), fog_image(True, FOG)).all()


# kernel 4 x HAS_BVH x LAY x 20 Shades and kernel 1 x MODE x 20, with fog; fast fog on LAY / MODE 1, slow fog on 0 and 2
CASES = ([(4, bvh, lay, i) for bvh in (1, 0) for lay in (0, 1, 2) for i in range(20)]
         + [(1, 1, mode, i) for mode in (0, 1, 2) for i in range(20)])


def _case_id(c):
    kernel, bvh, lay, i = c
    return (f"k4-{'bvh' if bvh else 'nobvh'}-lay{lay}" if kernel == 4 else f"k1-mode{lay}") + "-" + shade_id(i)


def test_the_cases_cover_every_fog_instance():
    assert len(CASES) == 180 and len(set(CASES)) == 180
    # the LAY rule moves exactly the BVH footprints with spec or NEE fields off the staged top table
    moved = {(bvh, spec, nee) for bvh in (0, 1) for spec in (0, 1) for nee in (0, 1) if fog_lay(bvh, 0, spec, nee) == 1}
    assert moved == {(1, 1, 0), (1, 0, 1), (1, 1, 1)}


@pytest.mark.gpu
@pytest.mark.parametrize("case", CASES, ids=_case_id)
def test_fog_instance(cuda_ctx, ctx_no_wide, loader, monkeypatch, case):  # noqa: F811
    kernel, bvh, lay, i = case
    spec, nee, biome = SHADES[i]
    flags = shade_flags(spec, nee, biome) | FOG
    fast = lay == 1
    p = fog_scene(fast, bvh)
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
        ran = fog_lay(bvh, lay, spec, nee != 0)
        sky = fog_staged(bvh, ran, spec, nee != 0, p.sky.shape[0])
    else:
        ran, sky = lay, 0
    assert ctx.last_render_n(8) == (kernel, bvh, ran, spec, nee, biome, sky, 1)
    assert ctx.last_render() == (kernel, bvh, ran, spec, nee, biome, sky)
    assert_bits(got, fog_image(fast, flags, bvh))


@pytest.mark.gpu
def test_kernel_choice_with_fog(cuda_ctx, loader):
    """Kernel 0 runs the wavefront kernel for a fog launch on the commit-time layouts, as without fog."""
    p = fog_scene(False)
    ctx = loader(cuda_ctx, p, (p.name, False))
    got = _render(ctx, p, SEEDS, 0, FOG)
    assert ctx.last_render_n(8) == (4, 1, 0, 0, 0, 0, fog_staged(1, 0, 0, 0, p.sky.shape[0]), 1)
    assert_bits(got, fog_image(False, FOG))
    _render(ctx, p, SEEDS, 4, 0)
    assert ctx.last_render_n(8)[7] == 0 and ctx.last_render_n(3) == (4, 1, 0)
    assert ctx.last_render_n(0) == ()


@pytest.mark.gpu
@pytest.mark.parametrize("kernel", [0, 1, 4])
def test_selection(cuda_ctx, kernel):
    """The fog switch is on exactly when the flag is set and the scene has fog (sigma > 0); otherwise the launch runs the
    kernel and bits it runs without the flag."""
    base = variant_scene(True)
    for fog in (None, (0.0, 0.5, (1.0, 1.0, 1.0), True), FOG_SLOW):
        p = dataclasses.replace(base, fog=fog)
        upload_scene(cuda_ctx, p)
        cuda_ctx.camera_set(p.projector_type, p.camera)
        off = _render(cuda_ctx, p, SEEDS, kernel, 0)
        rep_off = cuda_ctx.last_render_n(8)
        assert rep_off[7] == 0
        has_fog = fog is not None and fog[0] > 0
        on = _render(cuda_ctx, p, SEEDS, kernel, FOG)
        if has_fog:
            assert cuda_ctx.last_render_n(8) == rep_off[:7] + (1,)
            assert_bits(on, SO.FlagsOracle(p, FOG).render(SEEDS))
        else:
            assert cuda_ctx.last_render_n(8) == rep_off
            assert_bits(on, off)


@pytest.mark.gpu
def test_setter_checks_and_begin_clears(cuda_ctx):
    p = fog_scene(False)
    upload_scene(cuda_ctx, p)
    bad = [(-0.1, 0.5, (1, 1, 1), 0), (float("nan"), 0.5, (1, 1, 1), 0), (float("inf"), 0.5, (1, 1, 1), 0),
           (0.1, -0.01, (1, 1, 1), 0), (0.1, 1.01, (1, 1, 1), 0), (0.1, float("nan"), (1, 1, 1), 0),
           (0.1, 0.5, (1, -1, 1), 0), (0.1, 0.5, (1, 1, float("inf")), 0), (0.1, 0.5, (float("nan"), 1, 1), 0),
           (0.1, 0.5, (1, 1, 1), 2), (0.1, 0.5, (1, 1, 1), -1)]
    for args in bad:
        with pytest.raises(native.ChunkyCuError) as e:
            cuda_ctx.set_fog(*args)
        assert e.value.code == native.CCU_EINVAL, args
    lib = native.load()
    assert lib.ccu_scene_set_fog(cuda_ctx._h, 0.1, 0.5, None, 0) == native.CCU_EINVAL
    for args in [(0.0, 0.0, (0, 0, 0), 0), (0.1, 1.0, (2.0, 0.0, 1.0), 1)]:
        cuda_ctx.set_fog(*args)
    # ccu_scene_begin removes the fog: the same scene uploaded without it renders flag-on as flag-off
    q = dataclasses.replace(p, fog=None)
    upload_scene(cuda_ctx, q)
    cuda_ctx.camera_set(q.projector_type, q.camera)
    on = _render(cuda_ctx, q, SEEDS, 1, FOG)
    assert cuda_ctx.last_render_n(8)[7] == 0
    assert_bits(on, _render(cuda_ctx, q, SEEDS, 1, 0))


@pytest.mark.gpu
def test_group_replicates_fog():
    """Every member of a group of one (and of two where there are two GPUs) renders the fog image after replicate_scene."""
    p = fog_scene(True)
    want = fog_image(True, FOG)
    n = min(native.device_count(), 2)
    for k in sorted({1, n}):
        group = native.Group(devices=list(range(k)))
        try:
            upload_scene(group.member(0), p)
            group.replicate_scene()
            for i in range(k):
                m = group.member(i)
                m.camera_set(p.projector_type, p.camera)
                assert_bits(_render(m, p, SEEDS, 1, FOG), want)
                assert m.last_render_n(8)[7] == 1
        finally:
            group.close()


# the fog footprints of the wavefront kernel that launch: every one without BVHs, and with BVHs those that fit beside the
# staged top table (the others run on LAY 1, the footprints with tops = 0)
FOG_FOOTPRINTS = [fp for fp in FOOTPRINTS if not fp[1] or fog_lay(fp[0], 0, fp[2], fp[3]) == 0]
FOG_BOUNDARY = [(fp, r) for fp in FOG_FOOTPRINTS
                for r in (math.isqrt((Q_SMEM_LIMIT - q_smem_fog(*fp)) // 4), math.isqrt((Q_SMEM_LIMIT - q_smem_fog(*fp)) // 4) + 1)]


@pytest.mark.gpu
@pytest.mark.parametrize("case", FOG_BOUNDARY, ids=lambda c: "-".join(str(v) for v in c[0]) + f"-sky{c[1]}")
def test_fog_sky_staging_boundary(cuda_ctx, loader, monkeypatch, case):
    """The largest square sky that fits behind a fog footprint is staged and one more row is not; biome kernels, sun off
    (the fog's sky blend shows every sky lookup)."""
    (bvh, tops, spec, nee), res = case
    p = dataclasses.replace(E.without_sun(fog_scene(False, bvh)), sky=noise_sky(res, seed=res))
    p = dataclasses.replace(p, name=f"{p.name}_sky{res}")
    flags = BIOME | FOG | (SPEC if spec else 0) | (NEE if nee else 0)
    want = SO.FlagsOracle(p, flags).render(SEEDS)
    monkeypatch.setenv("CCU_SKY_SMEM_MAX", "1048576")
    if not tops:
        monkeypatch.setenv("CCU_NO_TOPS", "1")
    loader(cuda_ctx, p, p.name)
    got = _render(cuda_ctx, p, SEEDS, 4, flags)
    staged = res * res if q_smem_fog(bvh, tops, spec, nee) + res * res * 4 <= Q_SMEM_LIMIT else 0
    assert staged == (res * res if res == math.isqrt((Q_SMEM_LIMIT - q_smem_fog(bvh, tops, spec, nee)) // 4) else 0)
    assert cuda_ctx.last_render_n(8) == (4, bvh, 0 if tops else 1, spec, nee, 1, staged, 1)
    assert_bits(got, want)


SEEDS2 = pass_seeds(2)


@pytest.mark.gpu
@pytest.mark.parametrize("kernel", [0, 1])
def test_bit_identities_1080p(cuda_ctx, kernel):
    """DESIGN §14.5 at 1080p: flag on without fog = flag off; fog with the flag off = no fog; with the sun off, sky density 0
    and a sigma too small to move tau from 1, flag on = flag off."""
    base = E.without_sun(S.mixed_test_scene(64, 1920, 1080))

    def render(p, flags):
        upload_scene(cuda_ctx, p)
        cuda_ctx.camera_set(p.projector_type, p.camera)
        return _render(cuda_ctx, p, SEEDS2, kernel, flags)

    sun = S.mixed_test_scene(64, 1920, 1080)
    ref_sun = render(sun, 0)
    assert_bits(render(sun, FOG), ref_sun)
    assert_bits(render(dataclasses.replace(sun, fog=FOG_SLOW), 0), ref_sun)
    ref = render(base, 0)
    tiny = dataclasses.replace(base, fog=(1e-12, 0.0, (0.5, 0.6, 0.7), False))
    assert_bits(render(tiny, FOG), ref)
    assert cuda_ctx.last_render_n(8)[7] == 1 and cuda_ctx.last_render_n(8)[0] == (4 if kernel == 0 else 1)
