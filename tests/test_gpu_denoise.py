"""The guided denoiser on the GPU (DESIGN.md §17): ccu_denoise against the CPU restatement (specular_oracle.denoise) bit for bit
on random inputs with sky regions, zero albedo and non-finite pixels, at canvas shapes from 1 x 1 to 1920 x 1080; after real
renders and feature buffers; an output that aliases the colour; calls that grow and shrink the scratch; a call inside an open
render window; a group member's context; and the argument checks."""
import ctypes as C

import numpy as np
import pytest

import specular_oracle as SO
from chunkyclplugin_b200 import native
from chunkyclplugin_b200 import scenes as S
from chunkyclplugin_b200.javarandom import pass_seeds
from chunkyclplugin_b200.renderer import upload_scene

F = np.float32
SIGMAS = (4.0, 0.75)


def random_inputs(w, h, seed):
    """A piecewise image: 8 x 8 blocks of one albedo (some zero) and one normal (some the sky's zero normal) each, a smooth
    irradiance with 30 % multiplicative noise per pixel, and a sprinkling of NaN and inf components in every buffer."""
    rng = np.random.default_rng(seed)
    by, bx = (h + 7) // 8, (w + 7) // 8
    palette = np.array([[0.8, 0.2, 0.2], [0.2, 0.2, 0.8], [0.5, 0.5, 0.5], [0.0, 0.0, 0.0], [0.9, 0.85, 0.7]], F)
    normals = np.array([[0, 1, 0], [1, 0, 0], [0, 0, 0], [0, 0.6, 0.8], [-0.48, 0.6, 0.64]], F)
    pick = lambda k: np.kron(rng.integers(0, k, (by, bx)), np.ones((8, 8), int))[:h, :w]     # noqa: E731
    albedo = palette[pick(len(palette))]
    albedo = (albedo + rng.uniform(-0.02, 0.02, albedo.shape)).clip(0, 1).astype(F)
    normal = normals[pick(len(normals))].copy()
    yy, xx = np.mgrid[0:h, 0:w]
    light = 0.5 + 0.4 * np.sin(xx / 17.0)[..., None] * np.cos(yy / 11.0)[..., None]
    color = (albedo * light * np.clip(1 + 0.3 * rng.standard_normal((h, w, 1)), 0, None)).astype(np.float64)
    n = w * h
    for buf, values in ((color, (np.nan, np.inf, -np.inf)), (albedo, (np.nan, np.inf)), (normal, (np.nan, -np.inf))):
        flat = buf.reshape(-1)
        k = max(1, n // 500) if n > 4 else 0
        idx = rng.choice(flat.size, k, replace=False) if k else []
        flat[idx] = rng.choice(values, len(idx))
    return color, albedo, normal


def assert_same(got, want):
    got, want = np.asarray(got, np.float64), np.asarray(want, np.float64)
    nan = np.isnan(want)
    np.testing.assert_array_equal(np.isnan(got), nan)
    np.testing.assert_array_equal(got[~nan].view(np.uint64), want[~nan].view(np.uint64))


SHAPES = [(1, 1), (1, 97), (97, 1), (33, 65), (127, 129), (1920, 1080)]


@pytest.mark.gpu
@pytest.mark.parametrize("shape", SHAPES, ids=lambda s: "%dx%d" % s)
def test_denoise_matches_the_restatement(cuda_ctx, shape):
    w, h = shape
    color, albedo, normal = random_inputs(w, h, w * 7919 + h)
    launches = cuda_ctx.launch_count()
    calls = 0
    for iterations in (0, 1, 3, 5, 8):
        for sigma in SIGMAS:
            got = cuda_ctx.denoise(color, albedo, normal, iterations, sigma)
            calls += 2 + iterations
            want = SO.denoise(color, albedo, normal, iterations, sigma)
            assert_same(got, want)
            assert cuda_ctx.last_kernel_ms() > 0
    assert cuda_ctx.launch_count() == launches + calls


def rendered(ctx, p, spp):
    """Sample buffer (float64, Chunky layout) and 16-pass feature buffers of scene p from the GPU."""
    upload_scene(ctx, p)
    ctx.camera_set(p.projector_type, p.camera)
    ctx.render_begin(p.width, p.height)
    try:
        ctx.render_passes(np.asarray(pass_seeds(spp), np.int32))
        img, n = ctx.render_read()
        assert n == spp
        albedo, normal = ctx.render_features(np.asarray(pass_seeds(16, seed=3), np.int32))
    finally:
        ctx.render_end()
    return np.asarray(img, np.float64), albedo, normal


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["config1", "entities"])
def test_pipeline_matches_the_restatement(cuda_ctx, name):
    p = S.terrain_scene(256, 320, 180) if name == "config1" else S.entity_scene(128, 160, 90, n_world=96, n_actor=8, subdiv=1)
    color, albedo, normal = rendered(cuda_ctx, p, 4)
    for iterations in (1, 5):
        got = cuda_ctx.denoise(color, albedo, normal, iterations, 4.0, width=p.width, height=p.height)
        assert_same(got, SO.denoise(color, albedo, normal, iterations, 4.0, p.width, p.height))
        assert not np.array_equal(got, color)


@pytest.mark.gpu
def test_output_may_alias_the_colour_and_the_scratch_grows_and_shrinks(cuda_ctx):
    lib = native.load()
    vp = lambda a: a.ctypes.data_as(C.c_void_p)      # noqa: E731
    for (w, h) in ((33, 65), (640, 360), (7, 5), (127, 129), (1, 1), (640, 360)):
        color, albedo, normal = random_inputs(w, h, w + h)
        want = SO.denoise(color, albedo, normal, 3, 4.0)
        assert_same(cuda_ctx.denoise(color, albedo, normal, 3, 4.0), want)
        buf = np.ascontiguousarray(color.reshape(-1))
        rc = lib.ccu_denoise(cuda_ctx._h, w, h, vp(buf), vp(albedo.reshape(-1)), vp(normal.reshape(-1)), 3, C.c_float(4.0), vp(buf))
        assert rc == native.CCU_OK
        assert_same(buf, want)


@pytest.mark.gpu
@pytest.mark.parametrize("kernel", [1, 4])
def test_a_denoise_call_leaves_the_render_window_alone(cuda_ctx, kernel):
    p = S.mixed_test_scene()
    upload_scene(cuda_ctx, p)
    cuda_ctx.camera_set(p.projector_type, p.camera)
    seeds = np.asarray(pass_seeds(4), np.int32)
    color, albedo, normal = random_inputs(p.width, p.height, 5)

    def window(with_denoise):
        cuda_ctx.render_set_params(kernel=kernel)
        try:
            cuda_ctx.render_begin(p.width, p.height)
            cuda_ctx.render_passes(seeds[:2])
            rep = cuda_ctx.last_render_n(9)
            out = cuda_ctx.denoise(color, albedo, normal, 5, 4.0) if with_denoise else None
            rep_after = cuda_ctx.last_render_n(9)
            cuda_ctx.render_passes(seeds[2:], block=False)
            img, spp = cuda_ctx.render_read()
            cuda_ctx.render_end()
            return img, spp, rep, rep_after, out
        finally:
            cuda_ctx.render_set_params()

    img0, spp0, rep0, _, _ = window(False)
    img1, spp1, rep1, rep1_after, out = window(True)
    assert spp0 == spp1 == 4
    assert rep0 == rep1 == rep1_after
    np.testing.assert_array_equal(np.asarray(img1).view(np.uint32), np.asarray(img0).view(np.uint32))
    assert_same(out, SO.denoise(color, albedo, normal, 5, 4.0))


@pytest.mark.gpu
def test_group_member_denoises():
    w, h = 96, 54
    color, albedo, normal = random_inputs(w, h, 9)
    group = native.Group(devices=[0])
    try:
        got = group.member(0).denoise(color, albedo, normal, 5, 4.0)
    finally:
        group.close()
    assert_same(got, SO.denoise(color, albedo, normal, 5, 4.0))


@pytest.mark.gpu
def test_argument_checks(cuda_ctx):
    lib = native.load()
    w, h = 8, 6
    color, albedo, normal = random_inputs(w, h, 1)
    c, a, n = color.reshape(-1).copy(), albedo.reshape(-1).copy(), normal.reshape(-1).copy()
    out = np.zeros_like(c)
    vp = lambda x: x.ctypes.data_as(C.c_void_p)      # noqa: E731
    ok = (cuda_ctx._h, w, h, vp(c), vp(a), vp(n), 5, C.c_float(4.0), vp(out))
    assert lib.ccu_denoise(*ok) == native.CCU_OK

    def with_(i, v):
        args = list(ok)
        args[i] = v
        return args

    bad = [with_(0, None), with_(3, None), with_(4, None), with_(5, None), with_(8, None), with_(1, 0), with_(2, 0), with_(1, -3),
           with_(2, -1), with_(6, -1), with_(6, native.CCU_DENOISE_MAX_ITERATIONS + 1),
           with_(7, C.c_float(0.0)), with_(7, C.c_float(-1.0)), with_(7, C.c_float(float("inf"))), with_(7, C.c_float(float("nan")))]
    big = list(ok)
    big[1], big[2] = 2 ** 31 - 1, 2 ** 31 - 1            # 3 * W * H is beyond int64
    bad.append(big)
    launches = cuda_ctx.launch_count()
    for args in bad:
        assert lib.ccu_denoise(*args) == native.CCU_EINVAL, args
    assert cuda_ctx.launch_count() == launches
    for it in (0, native.CCU_DENOISE_MAX_ITERATIONS):
        assert lib.ccu_denoise(*with_(6, it)) == native.CCU_OK
