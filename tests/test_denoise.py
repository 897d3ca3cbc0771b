"""The guided denoiser (DESIGN.md §17) in the CPU restatement (specular_oracle.denoise): the round trip of zero iterations,
constant images, albedo, normal and sky edges, invalid pixels, the quality on a rendered scene against a converged one, and,
with the library stubbed, the binding's shape checks and the renderer's feature-then-denoise sequence."""
import ctypes as C
import types

import numpy as np
import pytest

import specular_oracle as SO
from chunkyclplugin_b200 import native
from chunkyclplugin_b200 import scenes as S
from chunkyclplugin_b200.javarandom import pass_seeds
from chunkyclplugin_b200.renderer import CudaPathTracingRenderer, DefaultRenderManager, Scene

F = np.float32


def ulps(got, want):
    """Distance in float32 units in the last place, per element."""
    g = np.asarray(got, F).view(np.int32).astype(np.int64)
    w = np.asarray(want, F).view(np.int32).astype(np.int64)
    return np.abs(g - w)


def round_trip(color, albedo):
    """§17 steps 1 and 4 alone: (double)((c / d) * d) with c = (float)color and d = fmaxf(albedo, 2^-8)."""
    c = np.asarray(color, np.float64).astype(F)
    d = np.fmax(np.asarray(albedo, F), F(2.0 ** -8))
    return ((c / d) * d).astype(np.float64)


def test_zero_iterations_is_the_round_trip():
    rng = np.random.default_rng(1)
    h, w = 23, 31
    color = rng.lognormal(-1.0, 1.5, (h, w, 3))
    albedo = rng.random((h, w, 3), dtype=F)
    albedo[3:6, 4:9] = 0                                    # below the 2^-8 floor
    normal = rng.standard_normal((h, w, 3)).astype(F)
    out = SO.denoise(color, albedo, normal, 0, 4.0)
    np.testing.assert_array_equal(out, round_trip(color, albedo).reshape(-1))
    assert ulps(out, color.astype(F).reshape(-1)).max() <= 1


@pytest.mark.parametrize("iterations", range(0, 9))
def test_a_constant_image_stays_constant(iterations):
    h, w = 40, 56
    albedo = np.broadcast_to(np.array([0.6, 0.4, 0.2], F), (h, w, 3))
    normal = np.broadcast_to(np.array([0, 1, 0], F), (h, w, 3))
    color = np.broadcast_to(np.array([0.3, 0.5, 0.7]), (h, w, 3))
    out = SO.denoise(color, albedo, normal, iterations, 4.0)
    assert ulps(out, color.astype(F).reshape(-1)).max() <= 4


def noisy_halves(h, w, left, right, rng, noise=0.3):
    """Colour = the half's mean colour times one multiplicative noise factor per pixel (about `noise` RMS)."""
    mean = np.empty((h, w, 3))
    mean[:, :w // 2] = left
    mean[:, w // 2:] = right
    factor = np.clip(1 + noise * rng.standard_normal((h, w, 1)), 0.05, None)
    return mean * factor, mean


def test_an_albedo_edge_keeps_its_hues():
    """Two halves of different albedo under the same light, 30 % noise: after five iterations the columns on either side of the
    edge keep their own half's mean colour within 2 %, channel by channel, and their own hue, so no hue crosses the edge."""
    rng = np.random.default_rng(2)
    h, w = 128, 64
    a_left, a_right = np.array([0.8, 0.2, 0.2], F), np.array([0.2, 0.2, 0.8], F)
    color, mean = noisy_halves(h, w, a_left, a_right, rng)
    albedo = np.empty((h, w, 3), F)
    albedo[:, :w // 2], albedo[:, w // 2:] = a_left, a_right
    normal = np.broadcast_to(np.array([0, 1, 0], F), (h, w, 3))
    out = SO.denoise(color, albedo, normal, 5, 4.0).reshape(h, w, 3)
    for x, half, a in ((w // 2 - 1, slice(0, w // 2), a_left), (w // 2, slice(w // 2, w), a_right)):
        np.testing.assert_allclose(out[:, x].mean(axis=0), color[:, half].mean(axis=(0, 1)), rtol=0.02)
        np.testing.assert_allclose(out[:, x] / out[:, x, :1], np.broadcast_to(a / a[0], (h, 3)), rtol=1e-5)
    # and the filter did filter: the noise left is a fraction of the input's
    assert np.std(out[:, 4:w // 2 - 4, 0] / 0.8) < 0.5 * np.std(color[:, 4:w // 2 - 4, 0] / 0.8)


def test_a_normal_edge_and_the_sky_keep_their_levels():
    """One albedo; a floor (0, 1, 0) lit at 1.0 next to a wall (1, 0, 0) lit at 0.25, and a sky band (zero normals) at 2.0 above
    both: each region's edge pixels keep their region's level within 2 %; sky blends with sky only."""
    rng = np.random.default_rng(3)
    h, w = 128, 64
    color, _ = noisy_halves(h, w, 1.0, 0.25, rng)
    albedo = np.full((h, w, 3), 0.5, F)
    color = color * 0.5
    normal = np.zeros((h, w, 3), F)
    normal[:, :w // 2, 1] = 1
    normal[:, w // 2:, 0] = 1
    sky = slice(0, 16)
    normal[sky] = 0
    color[sky] = 0.5 * 2.0 * np.clip(1 + 0.3 * rng.standard_normal((16, w, 1)), 0.05, None)
    out = SO.denoise(color, albedo, normal, 5, 4.0).reshape(h, w, 3)
    ground = slice(16, h)
    np.testing.assert_allclose(out[ground, w // 2 - 1].mean(axis=0), 0.5, rtol=0.02)
    np.testing.assert_allclose(out[ground, w // 2].mean(axis=0), 0.125, rtol=0.02)
    np.testing.assert_allclose(out[15].mean(axis=0), 1.0, rtol=0.02)        # the sky row next to the ground
    np.testing.assert_allclose(out[16, :w // 2].mean(axis=0), 0.5, rtol=0.02)
    assert np.std(out[2:13]) < 0.5 * np.std(color[2:13])                    # the sky was filtered


def test_invalid_pixels_keep_their_values_and_do_not_leak():
    rng = np.random.default_rng(4)
    h, w = 33, 47
    color = rng.lognormal(-1.0, 0.5, (h, w, 3))
    albedo = rng.uniform(0.2, 0.9, (h, w, 3)).astype(F)
    normal = np.broadcast_to(np.array([0, 1, 0], F), (h, w, 3)).copy()
    bad = np.zeros((h, w), bool)
    for (y, x), where, value in (((3, 4), "c", np.nan), ((10, 20), "c", np.inf), ((11, 20), "c", -np.inf), ((20, 30), "a", np.nan),
                                 ((25, 5), "n", np.inf), ((0, 0), "c", np.nan), ((h - 1, w - 1), "a", -np.inf)):
        {"c": color, "a": albedo, "n": normal}[where][y, x, 1] = value
        bad[y, x] = True
    for it in (1, 3, 5, 8):
        out = SO.denoise(color, albedo, normal, it, 4.0).reshape(h, w, 3)
        assert np.isfinite(out[~bad]).all()
        want = round_trip(color, albedo)
        np.testing.assert_array_equal(out[bad], want[bad])


def test_quality_on_a_rendered_scene():
    """mixed_test_scene rendered at 4 and 16 spp, with 16-pass feature buffers, against a 1024-spp render on other seeds: the
    denoised image is closer to the converged one than the noisy image is.  The ratios of RMSEs are the measured ones of
    DESIGN §17.6 with a margin of 0.005 (the restatement is deterministic)."""
    p = S.mixed_test_scene()
    o = SO.FlagsOracle(p, 0)
    ref = o.render(pass_seeds(1024, seed=12345)).astype(np.float64)
    albedo, normal = o.features(pass_seeds(16))
    rmse = lambda x: float(np.sqrt(np.mean((x - ref) ** 2)))        # noqa: E731
    for spp, bar in ((4, 0.969), (16, 0.995)):
        noisy = o.render(pass_seeds(spp)).astype(np.float64)
        out = SO.denoise(noisy, albedo, normal, 5, 4.0, p.width, p.height)
        assert rmse(out) <= bar * rmse(noisy), (spp, rmse(out) / rmse(noisy))


# ------------------------------------------------------------------------------------------------------------------------
# host side, with the library stubbed out
# ------------------------------------------------------------------------------------------------------------------------
class _StubLib:
    def __init__(self):
        self.calls = []

    def ccu_denoise(self, h, w, ht, color, albedo, normal, iterations, sigma, out):
        self.calls.append((w, ht, iterations, sigma.value))
        return native.CCU_OK

    def ccu_last_error(self):
        return b""


def _stub_context(monkeypatch):
    lib = _StubLib()
    monkeypatch.setattr(native, "load", lambda: lib)
    ctx = native.Context.__new__(native.Context)
    ctx._lib, ctx._h, ctx._owned = lib, C.c_void_p(1), False
    return ctx, lib


def test_the_binding_checks_shapes_before_the_call(monkeypatch):
    ctx, lib = _stub_context(monkeypatch)
    h, w = 5, 7
    c, a, n = np.zeros((h, w, 3)), np.zeros((h, w, 3), F), np.zeros((h, w, 3), F)
    with pytest.raises(ValueError):
        ctx.denoise(c.reshape(-1), a, n)                                 # a flat buffer needs width and height
    with pytest.raises(ValueError):
        ctx.denoise(c, a[:, :-1], n)
    with pytest.raises(ValueError):
        ctx.denoise(c, a, n.reshape(-1)[:-3])
    with pytest.raises(ValueError):
        ctx.denoise(c.reshape(-1), a, n, width=w + 1, height=h)
    assert lib.calls == []
    out = ctx.denoise(c, a, n)
    assert out.dtype == np.float64 and out.shape == (h * w * 3,)
    assert lib.calls == [(w, h, 5, 4.0)]
    ctx.denoise(c.reshape(-1), a.reshape(-1), n.reshape(-1), 3, 2.5, width=w, height=h)
    assert lib.calls[-1] == (w, h, 3, 2.5)


class _FakeDenoiseContext:
    def __init__(self):
        self.log = []

    def denoise(self, color, albedo, normal, iterations, sigma_luminance, width=None, height=None):
        self.log.append(("denoise", color.copy(), albedo, normal, iterations, sigma_luminance, width, height))
        return np.full(color.size, 7.0)


def test_renderer_denoise_renders_features_then_denoises(monkeypatch):
    p = S.mixed_test_scene()
    scene = Scene(p)
    scene.sample_buffer[:] = np.arange(scene.sample_buffer.size)
    before = scene.sample_buffer.copy()
    ctx = _FakeDenoiseContext()
    loader = types.SimpleNamespace(instance=types.SimpleNamespace(context=ctx), ensureLoad=lambda s: True)
    renderer = CudaPathTracingRenderer(loader)
    n = p.width * p.height * 3
    feats = (np.linspace(0, 1, n), np.linspace(-1, 1, n))

    def render_features(manager, spp):
        ctx.log.append(("render_features", spp))
        return feats

    monkeypatch.setattr(renderer, "render_features", render_features)
    out = renderer.denoise(DefaultRenderManager(scene), feature_spp=8, iterations=3, sigma_luminance=2.0)
    assert [e[0] for e in ctx.log] == ["render_features", "denoise"]
    assert ctx.log[0][1] == 8
    _, color, albedo, normal, it, sl, w, h = ctx.log[1]
    np.testing.assert_array_equal(color, before)
    assert albedo.dtype == normal.dtype == F
    np.testing.assert_array_equal(albedo, feats[0].astype(F))
    np.testing.assert_array_equal(normal, feats[1].astype(F))
    assert (it, sl, w, h) == (3, 2.0, p.width, p.height)
    assert (out == 7.0).all()
    np.testing.assert_array_equal(scene.sample_buffer, before)
