"""The denoiser's feature buffers (DESIGN.md §16) in the CPU restatement (FlagsOracle.features): the anchor to the parity oracle's
first hit, closed forms on a floor, the sky and a full cloud cover, the biome tint, the flags that do not act, and the PFM
writer."""
import ctypes as C
import dataclasses
import types

import numpy as np
import pytest

import oracle
import specular_oracle as SO
from chunkyclplugin_b200 import native
from chunkyclplugin_b200 import scenes as S
from chunkyclplugin_b200.javarandom import pass_seeds
from chunkyclplugin_b200.pfm import write_pfm
from chunkyclplugin_b200.renderer import CudaPathTracingRenderer, DefaultRenderManager, Scene
from test_biome_tint import FIXED, argb_floats, floor_scene
from test_gpu_variants import variant_scene

BIOME, CLOUDS, FOG = SO.CCU_RENDER_BIOME_TINT, SO.CCU_RENDER_CLOUDS, SO.CCU_RENDER_FOG
F = np.float32


def canonical(a):
    """float32 bits with -0 read as +0: the running mean folds the first pass as (0 * 0 + v) / 1, which maps -0 to +0."""
    return (np.ascontiguousarray(a, F) + F(0)).view(np.uint32)


def small_entity_scene():
    return S.entity_scene(128, 160, 90, n_world=96, n_actor=8, subdiv=1)


def anchor_check(p, flags=0):
    seed = pass_seeds(3)[2]
    fh = oracle.Oracle(p).first_hit(seed)
    albedo, normal = SO.FlagsOracle(p, flags).features([seed])
    hit = fh["kind"] != 0
    assert hit.mean() > 0.3
    color = fh["color"].reshape(-1, 4)[:, :3]
    np.testing.assert_array_equal(albedo.reshape(-1, 3)[hit].view(np.uint32), canonical(color[hit]))
    np.testing.assert_array_equal(normal.reshape(-1, 3)[hit].view(np.uint32), canonical(fh["normal"].reshape(-1, 3)[hit]))
    assert not normal.reshape(-1, 3)[~hit].any()
    return albedo, normal


@pytest.mark.parametrize("name", ["mixed", "entities"])
def test_one_pass_is_the_first_hit(name):
    """One pass: on every hit pixel the albedo is the first hit's colour and the normal its normal, bit for bit (up to the sign
    of a zero); the biome and clouds flags on a scene without biome colours or clouds change nothing."""
    p = S.mixed_test_scene() if name == "mixed" else small_entity_scene()
    a, n = anchor_check(p)
    b, m = SO.FlagsOracle(p, BIOME | CLOUDS).features([pass_seeds(3)[2]])
    assert np.array_equal(a.view(np.uint32), b.view(np.uint32)) and np.array_equal(n.view(np.uint32), m.view(np.uint32))


@pytest.mark.parametrize("passes", [1, 7, 64])
def test_floor_normals_are_exact(passes):
    """A flat floor filling the view: the normal of every pixel is exactly (0, 1, 0) whatever the number of passes.  The rays
    come down inside voxel columns, away from their edges (where the block test may report a side face)."""
    p = floor_scene(32, 24)
    rng = np.random.default_rng(passes)
    n = p.width * p.height
    o = np.stack([rng.integers(4, 60, n) + rng.uniform(0.25, 0.75, n), np.full(n, 20.0),
                  rng.integers(4, 60, n) + rng.uniform(0.25, 0.75, n)], 1)
    d = np.stack([rng.uniform(-0.005, 0.005, n), -np.ones(n), rng.uniform(-0.005, 0.005, n)], 1)
    rays = np.concatenate([o, d], 1).astype(F).reshape(-1)
    _, normal = SO.FlagsOracle(p, 0).features(pass_seeds(passes), rays=rays)
    want = np.tile(np.array([0, 1, 0], F), n)
    np.testing.assert_array_equal(normal.view(np.uint32), want.view(np.uint32))


def floor_albedo(p):
    """Per pixel of floor_scene: the biome-tinted colour of the one column the pixel's footprint lies in, or NaN where the
    footprint straddles columns (test_biome_tint.floor_expected before the shading)."""
    cam = np.asarray(p.camera, np.float64)
    o, M = cam[0:3], cam[3:12].reshape(3, 3)
    hw, ih = p.width / (2.0 * p.height), 1.0 / p.height
    px, py = np.meshgrid(np.arange(p.width), np.arange(p.height))
    cx, cz = [], []
    for jx, jy in ((0, 0), (1, 0), (0, 1), (1, 1)):
        x = -hw + (px + jx) * ih
        y = -0.5 + (py + jy) * ih
        d = np.stack([cam[14] * x, cam[14] * y, np.ones_like(x)], -1) @ M.T
        t = (1.0 - o[1]) / d[..., 1]
        cx.append(np.floor(o[0] + t * d[..., 0]))
        cz.append(np.floor(o[2] + t * d[..., 2]))
    cx, cz = np.stack(cx), np.stack(cz)
    one = (cx.min(0) == cx.max(0)) & (cz.min(0) == cz.max(0))
    chunks, rgb = p.biome
    tile = {(int(a), int(b)): i for i, (a, b) in enumerate(chunks)}
    base = F(192) / F(256)
    out = np.full((p.height, p.width, 3), np.nan, F)
    for j, i in zip(*np.nonzero(one)):
        x, z = int(cx[0, j, i]), int(cz[0, j, i])
        k = tile.get((x >> 4, z >> 4))
        c = rgb[k, 1, (z & 15) * 16 + (x & 15)] if k is not None else argb_floats(FIXED[1])
        out[j, i] = base * c.astype(F)
    return out.reshape(-1)


def fold(v, passes):
    """The running mean of `passes` equal values v, in float32 as the kernels fold it."""
    v = np.asarray(v, F)
    buf = np.zeros_like(v)
    for k in range(passes):
        buf = (buf * F(k) + v) / F(k + 1)
    return buf


@pytest.mark.parametrize("passes", [1, 7])
def test_biome_floor_matches_closed_form(passes):
    """The albedo of a biome-tinted grass floor is the tile's texel times the material colour, folded `passes` times."""
    p = floor_scene()
    want = fold(floor_albedo(p), passes)
    got, _ = SO.FlagsOracle(p, BIOME).features(pass_seeds(passes))
    ok = ~np.isnan(want)
    assert ok.sum() > 0.4 * want.size
    np.testing.assert_array_equal(got[ok].view(np.uint32), want[ok].view(np.uint32))
    assert len(np.unique(want[ok])) > 100
    # without the flag: the fixed grass tint everywhere
    plain, _ = SO.FlagsOracle(p, 0).features(pass_seeds(passes))
    fixed = fold(F(192) / F(256) * argb_floats(FIXED[1]).astype(F), passes)
    np.testing.assert_array_equal(plain.reshape(-1, 3)[ok.reshape(-1, 3).all(1)].view(np.uint32),
                                  np.broadcast_to(fixed, (int(ok.reshape(-1, 3).all(1).sum()), 3)).view(np.uint32))


def rays_from(o, d):
    return np.concatenate([np.broadcast_to(o, d.shape), d], 1).astype(F).reshape(-1)


def test_sky_is_clamped_and_has_no_normal():
    """Rays that leave the world upwards: albedo = min(sky radiance, 1), the radiance being what a one-segment render of the
    same rays sees; normal 0."""
    rng = np.random.default_rng(5)
    d = rng.normal(size=(4096, 3))
    d[:, 1] = np.abs(d[:, 1]) + 0.05
    base = S.mixed_test_scene()
    rays = rays_from(np.array([32.0, 80.0, 32.0]), d)
    p = dataclasses.replace(base, projector_type=-1, camera=rays, width=64, height=64, sky_intensity=2.5)
    albedo, normal = SO.FlagsOracle(p, 0).features([pass_seeds(1)[0]])
    sky = oracle.Oracle(p, max_depth=1).render([pass_seeds(1)[0]])
    assert (sky > 1).mean() > 0.1 and (sky < 1).mean() > 0.1
    np.testing.assert_array_equal(albedo.view(np.uint32), np.minimum(sky, F(1)).view(np.uint32))
    assert not normal.any()
    # FlagsOracle.features(rays=...) is the same as a scene with those rays
    q = dataclasses.replace(base, width=64, height=64, sky_intensity=2.5)
    a2, _ = SO.FlagsOracle(q, 0).features([pass_seeds(1)[0]], rays=rays)
    assert np.array_equal(a2.view(np.uint32), albedo.view(np.uint32))


def test_full_cloud_cover_is_white_with_the_top_face_normal():
    rng = np.random.default_rng(7)
    d = rng.normal(size=(4096, 3))
    d[:, 1] = -(np.abs(d[:, 1]) + 0.3)
    base = S.mixed_test_scene()
    p = dataclasses.replace(base, projector_type=-1, camera=rays_from(np.array([32.0, 90.0, 32.0]), d), width=64, height=64)
    q = S.with_clouds(p, np.ones((256, 256), np.uint8), size=3.0, y0=70.0, y1=74.0)
    seeds = pass_seeds(3)
    albedo, normal = SO.FlagsOracle(q, CLOUDS).features(seeds)
    np.testing.assert_array_equal(albedo, np.ones_like(albedo))
    np.testing.assert_array_equal(normal.view(np.uint32), np.tile(np.array([0, 1, 0], F), 4096).view(np.uint32))
    # without the flag the same rays see the world and the sky
    plain, _ = SO.FlagsOracle(q, 0).features(seeds)
    assert (plain != 1).mean() > 0.5


def test_flags_that_do_not_act():
    """Specular, emitter sampling (all three kinds) and fog leave the features as they are; the biome and clouds switches change
    them on a scene that has biome colours and clouds.  (The restatement applies no-sun to the scene, not as a flag; that
    the library's features ignore CCU_RENDER_NO_SUN is a GPU test.)"""
    from test_clouds import fixture_clouds
    p = dataclasses.replace(fixture_clouds(variant_scene(True)), fog=(0.02, 0.5, (0.5, 0.6, 0.7), 0))
    seeds = pass_seeds(2)
    for extra in (0, BIOME, CLOUDS, BIOME | CLOUDS):
        a, n = SO.FlagsOracle(p, extra).features(seeds)
        for f in (4, 8, 8 | 128, 8 | 256, 8 | 128 | 256, FOG, 4 | 8 | FOG):
            b, m = SO.FlagsOracle(p, extra | f).features(seeds)
            assert np.array_equal(a.view(np.uint32), b.view(np.uint32)), (extra, f)
            assert np.array_equal(n.view(np.uint32), m.view(np.uint32)), (extra, f)
    plain, _ = SO.FlagsOracle(p, 0).features(seeds)
    assert not np.array_equal(SO.FlagsOracle(p, BIOME).features(seeds)[0], plain)
    assert not np.array_equal(SO.FlagsOracle(p, CLOUDS).features(seeds)[0], plain)


def test_running_mean_is_the_render_kernels():
    """n passes fold as buf = (buf * k + v) / (k + 1) in float32, in pass order, from 0."""
    p = S.mixed_test_scene()
    seeds = pass_seeds(5)
    singles = [SO.FlagsOracle(p, 0).features([s]) for s in seeds]
    want_a = np.zeros_like(singles[0][0])
    want_n = np.zeros_like(singles[0][1])
    for k, (a, n) in enumerate(singles):
        want_a = (want_a * F(k) + a) / F(k + 1)
        want_n = (want_n * F(k) + n) / F(k + 1)
    got_a, got_n = SO.FlagsOracle(p, 0).features(seeds)
    np.testing.assert_array_equal(got_a.view(np.uint32), want_a.view(np.uint32))
    np.testing.assert_array_equal(got_n.view(np.uint32), want_n.view(np.uint32))


def read_pfm(path):
    with open(path, "rb") as f:
        assert f.readline() == b"PF\n"
        w, h = (int(v) for v in f.readline().split())
        scale = float(f.readline())
        data = np.frombuffer(f.read(), "<f4" if scale < 0 else ">f4")
    assert data.size == w * h * 3
    return w, h, scale, data.reshape(h, w, 3)[::-1].reshape(-1)


def test_pfm_round_trip(tmp_path):
    rng = np.random.default_rng(1)
    w, h = 7, 5
    rgb = rng.normal(size=w * h * 3).astype(F)
    path = str(tmp_path / "a.pfm")
    write_pfm(path, rgb.astype(np.float64), w, h)
    rw, rh, scale, back = read_pfm(path)
    assert (rw, rh, scale) == (w, h, -1.0)
    np.testing.assert_array_equal(back, rgb)
    # the first row of the file is the bottom row of the image
    raw = np.frombuffer(open(path, "rb").read()[len(b"PF\n7 5\n-1\n"):], "<f4")
    np.testing.assert_array_equal(raw[:w * 3], rgb[(h - 1) * w * 3:])
    with pytest.raises(ValueError):
        write_pfm(path, rgb[:-1], w, h)


# ------------------------------------------------------------------------------------------------------------------------
# host side, with the library stubbed out
# ------------------------------------------------------------------------------------------------------------------------
class _StubLib:
    """The entry points Context.render_features reaches; n_floats = None: no render target."""

    def __init__(self, n_floats):
        self.n_floats = n_floats
        self.feature_calls = []

    def ccu_render_device_buffer(self, h, ptr, n):
        if self.n_floats is None:
            return native.CCU_ESTATE
        n._obj.value = self.n_floats
        return native.CCU_OK

    def ccu_render_features(self, h, seeds, n_passes, albedo, normal):
        self.feature_calls.append((n_passes, albedo, normal))
        return native.CCU_OK

    def ccu_last_error(self):
        return b"no render target"


def _stub_context(monkeypatch, n_floats):
    lib = _StubLib(n_floats)
    monkeypatch.setattr(native, "load", lambda: lib)
    ctx = native.Context.__new__(native.Context)
    ctx._lib, ctx._h, ctx._owned = lib, C.c_void_p(1), False
    return ctx, lib


def test_render_features_takes_the_canvas_from_the_library(monkeypatch):
    """A context that has no render target (before render_begin, or a group member whose Python object never saw the canvas)
    raises CCU_ESTATE before ccu_render_features is called; with one, the outputs hold the target's 3 * W * H floats."""
    ctx, lib = _stub_context(monkeypatch, None)
    with pytest.raises(native.ChunkyCuError) as e:
        ctx.render_features([1, 2])
    assert e.value.code == native.CCU_ESTATE
    assert lib.feature_calls == []
    ctx, lib = _stub_context(monkeypatch, 3 * 7 * 5)
    a, n = ctx.render_features([1, 2])
    assert a.shape == n.shape == (105,) and a.dtype == n.dtype == np.float32
    assert len(lib.feature_calls) == 1 and lib.feature_calls[0][0] == 2
    a, n = ctx.render_features([1], normal=False)
    assert a.shape == (105,) and n is None and lib.feature_calls[-1][2] is None


class _FakeFeatureContext:
    """What CudaPathTracingRenderer.render_features uses of a context; every call returns fresh random means."""

    def __init__(self, n_floats):
        self.n_floats = n_floats
        self.seeds, self.outputs, self.log = [], [], []
        self.rng = np.random.default_rng(11)

    def camera_set(self, projector_type, settings):
        self.log.append("camera_set")

    def render_begin(self, width, height):
        self.log.append(("render_begin", width, height))

    def render_end(self):
        self.log.append("render_end")

    def render_features(self, seeds):
        self.seeds.append(np.asarray(seeds, np.int32).copy())
        out = (self.rng.random(self.n_floats, dtype=np.float32), self.rng.random(self.n_floats, dtype=np.float32))
        self.outputs.append(out)
        return out


def test_renderer_splits_long_feature_renders():
    """More than CCU_FEATURES_MAX_PASSES passes: calls of at most that many, on render()'s seeds in order, whose means are
    combined in double, weighted by their pass counts; the render target is closed afterwards."""
    p = S.mixed_test_scene()
    ctx = _FakeFeatureContext(p.width * p.height * 3)
    loader = types.SimpleNamespace(instance=types.SimpleNamespace(context=ctx), ensureLoad=lambda scene: True)
    spp = native.CCU_FEATURES_MAX_PASSES + 1
    albedo, normal = CudaPathTracingRenderer(loader).render_features(DefaultRenderManager(Scene(p)), spp)
    assert [s.size for s in ctx.seeds] == [native.CCU_FEATURES_MAX_PASSES, 1]
    np.testing.assert_array_equal(np.concatenate(ctx.seeds), np.asarray(pass_seeds(spp), np.int32))
    assert ctx.log[-1] == "render_end" and ("render_begin", p.width, p.height) in ctx.log
    (a1, n1), (a2, n2) = ctx.outputs
    m = native.CCU_FEATURES_MAX_PASSES
    want_a = (a1.astype(np.float64) * m + a2.astype(np.float64) * 1) / (m + 1)
    want_n = (n1.astype(np.float64) * m + n2.astype(np.float64) * 1) / (m + 1)
    assert albedo.dtype == np.float64
    np.testing.assert_array_equal(albedo, want_a)
    np.testing.assert_array_equal(normal, want_n)

