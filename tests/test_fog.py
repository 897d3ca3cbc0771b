"""CCU_RENDER_FOG on the CPU (DESIGN.md §14): the transmittance kernel, the restatement (specular_oracle.FlagsOracle) against
closed forms of the sky blend and the extinction, the bit-identities of §14.5, and the loader of Chunky's fog keys."""
import dataclasses
import math
import os

import numpy as np
import pytest

from chunkyclplugin_b200 import octree2
from chunkyclplugin_b200 import scenes as S
from chunkyclplugin_b200.javarandom import pass_seeds
from oracle import edge_rays as E

import specular_oracle as SO

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
FOG = SO.CCU_RENDER_FOG
F = np.float32


def test_expf_within_one_ulp():
    xs = np.concatenate([-np.geomspace(1e-8, 103.0, 2000), [0.0, -0.5, -1.0, -20.0]]).astype(np.float32)
    for x in xs:
        got = np.float32(SO.dm_expf(float(x)))
        want = math.exp(float(x))
        assert abs(float(got) - want) <= float(np.spacing(np.float32(want))), x
    assert SO.dm_expf(-200.0) == 0.0 and SO.dm_expf(0.0) == 1.0


def _rays(width, height, origin, seed):
    """Pre-generated rays from one origin in random, unnormalised directions."""
    rng = np.random.default_rng(seed)
    d = rng.normal(size=(width * height, 3)) * rng.uniform(0.5, 3.0, size=(width * height, 1))
    o = np.broadcast_to(np.asarray(origin, np.float64), d.shape)
    return np.ascontiguousarray(np.concatenate([o, d], 1).astype(np.float32).reshape(-1)), d.astype(np.float32)


def _scene(vox, rays, width, height, sun=False):
    pal = S.Palettes()
    tree, depth = S.build_octree(vox, pal.block_mapping)
    p = S._finish("fog", tree, depth, pal, rays, width, height, sun_draw=sun)
    flat = np.zeros((16, 16, 4), np.uint8)
    flat[...] = (200, 150, 90, 255)
    return dataclasses.replace(p, projector_type=-1, sky=flat)


def test_sky_blend_closed_form():
    """An empty world, a flat sky, no sun: every pixel is ((S (1 - f) + C f) T) with f = density * g(y)."""
    w, h = 24, 16
    rays, d = _rays(w, h, (8.0, 8.0, 8.0), 3)
    p = _scene(np.zeros((16, 16, 16), np.int32), rays, w, h)
    fog = (0.05, 0.7, (0.3, 0.5, 0.9), False)
    seeds = pass_seeds(1)
    sky = SO.FlagsOracle(p, 0).render(seeds).reshape(-1, 3)        # S(d): flat, the same for every ray
    got = SO.FlagsOracle(p, FOG, fog=fog).render(seeds).reshape(-1, 3)
    L = np.sqrt(np.array([math.fsum([float(c) * float(c) for c in v]) for v in d], np.float64)).astype(F)
    y = (d[:, 1] / L).astype(F)
    g = np.where(y > 0, (F(1) - y) * (F(1) - y), F(1)).astype(F)
    f = (F(fog[1]) * g).astype(F)
    want = (sky * (F(1) - f)[:, None] + np.asarray(fog[2], F)[None, :] * f[:, None]).astype(F)
    np.testing.assert_array_max_ulp(got, want, maxulp=4)
    assert not np.array_equal(got, sky)


def test_extinction_of_an_emissive_wall():
    """The sun off, a glowstone wall in front of every ray, max_depth 1: each pixel is tau(a) times its fog-free value, with
    a = the distance to the wall along the ray."""
    w, h = 16, 12
    rng = np.random.default_rng(5)
    d = np.stack([np.ones(w * h), rng.uniform(-0.4, 0.4, w * h), rng.uniform(-0.4, 0.4, w * h)], 1) * rng.uniform(0.5, 2.0, (w * h, 1))
    o = np.array([1.3, 8.2, 8.1])
    rays = np.concatenate([np.broadcast_to(o, d.shape), d], 1).astype(np.float32).reshape(-1)
    vox = np.zeros((16, 16, 16), np.int32)
    vox[12, :, :] = S.GLOWSTONE
    p = dataclasses.replace(_scene(vox, rays, w, h), name="wall")
    sigma = 0.08
    seeds = pass_seeds(1)
    off = SO.FlagsOracle(p, 0, max_depth=1).render(seeds).reshape(-1, 3).astype(np.float64)
    on = SO.FlagsOracle(p, FOG, fog=(sigma, 0.0, (1.0, 1.0, 1.0), False), max_depth=1).render(seeds).reshape(-1, 3)
    a = (12.0 - o[0]) / d[:, 0] * np.linalg.norm(d, axis=1)
    want = off * np.exp(-sigma * a)[:, None]
    assert (off > 0).all()
    np.testing.assert_allclose(on, want, rtol=2e-5)


def test_bit_identities():
    """§14.5: the flag without fog, and fog without the flag, render the flag-off bits; so do the flag and fog with the sun
    off, sky density 0 and a sigma for which tau is 1.0f on every segment."""
    p = S.mixed_test_scene(64, 48, 27)
    seeds = pass_seeds(2)
    off = SO.FlagsOracle(p, 0).render(seeds)
    assert np.array_equal(SO.FlagsOracle(p, FOG).render(seeds).view(np.uint32), off.view(np.uint32))
    fogged = dataclasses.replace(p, fog=(0.05, 0.5, (1.0, 1.0, 1.0), True))
    assert np.array_equal(SO.FlagsOracle(fogged, 0).render(seeds).view(np.uint32), off.view(np.uint32))
    assert not E.same_bits_or_nan(SO.FlagsOracle(fogged, FOG).render(seeds), off).all()
    q = E.without_sun(p)
    ref = SO.FlagsOracle(q, 0).render(seeds)
    tiny = SO.FlagsOracle(q, FOG, fog=(1e-12, 0.0, (0.5, 0.6, 0.7), False)).render(seeds)
    assert np.array_equal(tiny.view(np.uint32), ref.view(np.uint32))
    assert not np.array_equal(SO.FlagsOracle(q, FOG, fog=(0.05, 0.0, (0.5, 0.6, 0.7), False)).render(seeds), ref)


def test_fog_from_json_on_the_benchmark_scene():
    sigma, sky, color, fast = octree2.fog_from_json(os.path.join(ROOT, "tests", "golden", "opencl_test_fog.json"))
    assert sigma == 0.0 and sky == 1.0 and fast is True
    assert color == (0.42814502293337064, 0.5858024691358026, 1.0)


def test_fog_from_json_converts_the_density(tmp_path):
    path = tmp_path / "scene.json"
    path.write_text('{"fogDensity": 0.5, "skyFogDensity": 0.25, "fogColor": {"red": 1, "green": 0.5, "blue": 0}, "fastFog": false}')
    assert octree2.fog_from_json(str(path)) == (0.5 * octree2.FOG_EXTINCTION_FACTOR, 0.25, (1.0, 0.5, 0.0), False)


C_FOG = (0.6, 0.7, 0.9)


def _lit_scene(vox, o, d, altitude, azimuth):
    """Black untextured blocks, a flat sky and a flat sun texture, the sun at (altitude, azimuth), rays o + t d."""
    w = d.shape[0]
    rays = np.concatenate([np.broadcast_to(o, d.shape), d], 1).astype(np.float32).reshape(-1)
    pal = S.Palettes()
    black = pal.put_material(S.pack_material(0, 0, textured=False, argb=S._s32(0xFF000000)))
    pal.blocks[2 * S.STONE + 1] = black
    tree, depth = S.build_octree(vox, pal.block_mapping)
    p = S._finish("lit", tree, depth, pal, rays, w, 1)
    p.atlas[...] = (255, 230, 190, 255)
    sky = np.zeros((16, 16, 4), np.uint8)
    sky[...] = (120, 140, 200, 255)
    return dataclasses.replace(p, projector_type=-1, sky=sky, sun=S.pack_sun(*pal.sun_tex, altitude=altitude, azimuth=azimuth))


def _sun_radiance(altitude, azimuth):
    """S(w) for w in the sun disc: the flag-off image of one ray at the disc's centre in an empty world."""
    r = math.cos(altitude)
    d = np.array([[math.cos(azimuth) * r, math.sin(altitude), math.sin(azimuth) * r]], np.float32)
    p = _lit_scene(np.zeros((16, 16, 16), np.int32), np.array([8.0, 8.0, 8.0]), d, altitude, azimuth)
    return SO.FlagsOracle(p, 0).render(pass_seeds(1)).astype(np.float64)


def _rays_to_wall(n, x0, rng):
    d = np.stack([np.ones(n), rng.uniform(-0.05, 0.05, n), rng.uniform(-0.3, 0.3, n)], 1) * rng.uniform(0.5, 2.0, (n, 1))
    return np.array([x0, 4.5, 8.1]), d


def test_in_scatter_closed_form():
    """Fast fog, flat sun and sky, the sun unoccluded from every scattering point, a black wall at max_depth 1: each pixel is
    C (1 - tau(a)) S(w) exactly as the wall contributes nothing."""
    alt, az = 1.0, math.pi                       # the sun towards -x, away from the wall at x = 12
    rng = np.random.default_rng(9)
    o, d = _rays_to_wall(256, 1.3, rng)
    vox = np.zeros((16, 16, 16), np.int32)
    vox[12, :, :] = S.STONE
    p = _lit_scene(vox, o, d, alt, az)
    sigma = 0.06
    got = SO.FlagsOracle(p, FOG, fog=(sigma, 0.0, C_FOG, True), max_depth=1).render(pass_seeds(1)).reshape(-1, 3)
    a = (12.0 - o[0]) / d[:, 0] * np.linalg.norm(d, axis=1)
    want = np.asarray(C_FOG)[None, :] * (1 - np.exp(-sigma * a))[:, None] * _sun_radiance(alt, az).reshape(1, 3)
    assert (want > 0).all()
    np.testing.assert_allclose(got, want, rtol=1e-4)
    assert not SO.FlagsOracle(p, 0, max_depth=1).render(pass_seeds(1)).any()


@pytest.mark.parametrize("fast", [True, False], ids=["fast", "slow"])
def test_light_shaft_under_half_a_roof(fast):
    """The sun at the zenith and a black roof over the far half of every camera ray: the in-scattered light converges to the
    share of the unoccluded value that the lit half carries (1/2 for fast fog; (1 - e^(-e/2)) / (1 - e^(-e)) for the other),
    within 5 standard errors of the sample mean."""
    alt, az = math.pi / 2, 0.0
    rng = np.random.default_rng(21)
    n, passes = 2048, 8
    o, d = _rays_to_wall(n, 2.0, rng)
    d[:, 1] = 0.0                                # horizontal rays: the roof's edge is at x = 7 for every ray
    vox = np.zeros((16, 16, 16), np.int32)
    vox[12, :, :] = S.STONE
    vox[7:12, 14, :] = S.STONE
    p = _lit_scene(vox, o, d.astype(np.float32), alt, az)
    sigma = 0.08
    got = SO.FlagsOracle(p, FOG, fog=(sigma, 0.0, C_FOG, fast), max_depth=1).render(pass_seeds(passes)).reshape(-1, 3)
    a = (12.0 - o[0]) / d[:, 0] * np.linalg.norm(d, axis=1)
    e = sigma * a
    full = np.asarray(C_FOG)[None, :] * (1 - np.exp(-e))[:, None] * _sun_radiance(alt, az).reshape(1, 3)
    share = got[:, 0] / full[:, 0]
    want = 0.5 if fast else float(np.mean((1 - np.exp(-e / 2)) / (1 - np.exp(-e))))
    bound = 5 * float(np.std(share)) / math.sqrt(n) + 1e-3
    assert abs(float(np.mean(share)) - want) < bound, (float(np.mean(share)), want, bound)
    assert 0.02 < bound < 0.1
