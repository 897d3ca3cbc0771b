"""CCU_RENDER_EMITTER_SAMPLING on the CPU (DESIGN.md §10): the emitter table commit builds against a numpy restatement, and
the CPU restatement of the estimator (specular_oracle.FlagsOracle) against a closed-form form factor, against the flag-off
render in expectation, and for its variance.  Seeds are fixed, so every statistical check is deterministic."""
import dataclasses
import math
import os
import re

import numpy as np
import pytest

from chunkyclplugin_b200 import native
from chunkyclplugin_b200 import scenes as S
from chunkyclplugin_b200.javarandom import pass_seeds
from oracle import edge_rays as E

import specular_oracle as SO

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
NEE = 8


def cluster_scene(width=32, height=18):
    """A stone floor with a 2 x 2 x 2 glowstone block at even coordinates: one emitting leaf of level 1."""
    pal = S.Palettes()
    vox = np.zeros((16, 16, 16), np.int32)
    vox[:, :2, :] = S.STONE
    vox[6:8, 4:6, 6:8] = S.GLOWSTONE
    tree, depth = S.build_octree(vox, pal.block_mapping)
    cam = S.pinhole_camera((3.3, 7.2, 2.1), 35.0, -30.0, 80.0)
    return S._finish("cluster16", tree, depth, pal, cam, width, height, sun_draw=False)


def deep_indoor():
    """indoor64 in the low corner of a depth-13 world (the deep-world layout)."""
    p = S.indoor_scene(64, 40, 24)
    return dataclasses.replace(p, octree=E.embed_octree(p.octree, 7), octree_depth=p.octree_depth + 7, name="indoor64_deep13")


GRID_SCENES = {
    "indoor64": lambda: S.indoor_scene(64, 32, 18),
    "decorated": lambda: S.terrain_scene(64, 32, 18, seed=11, decorate=True),
    "cluster": cluster_scene,
    "deep13": deep_indoor,
    "none": lambda: S.terrain_scene(64, 32, 18, seed=7),
}


def _native_grid(p):
    return native.debug_emitter_grid(p.octree, p.octree_depth, p.block_palette, p.mat_palette)


@pytest.mark.parametrize("name", list(GRID_SCENES))
def test_grid_matches_numpy(name):
    p = GRID_SCENES[name]()
    want, got = SO.emitter_grid(p), _native_grid(p)
    for k in want:
        assert np.array_equal(np.asarray(got[k]), np.asarray(want[k])), k
    assert want["has_emitters"] == (name != "none")
    if name == "cluster":
        _, level, value = SO._leaves(p.octree, p.octree_depth)
        emits = SO.emitter_blocks(p.block_palette, p.mat_palette)
        assert any(l >= 1 and emits[v] for l, v in zip(level, value) if 0 <= v < emits.size)
        assert want["emit"].shape[0] == 8


def test_grid_lists_hold_the_neighbourhood():
    """Every list holds exactly the emitters whose cell is within Chebyshev distance 1, in ascending order."""
    g = SO.emitter_grid(S.indoor_scene(64, 32, 18))
    cell = (g["emit"][:, :3] - g["g0"]) >> g["shift"]
    dim = g["dim"]
    for ci in range(int(np.prod(dim))):
        c = np.array([ci // (dim[1] * dim[2]), (ci // dim[2]) % dim[1], ci % dim[2]])
        want = np.nonzero(np.abs(cell - c).max(1) <= 1)[0]
        assert np.array_equal(g["list"][g["off"][ci]:g["off"][ci + 1]], want)


def test_no_emitters_renders_as_flag_off():
    p = GRID_SCENES["none"]()
    seeds = pass_seeds(2)
    on = SO.FlagsOracle(p, flags=NEE).render(seeds)
    assert np.array_equal(on, SO.FlagsOracle(p, flags=0).render(seeds))


def test_flags_oracle_keeps_the_specular_restatement():
    p = S.glossy(S.indoor_scene(64, 24, 14))
    seeds = pass_seeds(2)
    assert np.array_equal(SO.FlagsOracle(p, flags=SO.CCU_RENDER_SPECULAR).render(seeds), SO.SpecularOracle(p).render(seeds))


# ---------------------------------------------------------------------------------------------------------
# analytic: a point on a flat floor under one flat-coloured emitter cube
# ---------------------------------------------------------------------------------------------------------
FLOOR_ARGB, EMIT_ARGB, EMIT_BYTE, SCALE = 0xFFC08040, 0xFFE0D0A0, 200, 13.0
CUBE = (7, 3, 8)          # the emitter voxel; the floor is the top of layer y = 1
X0 = (6.3, 2.0, 5.9)      # floor point the rays hit


def analytic_scene(n=4096):
    pal = S.Palettes()
    floor = pal.put_material(S.pack_material(0, 0, textured=False, argb=FLOOR_ARGB))
    lamp = pal.put_material(S.pack_material(0, 0, textured=False, argb=EMIT_ARGB, emittance=EMIT_BYTE / 255.0))
    b_floor = len(pal.blocks)
    pal.blocks += [1, floor]
    b_lamp = len(pal.blocks)
    pal.blocks += [1, lamp]
    vox = np.zeros((16, 16, 16), np.int64)
    vox[:, :2, :] = 1
    vox[CUBE] = 2
    mapping = np.array([0, b_floor, b_lamp], np.int64)
    tree, depth = S.build_octree(vox.astype(np.int32), mapping)
    p = S._finish("analytic", tree, depth, pal, S.pinhole_camera((6, 6, 6), 0, -90), n, 1, sun_draw=False)
    o = np.array([X0[0], 5.0, X0[2]], np.float32)
    d = np.array([0.0, -1.0, 0.0], np.float32)
    rays = np.tile(np.concatenate([o, d]), n).astype(np.float32)
    return dataclasses.replace(p, projector_type=-1, camera=rays, sky_intensity=0.0, sky=np.zeros_like(p.sky))


def form_factor(x, n):
    """Point-to-polygon form factor (Lambert's contour integral) summed over the cube faces x lies outside of."""
    e = np.array(CUBE, np.float64)
    total = 0.0
    for axis in range(3):
        for plane in ((e[axis], -1), (e[axis] + 1, 1)):
            if (x[axis] - plane[0]) * plane[1] <= 0:
                continue
            a, b = [k for k in range(3) if k != axis]
            quad = []
            for (da, db) in ((0, 0), (1, 0), (1, 1), (0, 1)):
                v = e.copy()
                v[axis] = plane[0]
                v[a] += da
                v[b] += db
                quad.append(v - x)
            f = 0.0
            for i in range(4):
                r0, r1 = quad[i], quad[(i + 1) % 4]
                c = np.cross(r0, r1)
                ang = math.acos(np.clip(np.dot(r0, r1) / np.linalg.norm(r0) / np.linalg.norm(r1), -1, 1))
                f += ang * np.dot(c / np.linalg.norm(c), n)
            total += abs(f) / (2 * math.pi)
    return total


def _argb(c):
    return np.array([(c >> 16) & 0xFF, (c >> 8) & 0xFF, c & 0xFF], np.float64) / 256.0


def analytic_expectation():
    ff = form_factor(np.array(X0, np.float64), np.array([0.0, 1.0, 0.0]))
    return _argb(FLOOR_ARGB) * _argb(EMIT_ARGB) ** 2 * (EMIT_BYTE / 255.0) * SCALE * ff


@pytest.mark.parametrize("flags", [0, NEE], ids=["off", "on"])
def test_analytic_floor(flags):
    p = analytic_scene()
    px = SO.FlagsOracle(p, flags=flags, max_depth=2, emitter_scale=SCALE).render(pass_seeds(1)).reshape(-1, 3).astype(np.float64)
    want = analytic_expectation()
    se = px.std(0, ddof=1) / math.sqrt(px.shape[0])
    assert np.all(np.abs(px.mean(0) - want) < 4 * se + 1e-3 * want), (px.mean(0), want, se)


def test_analytic_floor_standard_error():
    """Same spp: the flag-on standard error is well below the flag-off one (measured ratio 0.12)."""
    p = analytic_scene()
    se = {}
    for flags in (0, NEE):
        px = SO.FlagsOracle(p, flags=flags, max_depth=2, emitter_scale=SCALE).render(pass_seeds(1)).reshape(-1, 3)
        se[flags] = px.std(0, ddof=1).mean()
    assert se[NEE] < 0.3 * se[0], se


# ---------------------------------------------------------------------------------------------------------
# a small indoor scene: unbiased against the flag-off render, and less noisy at equal spp
# ---------------------------------------------------------------------------------------------------------
W, H, P = 64, 36, 512


def _passes(p, flags, seeds):
    o = SO.FlagsOracle(p, flags=flags)
    return np.stack([o.render([s]).reshape(-1, 3) for s in seeds])


@pytest.fixture(scope="module")
def indoor_passes():
    p = S.indoor_scene(64, W, H)
    seeds = pass_seeds(2 * P + 2048)
    return _passes(p, NEE, seeds[:P]), _passes(p, 0, seeds[P:2 * P]), _passes(p, 0, seeds[2 * P:]).mean(0)


def _regions(a):
    img = a.reshape(a.shape[0], H, W, 3).mean(-1)
    return np.stack([img[:, y:y + 12, x:x + 16].mean((1, 2)) for y in range(0, H, 12) for x in range(0, W, 16)], 1)


def test_unbiased_against_flag_off(indoor_passes):
    """Region means over 512 passes each, disjoint seed streams; the tolerance is the standard error measured from the
    passes.  Measured: largest |z| 2.3 over 12 regions."""
    on, off, _ = indoor_passes
    ron, roff = _regions(on), _regions(off)
    z = (ron.mean(0) - roff.mean(0)) / np.sqrt(ron.var(0, ddof=1) / P + roff.var(0, ddof=1) / P)
    assert np.abs(z).max() < 4.5, z


@pytest.mark.parametrize("spp", [4, 16])
def test_variance_reduction(indoor_passes, spp):
    """RMSE against a 2048-pass flag-off render at equal spp.  Measured ratio on / off: 0.33 at 4 spp, 0.34 at 16 spp."""
    on, off, ref = indoor_passes
    r_on = np.sqrt(((on[:spp].mean(0) - ref) ** 2).mean())
    r_off = np.sqrt(((off[:spp].mean(0) - ref) ** 2).mean())
    assert r_on < 0.6 * r_off, (r_on, r_off)


def test_set_params_checks_the_flags_first():
    """ccu_render_set_params validates the parameters before the context, so a host can check them without a GPU: an unknown
    bit is named as such, while the known ones get as far as the missing context."""
    import ctypes as C
    lib = native.load()
    for flags, msg in ((NEE | 4 | 2 | 1, "null"), (16, "unknown render flags"), (NEE | 32, "unknown render flags")):
        p = native.RenderParams(256, 5, 13.0, 0, flags)
        assert lib.ccu_render_set_params(None, C.byref(p)) == native.CCU_EINVAL
        assert msg in lib.ccu_last_error().decode(), (flags, lib.ccu_last_error())


def test_flag_constant_agrees():
    hdr = open(os.path.join(ROOT, "include", "chunkycu.h")).read()
    java = open(os.path.join(ROOT, "java", "dev", "thatredox", "chunkynative", "cuda", "ChunkyCu.java")).read()
    assert int(re.search(r"#define CCU_RENDER_EMITTER_SAMPLING (\d+)", hdr).group(1)) == NEE
    assert int(re.search(r"RENDER_EMITTER_SAMPLING = (\d+)", java).group(1)) == NEE
    assert native.CCU_RENDER_EMITTER_SAMPLING == NEE == SO.CCU_RENDER_EMITTER_SAMPLING
