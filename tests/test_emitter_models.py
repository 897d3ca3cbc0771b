"""CCU_RENDER_EMITTER_MODELS on the CPU (DESIGN.md §12): the wider emitter table and primitive lists commit builds against a
numpy restatement, and the CPU restatement of the estimator (specular_oracle.FlagsOracle) against a closed-form form factor,
against the bound of §12 item 6, against the flag-off render in expectation, and for its variance.  Seeds are fixed, so
every statistical check is deterministic."""
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
from test_emitter_sampling import EMIT_ARGB, EMIT_BYTE, FLOOR_ARGB, SCALE, X0, _argb

import specular_oracle as SO

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
NEE, NEAR, MODELS = 8, 128, 256
RHO = 0.125


def lantern_scene(width=32, height=18):
    """Lanterns on a dirt floor; material 0 (the lantern body's +z face, SURVEY Q10) made emissive, so that the +z face is
    an emitting primitive while the disabled -y face is not."""
    pal = S.Palettes()
    S.add_model_lights(pal)
    pal.mat[4] = 200
    vox = np.zeros((16, 16, 16), np.int32)
    vox[:, :2, :] = S.DIRT
    vox[4, 2, 5] = vox[9, 2, 9] = vox[9, 3, 9] = S.LANTERN
    tree, depth = S.build_octree(vox, pal.block_mapping)
    return S._finish("lanterns16", tree, depth, pal, S.pinhole_camera((3.3, 7.2, 2.1), 35.0, -30.0, 80.0), width, height,
                     sun_draw=False)


def deep_models():
    p = S.indoor_models_scene(64, 40, 24)
    return dataclasses.replace(p, octree=E.embed_octree(p.octree, 7), octree_depth=p.octree_depth + 7, name="indoor_models64_deep13")


# ---------------------------------------------------------------------------------------------------------
# analytic: a floor point under one flat-coloured, downward-facing emitting quad inside its voxel
# ---------------------------------------------------------------------------------------------------------
QV = (7, 3, 8)                 # the quad's voxel
QLO, QHI, QY = 0.25, 0.75, 0.5  # block-local: x, z in [QLO, QHI] at y = QY


def analytic_quad_scene(n=4096):
    pal = S.Palettes()
    floor = pal.put_material(S.pack_material(0, 0, textured=False, argb=FLOOR_ARGB))
    lamp = pal.put_material(S.pack_material(0, 0, textured=False, argb=EMIT_ARGB, emittance=EMIT_BYTE / 255.0))
    w = QHI - QLO
    qptr = len(pal.quad)
    pal.quad += [1] + list(S.f2i([QLO, QY, QLO, w, 0, 0, 0, 0, w, 0.0, 1.0, 0.0, 1.0])) + [lamp, 0]
    b_floor = len(pal.blocks)
    pal.blocks += [1, floor]
    b_quad = len(pal.blocks)
    pal.blocks += [3, qptr]
    vox = np.zeros((16, 16, 16), np.int64)
    vox[:, :2, :] = 1
    vox[QV] = 2
    tree, depth = S.build_octree(vox.astype(np.int32), np.array([0, b_floor, b_quad], np.int64))
    p = S._finish("analytic_quad", tree, depth, pal, S.pinhole_camera((6, 6, 6), 0, -90), n, 1, sun_draw=False)
    o = np.array([X0[0], 5.0, X0[2]], np.float32)
    rays = np.tile(np.concatenate([o, [0.0, -1.0, 0.0]]), n).astype(np.float32)
    return dataclasses.replace(p, projector_type=-1, camera=rays, sky_intensity=0.0, sky=np.zeros_like(p.sky))


def polygon_form_factor(x, n, poly):
    """Point-to-polygon form factor (Lambert's contour integral)."""
    f = 0.0
    for i in range(len(poly)):
        r0, r1 = poly[i] - x, poly[(i + 1) % len(poly)] - x
        c = np.cross(r0, r1)
        ang = math.acos(np.clip(np.dot(r0, r1) / np.linalg.norm(r0) / np.linalg.norm(r1), -1, 1))
        f += ang * np.dot(c / np.linalg.norm(c), n)
    return abs(f) / (2 * math.pi)


def analytic_quad_expectation():
    e = np.array(QV, np.float64)
    poly = [e + [a, QY, b] for a, b in ((QLO, QLO), (QHI, QLO), (QHI, QHI), (QLO, QHI))]
    ff = polygon_form_factor(np.array(X0, np.float64), np.array([0.0, 1.0, 0.0]), poly)
    return _argb(FLOOR_ARGB) * _argb(EMIT_ARGB) ** 2 * (EMIT_BYTE / 255.0) * SCALE * ff


def _analytic(flags):
    o = SO.FlagsOracle(analytic_quad_scene(), flags=flags, max_depth=2, emitter_scale=SCALE)
    return o.render(pass_seeds(1)).reshape(-1, 3).astype(np.float64)


GRID_SCENES = {
    "indoor_models": lambda: S.indoor_models_scene(64, 32, 18),
    "decorated_lit": lambda: S.emissive_models(S.terrain_scene(64, 32, 18, seed=11, decorate=True)),
    "models_only": lambda: analytic_quad_scene(4),
    "lanterns": lantern_scene,
    "deep13": deep_models,
    "none": lambda: S.terrain_scene(64, 32, 18, seed=7),
}


@pytest.mark.parametrize("name", list(GRID_SCENES))
def test_table_matches_numpy(name):
    p = GRID_SCENES[name]()
    want, got = SO.emitter_grid(p, models=True), native.debug_emitter_models(p)
    for k in want:
        assert np.array_equal(np.asarray(got[k]), np.asarray(want[k])), k
    assert want["has_emitters"] == (name != "none")
    if name == "lanterns":
        h = want["head"][S.LANTERN * 2]
        kinds = want["prim"][4 * h + 8::16][:want["prim"][4 * h]]
        # body: -x, +x, +y, -z and the +z face of material 0 (-y disabled); cap: its +z face only
        assert list(kinds) == [0, 1, 3, 4, 5, 5], kinds
    if name == "decorated_lit":
        assert (want["head"][want["emit"][:, 3]] < 0).any(), "cube and model emitters share the lists"


def test_cube_only_scene_renders_as_bit_8():
    p = S.indoor_scene(64, 24, 14)
    assert not SO.emitter_grid(p, models=True)["has_emitters"]
    seeds = pass_seeds(2)
    assert np.array_equal(SO.FlagsOracle(p, flags=NEE | MODELS).render(seeds), SO.FlagsOracle(p, flags=NEE).render(seeds))


@pytest.mark.parametrize("flags", [0, NEE | MODELS, NEE | MODELS | NEAR], ids=["off", "models", "models_near"])
def test_analytic_quad(flags):
    """The per-pixel samples against the closed-form form factor within 4 standard errors.  With the voxel occluding its own
    primitive (a shadow ray that counts the block hit beyond its limit), the flag-on mean would be 0."""
    px = _analytic(flags)
    want = analytic_quad_expectation()
    se = px.std(0, ddof=1) / math.sqrt(px.shape[0])
    assert np.all(np.abs(px.mean(0) - want) < 4 * se + 1e-3 * want), (px.mean(0), want, se)


def test_analytic_quad_standard_error():
    """Same spp: the flag-on standard error is well below the flag-off one (measured ratio 0.0059)."""
    se = {f: _analytic(f).std(0, ddof=1).mean() for f in (0, NEE | MODELS)}
    assert se[NEE | MODELS] < 0.05 * se[0], se


# ---------------------------------------------------------------------------------------------------------
# contact: a flat-coloured torch standing on a floor, floor points next to its stick
# ---------------------------------------------------------------------------------------------------------
GAPS = (1e-3, 1e-2, 0.05, 0.1, 0.2, 0.4)
REPS = 32
TV = (7, 3, 8)                  # the torch's voxel; the floor's top is y = 3
STICK_A, STICK_B, STICK_T = 7 / 16, 9 / 16, 10 / 16


def contact_points():
    cx, cz = TV[0], TV[2]
    pts = []
    for g in GAPS:
        for a in (0.45, 0.5):
            pts += [(cx + STICK_A - g, cz + a), (cx + STICK_B + g, cz + a), (cx + a, cz + STICK_A - g), (cx + a, cz + STICK_B + g)]
    return np.array(pts, np.float64)


def contact_scene():
    """One pre-generated downward ray per pixel, REPS pixels per floor point, black sky and the sun off: with max_depth 2 each
    1-pass pixel is the one emitter sample of its floor hit."""
    pal = S.Palettes()
    floor = pal.put_material(S.pack_material(0, 0, textured=False, argb=FLOOR_ARGB))
    lamp = pal.put_material(S.pack_material(0, 0, textured=False, argb=EMIT_ARGB, emittance=EMIT_BYTE / 255.0))
    qptr = len(pal.quad)
    pal.quad += S._torch_quads(lamp)
    b_floor = len(pal.blocks)
    pal.blocks += [1, floor]
    b_torch = len(pal.blocks)
    pal.blocks += [3, qptr]
    vox = np.zeros((16, 16, 16), np.int64)
    vox[:, :TV[1], :] = 1
    vox[TV] = 2
    tree, depth = S.build_octree(vox.astype(np.int32), np.array([0, b_floor, b_torch], np.int64))
    pts = contact_points()
    p = S._finish("torch_contact", tree, depth, pal, S.pinhole_camera((6, 6, 6), 0, -90), pts.shape[0] * REPS, 1, sun_draw=False)
    rays = np.zeros((pts.shape[0], REPS, 6), np.float32)
    rays[:, :, 0], rays[:, :, 1], rays[:, :, 2] = pts[:, None, 0], TV[1] + 0.3, pts[:, None, 1]
    rays[:, :, 4] = -1.0
    p = dataclasses.replace(p, projector_type=-1, camera=rays.reshape(-1), sky_intensity=0.0, sky=np.zeros_like(p.sky))
    return E.without_sun(p)


def contact_bound():
    """§12 item 6 for the floor's hits: T = the floor colour, N = 1, m = 5 quads, A_max = a side of the stick"""
    m, a_max = 5, (STICK_B - STICK_A) * STICK_T
    factor = max(1.0, m * a_max / (math.pi * RHO * RHO))
    return _argb(FLOOR_ARGB) * _argb(EMIT_ARGB) ** 2 * (EMIT_BYTE / 255.0) * SCALE * factor


def test_contact_contributions_are_bounded():
    """Every 1-pass pixel is one emitter sample, and none exceeds the bound with the near field; without it the area
    sampler's 1/d2 weight exceeds it next to the stick."""
    p = contact_scene()
    bound = contact_bound() * (1 + 1e-5)
    near = SO.FlagsOracle(p, flags=NEE | MODELS | NEAR, max_depth=2, emitter_scale=SCALE).render(pass_seeds(1)).reshape(-1, 3)
    assert np.all(near <= bound), (near.max(0), bound)
    assert near.max() > 0
    area = SO.FlagsOracle(p, flags=NEE | MODELS, max_depth=2, emitter_scale=SCALE).render(pass_seeds(1)).reshape(-1, 3)
    assert np.any(area > bound), (area.max(0), bound)


# ---------------------------------------------------------------------------------------------------------
# the small torch-lit indoor scene: unbiased against the flag-off render, and less noisy at equal spp
# ---------------------------------------------------------------------------------------------------------
W, H, P = 64, 36, 512


def _passes(p, flags, seeds):
    o = SO.FlagsOracle(p, flags=flags)
    return np.stack([o.render([s]).reshape(-1, 3) for s in seeds])


def _regions(a):
    img = a.reshape(a.shape[0], H, W, 3).mean(-1)
    return np.stack([img[:, y:y + 12, x:x + 16].mean((1, 2)) for y in range(0, H, 12) for x in range(0, W, 16)], 1)


@pytest.fixture(scope="module")
def indoor_passes():
    p = S.indoor_models_scene(64, W, H)
    seeds = pass_seeds(2 * P + 2048)
    return (_passes(p, NEE | MODELS, seeds[:P]), _passes(p, NEE | MODELS | NEAR, seeds[:P]), _passes(p, 0, seeds[P:2 * P]),
            _passes(p, 0, seeds[2 * P:]).mean(0))


@pytest.mark.parametrize("which", [0, 1], ids=["models", "models_near"])
def test_unbiased_against_flag_off(indoor_passes, which):
    """Region means over 512 passes each, disjoint seed streams; the tolerance is the standard error measured from the
    passes."""
    on, off = indoor_passes[which], indoor_passes[2]
    ron, roff = _regions(on), _regions(off)
    z = (ron.mean(0) - roff.mean(0)) / np.sqrt(ron.var(0, ddof=1) / P + roff.var(0, ddof=1) / P)
    assert np.abs(z).max() < 4.5, z


@pytest.mark.parametrize("spp", [4, 16])
def test_variance_reduction(indoor_passes, spp):
    """RMSE against a 2048-pass flag-off render at equal spp, averaged over the disjoint windows of the 512 passes.  Measured
    ratio on / off: 8 | 256 0.83 at 4 spp, 0.88 at 16 spp; 8 | 256 | 128 0.85 / 0.88.  Most of this scene's light reaches
    a pixel over more than one bounce, which NEE at the first hit does not shorten, hence the modest gain."""
    on, near, off, ref = indoor_passes

    def rmse(a):
        return np.mean([np.sqrt(((a[i:i + spp].mean(0) - ref) ** 2).mean()) for i in range(0, P, spp)])

    r_off = rmse(off)
    assert rmse(near) < 0.95 * r_off, (rmse(near), r_off)
    assert rmse(on) < 0.95 * r_off, (rmse(on), r_off)


def test_set_params_needs_emitter_sampling():
    """256 alone and 256 | 128 are refused, naming the flag they need; 8 | 256 and 8 | 256 | 128 get as far as the missing
    context."""
    import ctypes as C
    lib = native.load()
    for flags, msg in ((MODELS, "CCU_RENDER_EMITTER_MODELS needs CCU_RENDER_EMITTER_SAMPLING"),
                       (MODELS | NEAR, "needs CCU_RENDER_EMITTER_SAMPLING"), (MODELS | 4 | 2 | 1, "needs CCU_RENDER_EMITTER_SAMPLING"),
                       (NEE | MODELS, "null"), (NEE | MODELS | NEAR, "null"), (NEE | MODELS | NEAR | 4 | 2 | 1, "null")):
        p = native.RenderParams(256, 5, 13.0, 0, flags)
        assert lib.ccu_render_set_params(None, C.byref(p)) == native.CCU_EINVAL
        assert msg in lib.ccu_last_error().decode(), (flags, lib.ccu_last_error())


def test_flag_constant_agrees():
    hdr = open(os.path.join(ROOT, "include", "chunkycu.h")).read()
    java = open(os.path.join(ROOT, "java", "dev", "thatredox", "chunkynative", "cuda", "ChunkyCu.java")).read()
    assert int(re.search(r"#define CCU_RENDER_EMITTER_MODELS (\d+)", hdr).group(1)) == MODELS
    assert int(re.search(r"RENDER_EMITTER_MODELS = (\d+)", java).group(1)) == MODELS
    assert native.CCU_RENDER_EMITTER_MODELS == MODELS == SO.CCU_RENDER_EMITTER_MODELS
