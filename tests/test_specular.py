"""CCU_RENDER_SPECULAR on the CPU oracle: specular, metallic and rough materials from word 5 of the packed material (DESIGN
"Beyond the reference: specular materials").  The reference shades every surface diffuse, so there is nothing to be bit-exact
against: materials without a word 5 must render exactly as without the flag, a perfect mirror must show an emitter at its
closed-form value, and the event mix and the roughness blend must hold statistically."""
import os
import re

import numpy as np
import pytest

from chunkyclplugin_b200 import scenes as S
from chunkyclplugin_b200.javarandom import pass_seeds

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
EMITTER_SCALE = 13.0
FLOOR_TOP = 1.0              # the floor is the y = 0 layer of full cubes
EMIT_Y = 20                  # the emitters are the y = EMIT_Y layer over EMIT_X x EMIT_Z
EMIT_X, EMIT_Z = (10, 22), (20, 28)
EMIT_ARGB, EMIT_BYTE = 0xFFF0C080, 200
MIRROR_CAM = dict(pos=(16.3, 6.2, 3.7), yaw=0.0, pitch=-42.0, fov=40.0)


def _flat_scene(floor_words, emitter_words=None, sky_rgb=(0, 0, 0), sky_intensity=0.0, cam=MIRROR_CAM, width=96, height=64,
                max_world=32, gradient=False):
    """A 32^3 world: a floor of full cubes (material `floor_words`), optionally a rectangle of emissive full cubes at
    y = EMIT_Y, a uniform (or gradient) sky, no sun, pre-generated rays through the pixel centres (no jitter)."""
    pal_mat = list(floor_words)
    blocks = [0, 0, 1, 0]
    types = np.zeros((max_world,) * 3, np.int32)
    types[:, 0, :] = 1
    if emitter_words is not None:
        blocks += [1, len(pal_mat)]
        pal_mat += list(emitter_words)
        types[EMIT_X[0]:EMIT_X[1], EMIT_Y, EMIT_Z[0]:EMIT_Z[1]] = 2
    tree, depth = S.build_octree(types, np.arange(len(blocks) // 2, dtype=np.int64) * 2)
    atlas = np.zeros((1, 16, 16, 4), np.uint8)
    if gradient:
        sky = S.gradient_sky(32)
    else:
        sky = np.zeros((16, 16, 4), np.uint8)
        sky[..., :3] = sky_rgb
        sky[..., 3] = 255
    cam15 = S.pinhole_camera(cam["pos"], cam["yaw"], cam["pitch"], cam["fov"])
    return S.PackedScene(
        octree=tree, octree_depth=depth, block_palette=S._i32(blocks), quad_models=np.zeros(1, np.int32),
        aabb_models=np.zeros(1, np.int32), world_bvh=S.EMPTY_BVH.copy(), actor_bvh=S.EMPTY_BVH.copy(),
        bvh_trigs=np.zeros(1, np.int32), atlas=atlas, mat_palette=S._i32(pal_mat), sky=sky, sky_intensity=sky_intensity,
        sun=S.pack_sun((16 << 16) | 16, 0, draw=False), projector_type=-1, camera=S.pregenerated_rays(cam15, width, height),
        width=width, height=height, name="flat")


def mirror_scene(metal: bool, floor_argb: int = 0xFFE0A040):
    """A perfect mirror floor (white specular sp = 1, or a metal me = 1 of colour floor_argb) under a black sky, with the
    emitter rectangle out of the camera's direct view (every camera ray points down)."""
    word = S.specular_word(metalness=1.0) if metal else S.specular_word(specular=1.0)
    floor = S.pack_material(0, 0, textured=False, argb=S._s32(floor_argb))
    floor[5] = word
    emitter = S.pack_material(0, 0, textured=False, argb=S._s32(EMIT_ARGB), emittance=EMIT_BYTE / 255.0)
    assert emitter[4] == EMIT_BYTE
    return _flat_scene(floor, emitter)


def argb_color(argb: int) -> np.ndarray:
    """utils.h:6-14 (byte / 256) as float32 r, g, b"""
    return np.array([((argb >> 16) & 0xFF) / 256.0, ((argb >> 8) & 0xFF) / 256.0, (argb & 0xFF) / 256.0], np.float32)


def mirror_expectation(p, metal: bool, floor_argb: int = 0xFFE0A040, margin: float = 0.05):
    """Per pixel: the closed-form value where the mirrored camera ray lands inside the emitter rectangle by `margin`, 0
    where it misses it by `margin`, NaN (not checked) in between.  The value is applyRayColor's (kernel.h:33-44) for the
    emitter after the mirror bounce, in float32 and in its operation order: (c_e * (em * 13)) * (t * c_e) with t = 1 behind
    a white mirror and t = floor colour behind a metal one."""
    rays = p.camera.reshape(-1, 6).astype(np.float64)
    o, d = rays[:, :3], rays[:, 3:]
    assert (d[:, 1] < 0).all(), "the emitters must be out of the camera's direct view"
    t = (FLOOR_TOP - o[:, 1]) / d[:, 1]
    hit = o + d * t[:, None]
    on_floor = (hit[:, 0] > margin) & (hit[:, 0] < 32 - margin) & (hit[:, 2] > margin) & (hit[:, 2] < 32 - margin)
    r = d * np.array([1.0, -1.0, 1.0])
    # where the mirrored ray enters (q0) and leaves (q1) the emitter layer EMIT_Y <= y <= EMIT_Y + 1
    q0 = hit + r * ((EMIT_Y - hit[:, 1]) / r[:, 1])[:, None]
    q1 = hit + r * ((EMIT_Y + 1 - hit[:, 1]) / r[:, 1])[:, None]
    inside = ((q0[:, 0] > EMIT_X[0] + margin) & (q0[:, 0] < EMIT_X[1] - margin) & (q0[:, 2] > EMIT_Z[0] + margin)
              & (q0[:, 2] < EMIT_Z[1] - margin))
    # a miss crosses the whole layer beyond one edge of the rectangle (it can enter a side face otherwise)
    outside = np.zeros_like(inside)
    for k, (lo, hi) in ((0, EMIT_X), (2, EMIT_Z)):
        outside |= (q0[:, k] < lo - margin) & (q1[:, k] < lo - margin)
        outside |= (q0[:, k] > hi + margin) & (q1[:, k] > hi + margin)
    ce = argb_color(EMIT_ARGB)
    em = np.float32(np.float32(EMIT_BYTE) / np.float32(255.0))
    t_floor = argb_color(floor_argb) if metal else np.ones(3, np.float32)
    value = (ce * (em * np.float32(EMITTER_SCALE))) * (t_floor * ce)
    want = np.full((rays.shape[0], 3), np.nan, np.float32)
    want[on_floor & inside] = value
    want[on_floor & outside] = 0.0
    return want.reshape(-1), int((on_floor & inside).sum()), int((on_floor & outside).sum())


def assert_mirror(img, want):
    checked = ~np.isnan(want)
    bad = np.nonzero(checked & (img != want))[0]
    assert bad.size == 0, (bad[:6] // 3, img[bad[:6]], want[bad[:6]])


def _oracle(p, specular=False, **kw):
    """the parity oracle, or with specular=True its restatement of CCU_RENDER_SPECULAR"""
    import oracle
    from specular_oracle import SpecularOracle
    return (SpecularOracle if specular else oracle.Oracle)(p, emitter_scale=EMITTER_SCALE, **kw)


@pytest.mark.parametrize("name", ["terrain64", "decorated", "mixed", "indoor", "entities"])
def test_zero_words_render_as_without_the_flag(scenes, name):
    """Every existing scene has word 5 = 0 everywhere: no event draws, so the specular restatement renders exactly what the
    parity oracle renders (this also holds its restated intersection functions to the oracle's)."""
    p = scenes(name)
    assert not (p.mat_palette[5::6] != 0).any()
    seeds = pass_seeds(2)
    off = _oracle(p).render(seeds)
    on = _oracle(p, specular=True).render(seeds)
    assert np.array_equal(on.view(np.uint32), off.view(np.uint32))


@pytest.mark.parametrize("metal", [False, True], ids=["white_mirror", "metal_mirror"])
def test_mirror_shows_the_emitter_at_its_closed_form_value(metal):
    p = mirror_scene(metal)
    want, n_in, n_out = mirror_expectation(p, metal)
    assert n_in > 200 and n_out > 200
    img = _oracle(p, max_depth=2, specular=True).render(pass_seeds(1))
    assert_mirror(img, want)
    # without the flag the floor is diffuse: the emitter is reached by a diffuse bounce only, never at the mirror value
    off = _oracle(p, max_depth=2).render(pass_seeds(1))
    inside = ~np.isnan(want) & (want != 0)
    assert (off[inside] != want[inside]).mean() > 0.9


def _floor_and_sky(p):
    import oracle
    kind = oracle.Oracle(p).first_hit(0)["kind"]
    return kind == 1, kind == 0


@pytest.mark.parametrize("s", [0.25, 0.7])
def test_event_mix_is_s_times_mirror_plus_rest_times_diffuse(s):
    """Floor colour c, specular s under a uniform sky, no sun: a sample is L (specular event, white) or c L (diffuse event,
    bounce to the sky), so the image mean over the floor is s L + (1 - s) c L."""
    argb = 0xFF4080C0
    floor = S.pack_material(0, 0, textured=False, argb=S._s32(argb), specular=s)
    p = _flat_scene(floor, sky_rgb=(200, 150, 100), sky_intensity=1.5, cam=dict(pos=(16.3, 4.2, 3.7), yaw=0.0, pitch=-10.0, fov=60.0))
    floor_px, sky_px = _floor_and_sky(p)
    assert floor_px.sum() > 2000 and sky_px.sum() > 100
    img = _oracle(p, specular=True).render(pass_seeds(16)).reshape(-1, 3).astype(np.float64)
    L = img[np.nonzero(sky_px)[0][0]]
    sp = int(s * 255.0) / 255.0
    want = sp * L + (1 - sp) * argb_color(argb).astype(np.float64) * L
    px = img[floor_px]
    se = px.std(axis=0) / np.sqrt(px.shape[0])
    assert (np.abs(px.mean(axis=0) - want) < 5 * se).all(), (px.mean(axis=0), want, se)


def test_roughness_one_is_the_diffuse_floor():
    """sp = 1, ro = 1: the direction is the cosine-weighted one, the throughput stays 1 (white specular event), so the floor
    converges to the white diffuse floor (flag off) divided by its colour 255 / 256."""
    white = S.pack_material(0, 0, textured=False, argb=S._s32(0xFFFFFFFF))
    rough = S.pack_material(0, 0, textured=False, argb=S._s32(0xFFFFFFFF), specular=1.0, roughness=1.0)
    cam = dict(pos=(16.3, 4.2, 3.7), yaw=0.0, pitch=-10.0, fov=60.0)
    p_rough = _flat_scene(rough, sky_intensity=1.0, cam=cam, gradient=True)
    p_diffuse = _flat_scene(white, sky_intensity=1.0, cam=cam, gradient=True)
    floor_px, _ = _floor_and_sky(p_rough)
    seeds = pass_seeds(16)
    a = _oracle(p_rough, specular=True).render(seeds).reshape(-1, 3)[floor_px].astype(np.float64) * (255 / 256)
    b = _oracle(p_diffuse).render(seeds).reshape(-1, 3)[floor_px].astype(np.float64)
    se = np.sqrt(a.var(axis=0) / a.shape[0] + b.var(axis=0) / b.shape[0])
    assert (np.abs(a.mean(axis=0) - b.mean(axis=0)) < 5 * se).all(), (a.mean(axis=0), b.mean(axis=0), se)
    assert not np.array_equal(a, b)      # different random streams: the event draw comes first


def test_flag_constant_agrees_across_header_bindings_and_java():
    from chunkyclplugin_b200 import native
    hdr = open(os.path.join(ROOT, "include", "chunkycu.h")).read()
    assert re.search(r"#define CCU_RENDER_SPECULAR 4\b", hdr)
    assert native.CCU_RENDER_SPECULAR == 4
    java = open(os.path.join(ROOT, "java", "dev", "thatredox", "chunkynative", "cuda", "ChunkyCu.java")).read()
    assert re.search(r"RENDER_SPECULAR = 4\b", java)


def test_pack_material_word_5():
    """Defaults reproduce the words the packer wrote before (specular byte only); the three bytes of
    PackedMaterial.java:69-71 otherwise."""
    assert S.pack_material(16, 3, emittance=0.5, specular=0.3) == [4, 0, 16, 3, 127, 76]
    assert S.pack_material(0, 0, textured=False, argb=S._s32(0xFF102030)) == [0, 0, -1, S._s32(0xFF102030), 0, 0]
    assert S.pack_material(1, 2, specular=0.2, metalness=0.6, roughness=1.0)[5] == 51 | (153 << 8) | (255 << 16)


def test_glossy_scenes_cover_every_kind_of_material(scenes):
    g = S.glossy(scenes("mixed"))
    words = g.mat_palette[5::6]
    kinds = {(w & 0xFF > 0, (w >> 8) & 0xFF > 0, (w >> 16) & 0xFF > 0) for w in words.tolist()}
    assert {(True, False, False), (False, True, False), (True, False, True), (False, False, False)} <= kinds
    emissive = (g.mat_palette[4::6] & 0xFF) > 0
    assert emissive.any() and (words[emissive] == S.specular_word(0.5)).all()
    assert np.array_equal(np.delete(g.mat_palette, np.s_[5::6]), np.delete(scenes("mixed").mat_palette, np.s_[5::6]))
