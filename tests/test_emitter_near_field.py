"""CCU_RENDER_EMITTER_NEAR_FIELD on the CPU (DESIGN.md §11): the CPU restatement of the estimator (specular_oracle.FlagsOracle)
with flags 8 | 128 against bit 8 alone where no sample is near, against the bound of §11 item 6 and a closed-form form factor
where a floor meets an emitter cube, and against the flag-off render in expectation.  Seeds are fixed, so every statistical
check is deterministic."""
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
from test_emitter_sampling import (CUBE, EMIT_ARGB, EMIT_BYTE, FLOOR_ARGB, GRID_SCENES, H, P, SCALE, W, _argb, _passes, _regions,
                                   analytic_scene, form_factor)

import specular_oracle as SO

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
NEE, NEAR = 8, 128
RHO = 0.125                                      # DESIGN §11
BOUND_FACTOR = max(1.0, 3.0 / (math.pi * RHO * RHO))


def test_far_floor_renders_as_bit_8():
    """On §10's analytic floor the hit point lies 1 from the cube's box, so no sample is near."""
    p = analytic_scene(1024)
    seeds = pass_seeds(4)
    kw = dict(max_depth=2, emitter_scale=SCALE)
    assert np.array_equal(SO.FlagsOracle(p, flags=NEE | NEAR, **kw).render(seeds), SO.FlagsOracle(p, flags=NEE, **kw).render(seeds))


# ---------------------------------------------------------------------------------------------------------
# contact: a flat emitter cube standing on a flat floor, rays onto floor points next to its side faces
# ---------------------------------------------------------------------------------------------------------
GAPS = (1e-3, 3e-3, 1e-2, 3e-2, 0.1, 0.2, 0.4, 0.8)    # distance of the floor point to the cube's side face
REPS = 64                                              # pixels per floor point


def contact_points():
    """Floor points (x, z) at each gap from each of the four side faces, at two positions along the face."""
    cx, cz = CUBE[0], CUBE[2]
    pts = []
    for g in GAPS:
        for a in (0.3, 0.7):
            pts += [(cx - g, cz + a), (cx + 1 + g, cz + a), (cx + a, cz - g), (cx + a, cz + 1 + g)]
    return np.array(pts, np.float64)


def contact_scene():
    """CUBE on a floor whose top is y = CUBE[1]; one pre-generated downward ray per pixel, REPS pixels per floor point, black
    sky and the sun off: with max_depth 2 each 1-pass pixel is exactly the one emitter sample of its floor hit."""
    pal = S.Palettes()
    floor = pal.put_material(S.pack_material(0, 0, textured=False, argb=FLOOR_ARGB))
    lamp = pal.put_material(S.pack_material(0, 0, textured=False, argb=EMIT_ARGB, emittance=EMIT_BYTE / 255.0))
    b_floor = len(pal.blocks)
    pal.blocks += [1, floor]
    b_lamp = len(pal.blocks)
    pal.blocks += [1, lamp]
    vox = np.zeros((16, 16, 16), np.int64)
    vox[:, :CUBE[1], :] = 1
    vox[CUBE] = 2
    tree, depth = S.build_octree(vox.astype(np.int32), np.array([0, b_floor, b_lamp], np.int64))
    pts = contact_points()
    n = pts.shape[0] * REPS
    p = S._finish("contact", tree, depth, pal, S.pinhole_camera((6, 6, 6), 0, -90), n, 1, sun_draw=False)
    rays = np.zeros((pts.shape[0], REPS, 6), np.float32)
    rays[:, :, 0], rays[:, :, 1], rays[:, :, 2] = pts[:, None, 0], CUBE[1] + 2.0, pts[:, None, 1]
    rays[:, :, 4] = -1.0
    p = dataclasses.replace(p, projector_type=-1, camera=rays.reshape(-1), sky_intensity=0.0, sky=np.zeros_like(p.sky))
    return E.without_sun(p)


def _contact(flags, passes):
    p = contact_scene()
    o = SO.FlagsOracle(p, flags=flags, max_depth=2, emitter_scale=SCALE)
    return o.render(pass_seeds(passes)).reshape(-1, REPS, 3).astype(np.float64)


def _bound():
    """§11 item 6 for the floor's hits: T = the floor colour, N = 1 emitter in the list"""
    return _argb(FLOOR_ARGB) * _argb(EMIT_ARGB) ** 2 * (EMIT_BYTE / 255.0) * SCALE * BOUND_FACTOR


def test_contact_contributions_are_bounded():
    """Every 1-pass pixel is one emitter sample, and none exceeds the bound; with bit 8 alone the area sampler's 1/d2 weight
    exceeds it next to the faces (measured: largest pixel 1.6 times the bound, against 0.04 with the near field)."""
    bound = _bound() * (1 + 1e-5)
    near = _contact(NEE | NEAR, 1)
    assert np.all(near <= bound), (near.max(axis=(0, 1)), bound)
    assert near.max() > 0
    area = _contact(NEE, 1)
    assert np.any(area > bound), (area.max(axis=(0, 1)), bound)


def test_contact_matches_the_form_factor():
    """256 passes: the mean of each floor point's REPS pixels against the closed-form form factor within 4 standard errors
    (the pixels of a point are independent means of 256 samples)."""
    px = _contact(NEE | NEAR, 256)
    base = _argb(FLOOR_ARGB) * _argb(EMIT_ARGB) ** 2 * (EMIT_BYTE / 255.0) * SCALE
    for i, (x, z) in enumerate(contact_points()):
        want = base * form_factor(np.array([x, CUBE[1], z]), np.array([0.0, 1.0, 0.0]))
        se = px[i].std(0, ddof=1) / math.sqrt(REPS)
        assert np.all(np.abs(px[i].mean(0) - want) < 4 * se + 1e-3 * want), (x, z, px[i].mean(0), want, se)


# ---------------------------------------------------------------------------------------------------------
# indoor64: unbiased against the flag-off render, and the error at equal spp against bit 8
# ---------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def indoor_passes():
    p = S.indoor_scene(64, W, H)
    seeds = pass_seeds(2 * P + 2048)
    return (_passes(p, NEE | NEAR, seeds[:P]), _passes(p, NEE, seeds[:P]), _passes(p, 0, seeds[P:2 * P]),
            _passes(p, 0, seeds[2 * P:]).mean(0))


def test_unbiased_against_flag_off(indoor_passes):
    """Region means over 512 passes each, disjoint seed streams; the tolerance is the standard error measured from the
    passes."""
    near, _, off, _ = indoor_passes
    rn, ro = _regions(near), _regions(off)
    z = (rn.mean(0) - ro.mean(0)) / np.sqrt(rn.var(0, ddof=1) / P + ro.var(0, ddof=1) / P)
    assert np.abs(z).max() < 4.5, z


@pytest.mark.parametrize("spp", [4, 16, 64])
def test_error_against_bit_8(indoor_passes, spp):
    """RMSE against a 2048-pass flag-off render at equal spp, averaged over the disjoint windows of the 512 passes, with the
    same seeds for both samplers.  Indoor64 has few hits near an emitter face, so the near field does not lower the error
    here: measured ratio near / bit 8 1.009 at 4, 16 and 64 spp.  The check holds it within 3 % of bit 8."""
    near, area, _, ref = indoor_passes

    def rmse(a):
        return np.mean([np.sqrt(((a[i:i + spp].mean(0) - ref) ** 2).mean()) for i in range(0, P, spp)])

    r_near, r_area = rmse(near), rmse(area)
    assert r_near < 1.03 * r_area, (r_near, r_area)


def test_no_emitters_renders_as_flag_off():
    p = GRID_SCENES["none"]()
    seeds = pass_seeds(2)
    assert np.array_equal(SO.FlagsOracle(p, flags=NEE | NEAR).render(seeds), SO.FlagsOracle(p, flags=0).render(seeds))


def test_set_params_needs_emitter_sampling():
    """128 alone is refused, naming the flag it needs; 8 | 128 is valid and gets as far as the missing context."""
    import ctypes as C
    lib = native.load()
    for flags, msg in ((NEAR, "CCU_RENDER_EMITTER_NEAR_FIELD needs CCU_RENDER_EMITTER_SAMPLING"),
                       (NEAR | 4 | 2 | 1, "needs CCU_RENDER_EMITTER_SAMPLING"), (NEE | NEAR, "null"), (NEE | NEAR | 4 | 2 | 1, "null")):
        p = native.RenderParams(256, 5, 13.0, 0, flags)
        assert lib.ccu_render_set_params(None, C.byref(p)) == native.CCU_EINVAL
        assert msg in lib.ccu_last_error().decode(), (flags, lib.ccu_last_error())


def test_flag_constant_agrees():
    hdr = open(os.path.join(ROOT, "include", "chunkycu.h")).read()
    java = open(os.path.join(ROOT, "java", "dev", "thatredox", "chunkynative", "cuda", "ChunkyCu.java")).read()
    assert int(re.search(r"#define CCU_RENDER_EMITTER_NEAR_FIELD (\d+)", hdr).group(1)) == NEAR
    assert int(re.search(r"RENDER_EMITTER_NEAR_FIELD = (\d+)", java).group(1)) == NEAR
    assert native.CCU_RENDER_EMITTER_NEAR_FIELD == NEAR == SO.CCU_RENDER_EMITTER_NEAR_FIELD
