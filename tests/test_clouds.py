"""CCU_RENDER_CLOUDS on the CPU (DESIGN.md §15): the restatement's cloud walk (specular_oracle.cloud_hit) against a brute force
over every box, the flag-off identities, a closed form under full cover, the shadow share under a striped layer, and the loader
of Chunky's cloud keys."""
import dataclasses
import json
import math
import os

import numpy as np
import pytest

from chunkyclplugin_b200 import octree2
from chunkyclplugin_b200 import scenes as S
from chunkyclplugin_b200.javarandom import pass_seeds
from oracle import edge_rays as E
from test_gpu_variants import SEEDS, variant_scene

import specular_oracle as SO

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CLOUDS = SO.CCU_RENDER_CLOUDS
CELLS = 1024           # §15.2: cells the walk visits at most
F = np.float32


# ---------------------------------------------------------------------------------------------------------
# the walk against a brute force over every box
# ---------------------------------------------------------------------------------------------------------
def _axis(o, d, c):
    """The ray's parameter interval in cell c of one cell axis (all float32, as §15.2 writes it)."""
    if d == 0:
        inside = (c < o) & (o < c + 1)
        return np.where(inside, -np.inf, np.nan).astype(F), np.where(inside, np.inf, np.nan).astype(F)
    a = (c.astype(F) - o) / d
    b = ((c + 1).astype(F) - o) / d
    return (a, b) if d > 0 else (b, a)


def brute(clouds, o, d, limit):
    """The nearest entry t > 0 below `limit` into the box of any set cell the segment's xz bounding box covers, and its normal
    (ties between axes: y, x, z); (nan, 0) for none."""
    mask, size, y0, y1, u0, v0 = clouds
    inv = F(1) / F(size)
    o, d = o.astype(F), d.astype(F)
    if d[1] == 0:
        if not (F(y0) < o[1] < F(y1)):
            return math.nan, np.zeros(3, F)
        ylo, yhi = F(-np.inf), F(np.inf)
    else:
        a, b = (F(y0) - o[1]) / d[1], (F(y1) - o[1]) / d[1]
        ylo, yhi = (a, b) if d[1] > 0 else (b, a)
    t0, t1 = max(float(ylo), 0.0), min(float(yhi), float(limit))
    if not t0 < t1:
        return math.nan, np.zeros(3, F)
    ox, dx = o[0] * inv + F(u0), d[0] * inv
    oz, dz = o[2] * inv + F(v0), d[2] * inv
    xs = [float(ox) + float(dx) * t for t in (t0, t1)]
    zs = [float(oz) + float(dz) * t for t in (t0, t1)]
    i = np.arange(math.floor(min(xs)) - 1, math.floor(max(xs)) + 2)
    k = np.arange(math.floor(min(zs)) - 1, math.floor(max(zs)) + 2)
    ii, kk = np.meshgrid(i, k, indexing="ij")
    ii, kk = ii.reshape(-1), kk.reshape(-1)
    set_ = mask[kk & 255, ii & 255] != 0
    ii, kk = ii[set_], kk[set_]
    if ii.size == 0:
        return math.nan, np.zeros(3, F)
    xlo, xhi = _axis(ox, dx, ii)
    zlo, zhi = _axis(oz, dz, kk)
    with np.errstate(invalid="ignore"):
        tn = np.full(ii.size, ylo, F)
        axis = np.ones(ii.size, int)
        sel = xlo > tn
        tn[sel], axis[sel] = xlo[sel], 0
        sel = zlo > tn
        tn[sel], axis[sel] = zlo[sel], 2
        tf = np.minimum(np.minimum(np.full(ii.size, yhi, F), xhi), zhi)
        ok = (tn > 0) & (tn < tf) & (tn < F(limit)) & ~np.isnan(xlo) & ~np.isnan(zlo)
    if not ok.any():
        return math.nan, np.zeros(3, F)
    j = int(np.flatnonzero(ok)[np.argmin(tn[ok])])
    n = np.zeros(3, F)
    n[axis[j]] = -1.0 if (dx, d[1], dz)[axis[j]] > 0 else 1.0
    return float(tn[j]), n


def _check(clouds, o, d, limit):
    t, n, visited = SO.cloud_hit(clouds, o, d, limit)
    assert (visited < CELLS).all(), "the cap must not act on these rays"
    hits = 0
    for r in range(o.shape[0]):
        bt, bn = brute(clouds, o[r], d[r], limit[r])
        if math.isnan(bt):
            assert math.isnan(t[r]), (r, o[r], d[r], limit[r], t[r])
            continue
        hits += 1
        assert F(t[r]).view(np.uint32) == F(bt).view(np.uint32), (r, o[r], d[r], limit[r], t[r], bt)
        assert np.array_equal(n[r], bn), (r, n[r], bn)
    return hits


@pytest.mark.parametrize("size,u0,v0", [(1.0, 0.0, 0.0), (3.7, 0.25, -0.6), (12.0, -3.5, 17.2), (0.61, 1e-3, -250.9)])
def test_walk_matches_brute_force(size, u0, v0):
    rng = np.random.default_rng(int(size * 100))
    mask = S.cloud_mask(seed=int(size * 10), cover=0.4)
    y0, y1 = 20.0, 24.5
    clouds = (mask, size, y0, y1, u0, v0)
    n = 3000
    o = np.stack([rng.uniform(-700, 700, n), rng.uniform(5, 40, n), rng.uniform(-700, 700, n)], 1)
    d = rng.normal(size=(n, 3)) * rng.uniform(0.3, 3.0, (n, 1))
    # axis-aligned directions, and rays that run parallel to the slab inside it
    d[:300] = np.eye(3)[rng.integers(0, 3, 300)] * rng.choice([-1.0, 1.0], (300, 1)) * rng.uniform(0.5, 2, (300, 1))
    d[300:700, 1] = 0.0
    o[300:700, 1] = rng.uniform(y0, y1, 400)
    o[300:350, 1] = y0                                  # in the bottom face's plane: never enters a box
    o[350:400, 1] = y1
    limit = rng.uniform(1, 40, n) / np.linalg.norm(d, axis=1)
    o, d, limit = o.astype(F), d.astype(F), limit.astype(F)
    hits = _check(clouds, o, d, limit)
    assert hits > 400


def test_walk_on_faces_and_inside_boxes():
    """Origins on the faces of set boxes (going in or out) and inside them, at integral cell coordinates (size 1, no offset)."""
    rng = np.random.default_rng(7)
    mask = S.cloud_mask(seed=2, cover=0.5)
    clouds = (mask, 1.0, 10.0, 12.0, 0.0, 0.0)
    n = 2000
    ij = rng.integers(-300, 300, (n, 2))
    o = np.stack([ij[:, 0] + rng.uniform(0, 1, n), rng.uniform(10, 12, n), ij[:, 1] + rng.uniform(0, 1, n)], 1)
    face = rng.integers(0, 4, n)                        # 0: x face, 1: z face, 2: bottom face, 3: inside
    o[face == 0, 0] = np.round(o[face == 0, 0])
    o[face == 1, 2] = np.round(o[face == 1, 2])
    o[face == 2, 1] = 10.0
    d = rng.normal(size=(n, 3))
    d[::5, 1] = 0.0
    limit = np.full(n, 30.0)
    o, d, limit = o.astype(F), d.astype(F), limit.astype(F)
    t, _, _ = SO.cloud_hit(clouds, o, d, limit)
    inside = (face == 3) & (mask[np.floor(o[:, 2]).astype(int) & 255, np.floor(o[:, 0]).astype(int) & 255] != 0)
    assert inside.sum() > 100
    assert (np.isnan(t) | (t > 0)).all()
    assert _check(clouds, o, d, limit) > 300


def test_unbounded_rays_and_bad_inputs():
    mask = np.ones((256, 256), np.uint8)
    clouds = (mask, 2.0, 30.0, 34.0, 0.5, 0.5)
    o = np.array([[5.3, 10.0, 5.3], [5.3, 40.0, 5.3], [5.3, 10.0, 5.3], [np.nan, 10.0, 5.3], [5.3, 10.0, 5.3], [5.3, 32.0, 5.3],
                  [5.3, 10.0, 5.3], [5.3, 36.0, 5.3]], F)
    d = np.array([[0.0, 2.0, 0.0], [0.0, -1.0, 0.0], [0.0, -1.0, 0.0], [0.0, 1.0, 0.0], [np.inf, 1.0, 0.0], [1.0, 0.0, 0.0],
                  [0.0, 0.0, 0.0], [0.0, 1.0, 0.0]], F)
    t, n, _ = SO.cloud_hit(clouds, o, d)
    assert t[0] == F(10.0) and np.array_equal(n[0], [0, -1, 0])     # camera-style unnormalised ray: t in its own units
    assert t[1] == F(6.0) and np.array_equal(n[1], [0, 1, 0])
    # inside a box the ray leaves it without a hit and hits the next set box it enters: cell x 3.15 -> 4 at t = 1.7
    assert F(t[5]) == (F(4.0) - (F(5.3) * F(0.5) + F(0.5))) / F(0.5) and np.array_equal(n[5], [-1, 0, 0])
    assert np.isnan(t[[2, 3, 4, 6, 7]]).all()                        # away, NaN, infinite, zero, above


def test_the_cell_cap():
    """A ray inside the slab crosses row k = 1 (empty) at a shallow angle into row k = 0 (set): the walk reports the hit while
    it reaches row 0 within 1024 cells, and a miss after; the brute force finds it in both cases."""
    mask = np.zeros((256, 256), np.uint8)
    mask[0, :] = 1
    clouds = (mask, 1.0, 0.0, 4.0, 0.0, 0.0)
    for cells, hit in ((1000, True), (1100, False)):
        o = np.array([[0.5, 2.0, 1.5]], F)
        d = np.array([[1.0, 0.0, -0.5 / (cells + 0.25)]], F)
        t, _, visited = SO.cloud_hit(clouds, o, d, np.array([2000.0], F))
        bt, _ = brute(clouds, o[0], d[0], 2000.0)
        assert not math.isnan(bt)
        if hit:
            assert F(t[0]) == F(bt) and visited[0] <= CELLS
        else:
            assert np.isnan(t[0]) and visited[0] == CELLS


# ---------------------------------------------------------------------------------------------------------
# rendering
# ---------------------------------------------------------------------------------------------------------
def fixture_clouds(p):
    """The cloud layer the GPU tests put on the variant fixture: half the cells, over the terrain, under the sun."""
    return S.with_clouds(p, S.cloud_mask(seed=3, cover=0.5), size=4.0, y0=40.0, y1=44.0, u0=0.25, v0=-0.5)


def test_flag_off_identities():
    """§15.5 on the variant fixture: the flag without clouds, clouds without the flag and the flag with an all-zero mask render
    the flag-off bits; the flag with clouds changes most pixels, and with the sun off and one segment shows the cells."""
    p = variant_scene(True)
    off = SO.FlagsOracle(p, 0).render(SEEDS)
    assert np.array_equal(SO.FlagsOracle(p, CLOUDS).render(SEEDS).view(np.uint32), off.view(np.uint32))
    q = fixture_clouds(p)
    assert np.array_equal(SO.FlagsOracle(q, 0).render(SEEDS).view(np.uint32), off.view(np.uint32))
    empty = dataclasses.replace(q, clouds=(np.zeros((256, 256), np.uint8),) + q.clouds[1:])
    assert np.array_equal(SO.FlagsOracle(empty, CLOUDS).render(SEEDS).view(np.uint32), off.view(np.uint32))
    on = SO.FlagsOracle(q, CLOUDS).render(SEEDS)
    assert np.mean(~E.same_bits_or_nan(on, off).reshape(-1, 3).all(1)) > 0.5
    dark = E.without_sun(q)
    seen = SO.FlagsOracle(dark, CLOUDS, max_depth=1).render(SEEDS).reshape(-1, 3)
    sky = SO.FlagsOracle(dark, 0, max_depth=1).render(SEEDS).reshape(-1, 3)
    assert np.mean((seen == 0).all(1) & (sky > 0).any(1)) > 0.02      # camera rays that hit a cloud (white, no emission)


def _floor_scene(o, d, altitude, azimuth):
    """A white stone floor (top face y = 1) in a 64^3 world, a black sky and a flat sun at (altitude, azimuth); rays o + t d."""
    vox = np.zeros((64, 64, 64), np.int32)
    vox[:, 0, :] = S.STONE
    rays = np.concatenate([o, d], 1).astype(F).reshape(-1)
    pal = S.Palettes()
    tree, depth = S.build_octree(vox, pal.block_mapping)
    p = S._finish("floor", tree, depth, pal, rays, o.shape[0], 1)
    p.atlas[...] = 255
    sky = np.zeros((16, 16, 4), np.uint8)
    sky[..., 3] = 255
    return dataclasses.replace(p, projector_type=-1, sky=sky, sun=S.pack_sun(*pal.sun_tex, altitude=altitude, azimuth=azimuth))


def test_full_cover_is_black():
    """An all-ones mask above the world, a black sky, the sun on, no emitters, the camera below the layer: the sun sample of
    every camera-ray hit, on the floor or on a cloud's underside, is blocked, so the image is exactly 0 (and not without the
    clouds).  One segment, and rays at least 15 degrees off the horizon: a hit thousands of blocks away (a grazing bounce) is
    placed on the face itself, where the offset of §15.3 is below an ulp, and its sun sample then leaves the box unblocked."""
    rng = np.random.default_rng(3)
    n = 1024
    d = rng.normal(size=(n, 3))
    d = d[np.abs(d[:, 1]) > 0.27 * np.linalg.norm(d, axis=1)]
    o = np.broadcast_to(np.array([32.0, 60.0, 32.0]), d.shape)
    p = _floor_scene(o, d, 1.1, 0.7)
    q = S.with_clouds(p, np.ones((256, 256), np.uint8), size=3.0, y0=70.0, y1=74.0)
    seeds = pass_seeds(4)
    assert (SO.FlagsOracle(p, CLOUDS, max_depth=1).render(seeds).reshape(-1, 3) > 0).any(1).mean() > 0.05
    assert not SO.FlagsOracle(q, CLOUDS, max_depth=1).render(seeds).any()


def test_striped_layer_shadows_half_the_floor():
    """Stripes of cells along z (every second column set) above a white floor, the sun tilted along z only: the direct sunlight
    on uniformly spread floor points converges to the unshadowed share 1/2 of the cloud-free value, within 5 standard errors."""
    alt, az = 1.0, math.pi / 2                          # the sun direction has no x component
    rng = np.random.default_rng(11)
    n = 4096
    o = np.stack([rng.uniform(4, 60, n), np.full(n, 6.0), rng.uniform(4, 60, n)], 1)
    d = np.stack([np.zeros(n), -np.ones(n), np.zeros(n)], 1)
    p = _floor_scene(o, d, alt, az)
    mask = np.zeros((256, 256), np.uint8)
    mask[:, 0::2] = 1
    q = S.with_clouds(p, mask, size=2.0, y0=80.0, y1=90.0, u0=0.3)
    seeds = pass_seeds(1)
    free = SO.FlagsOracle(p, CLOUDS, max_depth=1).render(seeds).reshape(-1, 3)[:, 0].astype(np.float64)
    lit = SO.FlagsOracle(q, CLOUDS, max_depth=1).render(seeds).reshape(-1, 3)[:, 0].astype(np.float64)
    assert (free > 0).all()
    share = lit / free
    bound = 5 * float(np.std(share)) / math.sqrt(n)
    assert abs(float(np.mean(share)) - 0.5) < bound, (float(np.mean(share)), bound)
    assert 0.01 < bound < 0.05


# ---------------------------------------------------------------------------------------------------------
# loader
# ---------------------------------------------------------------------------------------------------------
def test_clouds_from_json_on_the_benchmark_keys(tmp_path):
    """The benchmark scene's sky keys (clouds off), and the same keys with clouds on: the layer in the plugin's frame."""
    path = os.path.join(ROOT, "tests", "golden", "opencl_test_clouds.json")
    mask = S.cloud_mask(seed=1)
    assert octree2.clouds_from_json(path, mask) is None
    d = json.load(open(path))
    d["sky"]["cloudsEnabled"] = True
    d["sky"]["cloudOffset"] = {"x": 10.0, "y": 128.0, "z": -6.0}
    on = tmp_path / "clouds.json"
    on.write_text(json.dumps(d))
    m, size, y0, y1, u0, v0 = octree2.clouds_from_json(str(on), mask)
    assert np.array_equal(m, mask) and size == 64.0
    assert y0 == 128.0 and y1 == 128.0 + octree2.CLOUD_THICKNESS
    # the frame's origin is the chunk rectangle's low corner: chunk (-41, -26) -> (-656, -416)
    assert u0 == (-656 + octree2.CLOUD_OFFSET_SIGN * 10.0) / 64.0 and v0 == (-416 + octree2.CLOUD_OFFSET_SIGN * -6.0) / 64.0
    with pytest.raises(ValueError):
        octree2.clouds_from_json(str(on), np.zeros((16, 16), np.uint8))
