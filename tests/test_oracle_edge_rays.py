"""The ray catalogue of oracle/edge_rays.py (CPU only): what each class contains, the oracle against the reference's own
kernel on every catalogue scene (tests/golden/clref_edge_rays.npz, written on a B200 by scripts/edge_rays_golden.py
from the strict build), and the oracle against an independent geometric answer for axis-aligned rays."""
import os

import numpy as np
import pytest

import oracle
from chunkyclplugin_b200.javarandom import pass_seeds
from oracle import edge_rays as E

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "clref_edge_rays.npz")
EDGE = [f"edge_{n}" for n in E.BASES]
SUN = [f"sun_{b}_{v}" for b in E.SUN_BASES for v in E.sun_variants()]


@pytest.fixture(scope="module")
def catalogue():
    return E.scenes()


@pytest.fixture(scope="module")
def golden():
    return np.load(GOLDEN)


@pytest.fixture(scope="module")
def oracle_out(catalogue):
    """name -> oracle outputs, computed once"""
    cache = {}

    def get(name):
        if name not in cache:
            p = catalogue[name]
            o = oracle.Oracle(p)
            r = dict(rad_sun=o.render(pass_seeds(E_PASSES)))
            if name.startswith("edge_"):
                r.update(fh=o.first_hit(pass_seeds(1)[0]), pv=o.preview(),
                         rad_nosun=oracle.Oracle(E.without_sun(p)).render(pass_seeds(E_PASSES)))
            cache[name] = r
        return cache[name]
    return get


E_PASSES = 4


def _neg_zero(a):
    return (a == 0) & np.signbit(a)


def _one_ulp_off_integer(a):
    """coordinates that are 1 ulp above or below an integer (not themselves integers)"""
    a = np.asarray(a, np.float32)
    r = np.round(a).astype(np.float32)
    return (a != r) & ((np.nextafter(r, np.float32(np.inf)) == a) | (np.nextafter(r, np.float32(-np.inf)) == a))


def _outside(o, depth):
    """octree.h:52: the origin's voxel, as f2i (saturating, NaN -> 0) computes it, lies outside the cube"""
    with np.errstate(invalid="ignore"):
        f = np.floor(o.astype(np.float64))
        v = np.where(np.isnan(f), 0, np.clip(f, -2.0 ** 31, 2.0 ** 31 - 1)).astype(np.int64)
    return ((v >> depth) != 0).any(axis=1)


# ---------------------------------------------------------------------------------------------------------
# the catalogue holds what it claims
# ---------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", EDGE)
def test_catalogue_classes(catalogue, name):
    p = catalogue[name]
    depth, n = p.octree_depth, 1 << p.octree_depth
    planes = [float(1 << l) for l in range(1, depth)]
    assert p.projector_type == -1 and p.width == E.WIDTH and p.camera.size == 6 * p.width * p.height

    _, a = E.class_rays(p, "A")
    o, d = a[:, :3], a[:, 3:]
    assert ((np.abs(d) == 1).sum(axis=1) == 1).all() and ((d == 0).sum(axis=1) == 2).all()
    assert _neg_zero(d).sum() > 100 and ((d == 0) & ~np.signbit(d)).sum() > 100
    perp = o[d == 0]
    assert np.isin(perp, planes).sum() > 20                            # on the leaf-cube planes 2^l
    assert np.isin(perp, [0.0, 1.0, n - 1.0]).sum() > 20
    assert ((perp % 1) == 0.5).sum() > 20
    assert _one_ulp_off_integer(perp).sum() > 20
    along = o[np.abs(d) == 1]
    assert (along == n).sum() > 10 and (along == 0).sum() > 10        # on the cube's planes 0 and 2^depth

    _, b = E.class_rays(p, "B")
    o, d = b[:, :3], b[:, 3:]
    assert ((d == 0).sum(axis=1) == 1).sum() > 40
    assert ((np.abs(d) == 1).all(axis=1)).sum() > 20                   # (1,1,1) diagonals
    assert ((o % 1 == 0).sum(axis=1) >= 2).sum() > 40                 # on voxel edges and corners
    assert _one_ulp_off_integer(o).any(axis=1).sum() > 20

    _, c = E.class_rays(p, "C")
    o, d = c[:, :3], c[:, 3:]
    assert _outside(o, depth).all()
    on_plane = ((o == 0) | (o == n)) & (d == 0)                      # grazing: in a face's plane, parallel to it
    assert on_plane.any(axis=1).sum() >= 18
    assert (_one_ulp_off_integer(o) & (d == 0)).any(axis=1).sum() >= 24
    assert (np.abs(o) == np.float32(3e9)).any() and (o == np.float32(1e4)).any()
    regions = {tuple(np.sign(np.floor(v) // n).astype(int)) for v in o[(np.abs(o) < 4 * n).all(axis=1)]}
    assert len(regions) == 26                                          # 6 faces, 12 edges, 8 corners

    _, dd = E.class_rays(p, "D")
    o = dd[:, :3]
    inside = ~_outside(o, depth)
    vox = E.leaf_values(p, np.floor(o[inside]).astype(np.int64))
    below = np.floor(o[inside]).astype(np.int64) - [0, 1, 0]
    ok = (below >= 0).all(axis=1)
    on_top = np.zeros(inside.sum(), bool)
    on_top[ok] = (E.leaf_values(p, below[ok]) != 0) & (o[inside][ok, 1] % 1 == 0)
    assert (vox != 0).sum() >= 8 and on_top.sum() >= 8                  # in solid blocks, on a block's top face
    assert (o == 0).all(axis=1).any() and (o == np.nextafter(np.float32(n), np.float32(0))).all(axis=1).any()

    _, e = E.class_rays(p, "E")
    o, d = e[:, :3], e[:, 3:]
    assert (d == 0).all(axis=1).any()
    assert ((np.abs(d) > 0) & (np.abs(d) < np.finfo(np.float32).tiny)).any()
    assert (np.abs(d) == np.float32(1e30)).any()
    for k in (1, 2, 3):
        assert (np.isinf(d).sum(axis=1) == k).any(), k
        assert (np.isnan(d).sum(axis=1) == k).any(), k
    assert np.isnan(o).any(axis=1).sum() >= 8
    length = np.linalg.norm(d.astype(np.float64), axis=1)
    assert np.isclose(length, 1e-3).any() and np.isclose(length, 1e3).any()

    if "F" in p.meta["rows"]:
        _, f = E.class_rays(p, "F")
        o, d = f[:, :3], f[:, 3:]
        tf = p.bvh_trigs.view(np.float32)
        verts = {tuple(tf[i:i + 3]) for i in range(0, tf.size - 2)}
        moved = [tuple(np.where(d[i] != 0, np.nan, o[i])) for i in range(o.shape[0])]
        on_vertex = sum(any(all(np.isnan(m[k]) or m[k] == v[k] for k in range(3)) for v in verts) for m in moved[:60])
        assert on_vertex >= 20                                         # aimed exactly at packed triangle coordinates
        boxes = np.concatenate([p.world_bvh.reshape(-1, 7)[:, 1:], p.actor_bvh.reshape(-1, 7)[:, 1:]]).view(np.float32)
        assert np.isin(o, boxes).any(axis=1).sum() >= 16              # on a BVH node box's plane


def test_switch_azimuths_select_different_sun_bases():
    """Sun_new takes su = (0,1,0) for |sw.x| > 0.1 and (1,0,0) otherwise (sky.h:31); the two catalogue azimuths are
    adjacent float32 values on either side of that switch, in the oracle (whose cos is the device's)."""
    a, b = E.switch_azimuths()
    assert np.nextafter(np.float32(a), np.float32(np.inf)) == np.float32(b)
    basis = {v: oracle.Oracle(E.sun_scene("terrain64", v)).sun_basis() for v in ("az_switch_above", "az_switch_below")}
    sw_a, sw_b = basis["az_switch_above"][0], basis["az_switch_below"][0]
    assert abs(sw_a[0]) > np.float32(0.1) >= abs(sw_b[0])
    # su = cross(sv, sw) with sv = normalize(cross(sw, su0)): su0 = (0,1,0) leaves sv.y = 0, su0 = (1,0,0) leaves sv.x = 0
    assert basis["az_switch_above"][2][1] == 0 and basis["az_switch_below"][2][0] == 0
    assert not np.array_equal(basis["az_switch_above"][1], basis["az_switch_below"][1])
    sw_pi = oracle.Oracle(E.sun_scene("terrain64", "az_pi")).sun_basis()
    assert sw_pi[0][0] < -0.9 and sw_pi[2][1] == 0                    # sw.x < -0.1: the fabs decides


# ---------------------------------------------------------------------------------------------------------
# an answer that depends on neither implementation
# ---------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("base", E.FULL_CUBE_SCENES)
def test_axis_rays_hit_the_first_solid_voxel(catalogue, oracle_out, base):
    name = f"edge_{base}"
    checked = check_axis_hits(catalogue[name], oracle_out(name)["fh"])
    assert checked["hit"] >= 10 and checked["miss"] >= 10, checked


def check_axis_hits(p, fh):
    """Asserts the first-hit buffers `fh` of catalogue scene `p` against E.axis_hits; returns the counts checked."""
    counts = {"hit": 0, "miss": 0}
    for gid, want in E.axis_hits(p):
        if want is None:
            assert fh["kind"][gid] == 0, gid
            counts["miss"] += 1
            continue
        t, normal = want
        assert fh["kind"][gid] == 1, (gid, p.camera.reshape(-1, 6)[gid])
        assert abs(float(fh["t"][gid]) - t) <= 1e-3, (gid, fh["t"][gid], t)
        assert np.array_equal(fh["normal"].reshape(-1, 3)[gid], normal), gid
        counts["hit"] += 1
    return counts


# ---------------------------------------------------------------------------------------------------------
# the oracle against the reference kernel
# ---------------------------------------------------------------------------------------------------------
def assert_first_hit_matches_golden(g, name, fh):
    """fh (oracle or CUDA first-hit buffers) against the reference's probe_first_hit buffers of scene `name`."""
    hit = fh["kind"] > 0
    assert np.array_equal(g[f"{name}__hit"].astype(bool), hit)
    assert np.array_equal(g[f"{name}__block"][hit], fh["block"][hit])
    for k in ("t", "normal", "color"):
        assert E.same_bits_or_nan(g[f"{name}__{k}"], fh[k]).all(), k


def test_golden_is_the_current_catalogue(catalogue, golden):
    assert int(golden["seed"]) == pass_seeds(1)[0] and int(golden["passes"]) == E_PASSES
    assert "B200" in str(golden["device"])
    for name, p in catalogue.items():
        n = p.width * p.height
        assert golden[f"{name}__rad_sun"].size == 3 * n, name
        if name.startswith("edge_"):
            assert golden[f"{name}__hit"].size == n, name
    assert os.path.getsize(GOLDEN) < 1 << 20


@pytest.mark.parametrize("name", EDGE)
def test_first_hit_matches_reference(golden, oracle_out, name):
    assert_first_hit_matches_golden(golden, name, oracle_out(name)["fh"])


@pytest.mark.parametrize("name", EDGE)
def test_preview_matches_reference(catalogue, golden, oracle_out, name):
    """Exact where the primary ray hits; the sky goes through the texture unit's 8-bit filter weights in the reference,
    so sky pixels may differ by 1 in a channel (as in test_oracle_golden)."""
    a, b = golden[f"{name}__preview"].view(np.uint32), oracle_out(name)["pv"].view(np.uint32)
    hit = oracle_out(name)["fh"]["kind"] > 0
    assert np.array_equal(a[hit], b[hit])
    sh = np.array([24, 16, 8, 0], dtype=np.uint32)
    d = np.abs(((a[:, None] >> sh) & 255).astype(np.int32) - ((b[:, None] >> sh) & 255).astype(np.int32))
    known = ~hit & E.sky_lookup_differs(catalogue[name].camera)
    assert d[~known].max() <= 1
    assert known.sum() >= 4 and (d[known].max(axis=1) > 1).any()        # the open differences are still there


@pytest.mark.parametrize("sun", ["sun", "nosun"])
@pytest.mark.parametrize("name", EDGE)
def test_radiance_matches_reference(catalogue, golden, oracle_out, name, sun):
    miss = oracle_out(name)["fh"]["kind"] == 0
    known = miss & E.sky_lookup_differs(catalogue[name].camera)
    check_radiance(golden[f"{name}__rad_{sun}"], oracle_out(name)[f"rad_{sun}"], miss, known)


@pytest.mark.parametrize("name", SUN)
def test_sun_scene_radiance_matches_reference(golden, oracle_out, name):
    check_radiance(golden[f"{name}__rad_sun"], oracle_out(name)["rad_sun"], None, None)


def check_radiance(ref, got, primary_miss, known):
    """The reference's transcendentals are not the oracle's (a few ulp), so paths part after their first bounce: the
    same non-finite pixels, primary misses (sky only) within the sky filter's error, and no bias over the image.
    `known`: pixels of E.sky_lookup_differs, left out (the reference's radiance there is a texel, the oracle's NaN or another
    texel)."""
    ref, got = ref.reshape(-1, 3), got.reshape(-1, 3)
    if known is not None:
        assert np.isfinite(ref[known]).all()
        ref, got = ref[~known], got[~known]
        primary_miss = primary_miss[~known]
    assert np.array_equal(np.isnan(ref), np.isnan(got))
    assert np.array_equal(np.isinf(ref), np.isinf(got)) and np.array_equal(ref[np.isinf(ref)], got[np.isinf(got)])
    fin = np.isfinite(ref).all(axis=1) & np.isfinite(got).all(axis=1)
    if primary_miss is not None:
        m = primary_miss & fin
        assert np.abs(ref[m].astype(np.float64) - got[m]).max(initial=0) <= RADIANCE_SKY_ABS
    a, b = ref[fin].astype(np.float64), got[fin].astype(np.float64)
    assert abs(a.mean() - b.mean()) <= RADIANCE_MEAN_REL * b.mean()


RADIANCE_SKY_ABS = 2e-2
RADIANCE_MEAN_REL = 5e-2
