"""A catalogue of hand-built rays that the synthetic cameras never produce.  TEST INFRASTRUCTURE ONLY.

Every scene camera sits inside the octree cube at a non-integer position and shoots jittered pinhole rays, so no
component of a ray is ever exactly zero.  Real hosts do better: a parallel projection gives axis-aligned directions, a
panoramic projector exact zeros on its centre row and column, a camera above build height starts outside the cube.
The scenes here carry one float32 ray per pixel (projectorType -1), 64 pixels a row, and each class of rays fills rows
of its own:

  A  axis-aligned directions (other components +0, then -0) from perpendicular coordinates k, k + 0.5 and k +- 1 ulp,
     k = 0, 1, the leaf-cube boundaries 2^l and 2^depth - 1; some origins on the plane 2^depth
  B  directions with one zero component, (1,1,0) and (1,1,1), through voxel edges and corners and 1 ulp beside them
  C  origins outside the cube beyond each face, edge and corner: rays that enter, miss or point away; grazing rays in
     a face's plane (and 1 ulp off it) parallel to the face; origins at 1e4 and +-3e9 (where f2i saturates)
  D  origins on or inside solid blocks: on a block's top face, inside stone, at (0,0,0), at the far corner - 1 ulp
  E  extreme directions: zero, denormal (+-1e-40), 1e30, lengths 1e-3 and 1e3, one to three +-inf or NaN components,
     a NaN origin component
  F  (scenes with BVHs) axis-aligned rays onto triangle vertices and shared edges, rays from a BVH node box's plane

Class G varies the sun instead (sun_scenes): a normal pinhole camera on terrain64 and mixed, with the altitude at
+-pi/2, 0 and -0.3, the azimuth at 0, pi/2 and pi, and the two adjacent float32 azimuths on either side of the
|sw.x| > 0.1 switch of Sun_new (sky.h:31).
"""
from __future__ import annotations

import dataclasses
import math
from typing import Callable, Dict, List, Tuple

import numpy as np

from chunkyclplugin_b200 import scenes as S

F = np.float32
WIDTH = 64
OFFSET = F(0.0001)          # constants.h:5
INF, NAN = F(np.inf), F(np.nan)
CLASSES = ("A", "B", "C", "D", "E", "F")


def up(x) -> np.float32:
    return np.nextafter(F(x), F(np.inf))


def down(x) -> np.float32:
    return np.nextafter(F(x), F(-np.inf))


def embed_octree(tree: np.ndarray, extra_levels: int) -> np.ndarray:
    """The same voxels in the low corner of a cube 2^extra_levels times larger (all other octants air)."""
    tree = np.asarray(tree, np.int32)
    k = extra_levels
    shift = 8 * k
    out = np.zeros(1 + 8 * k + tree.size - 1, np.int32)
    out[0] = 1
    for i in range(k):
        out[1 + 8 * i] = 1 + 8 * (i + 1) if i + 1 < k else (tree[0] + shift if tree[0] > 0 else tree[0])
    body = tree[1:].copy()
    body[body > 0] += shift
    out[1 + 8 * k:] = body
    return out


def _deep13():
    p = S.terrain_scene(128, 160, 90, seed=5)
    return dataclasses.replace(p, octree=embed_octree(p.octree, 6), octree_depth=p.octree_depth + 6)


BASES: Dict[str, Callable[[], S.PackedScene]] = {
    "tiny8": lambda: S.terrain_scene(8, 64, 36, seed=3),                       # depth 3
    "terrain64": lambda: S.terrain_scene(64, 160, 90, seed=7),                 # depth 6
    "decorated": lambda: S.terrain_scene(64, 160, 90, seed=11, decorate=True),  # quad and AABB models
    "mixed": S.mixed_test_scene,                                               # models, both BVHs, DoF camera
    "large512": lambda: S.large_world_scene(512, 64, 512, 160, 90),            # depth 9, top table in global memory
    "deep13": _deep13,                                                         # depth 13, 64-ary nodes (layout 2)
    "entities": lambda: S.entity_scene(128, 160, 90, n_world=96, n_actor=8, subdiv=1),
}
# scenes whose only geometry is full cubes (no models, no BVH): the independent geometric check applies
FULL_CUBE_SCENES = ("tiny8", "terrain64", "large512")


# ---------------------------------------------------------------------------------------------------------
# voxel queries (numpy restatement of octree.h:23-39, vectorised)
# ---------------------------------------------------------------------------------------------------------
def leaf_values(p: S.PackedScene, xyz: np.ndarray) -> np.ndarray:
    """Leaf value (block palette pointer, 0 = air) of each voxel of int[n, 3] `xyz` inside the cube."""
    tree = np.asarray(p.octree, np.int64)
    xyz = np.asarray(xyz, np.int64).reshape(-1, 3)
    assert ((xyz >= 0) & (xyz < (1 << p.octree_depth))).all()
    data = np.full(xyz.shape[0], tree[0])
    level = np.full(xyz.shape[0], p.octree_depth)
    while (data > 0).any():
        m = data > 0
        level[m] -= 1
        bits = (((xyz[m, 0] >> level[m]) & 1) << 2) | (((xyz[m, 1] >> level[m]) & 1) << 1) | ((xyz[m, 2] >> level[m]) & 1)
        data[m] = tree[data[m] + bits]
    return -data


def column_top(p: S.PackedScene, x: int, z: int) -> int:
    """Highest non-air y of the column (x, z), -1 for an empty column."""
    n = 1 << p.octree_depth
    ys = np.arange(min(n, 512))
    v = leaf_values(p, np.stack([np.full_like(ys, x), ys, np.full_like(ys, z)], axis=1))
    nz = np.nonzero(v)[0]
    return int(ys[nz[-1]]) if nz.size else -1


def opaque_full_cubes(p: S.PackedScene) -> set:
    """Palette pointers of blocks that are full cubes (model type 1) whose material is opaque at every texel."""
    bp = np.asarray(p.block_palette, np.int64)
    mats = np.asarray(p.mat_palette, np.int64)
    out = set()
    for ptr in range(2, bp.size - 1, 2):
        if bp[ptr] != 1:
            continue
        flags, _tint, size, loc = (int(w) & 0xFFFFFFFF for w in mats[bp[ptr + 1]:bp[ptr + 1] + 4])
        if flags & 4:
            w, h = size >> 16, size & 0xFFFF
            x0, y0 = ((loc >> 22) & 0x1FF) * 16, ((loc >> 13) & 0x1FF) * 16
            layer = min(loc & 0x7FFFF, p.atlas.shape[0] - 1)
            opaque = bool((p.atlas[layer, y0:y0 + h, x0:x0 + w, 3] > 0).all())
        else:
            opaque = (loc >> 24) > 0
        if opaque:                        # a tint never lowers alpha: the tints of material.h:66-69 have alpha 255
            out.add(ptr)
    return out


# ---------------------------------------------------------------------------------------------------------
# ray classes: each returns float32[n, 6] (origin, direction)
# ---------------------------------------------------------------------------------------------------------
def k_values(depth: int) -> List[int]:
    n = 1 << depth
    return sorted({0, 1, n - 1} | {1 << l for l in range(1, depth)})


def _rays(rows) -> np.ndarray:
    return np.array(rows, dtype=np.float32).reshape(-1, 6)


def _axis_dir(axis: int, sign: float, zero: float) -> List[float]:
    d = [zero, zero, zero]
    d[axis] = sign
    return d


def class_a(p: S.PackedScene) -> np.ndarray:
    """Axis-aligned rays.  The perpendicular coordinates pair k_i with k_(i+1) in six combinations of k, k + 0.5 and
    k +- 1 ulp; the coordinate along the axis starts inside (0.5 / n - 0.5), on the near cube plane (0 / n, the plane
    2^depth) or outside (-3 / n + 3), cycling over the pairs."""
    n = 1 << p.octree_depth
    ks = k_values(p.octree_depth)
    pairs = []
    for i, k in enumerate(ks):
        j = ks[(i + 1) % len(ks)]
        pairs += [(F(k + 0.5), F(j + 0.5)), (F(k), F(j + 0.5)), (up(k), F(j)), (down(k), down(j)), (F(k), F(j)),
                  (F(k + 0.5), up(j))]
    rows = []
    for axis in range(3):
        a, b = [c for c in range(3) if c != axis]
        for sign in (1.0, -1.0):
            starts = (F(0.5), F(0), F(-3)) if sign > 0 else (F(n - 0.5), F(n), F(n + 3))
            for zero in (0.0, -0.0):
                for i, (pa, pb) in enumerate(pairs):
                    o = [0.0, 0.0, 0.0]
                    o[axis], o[a], o[b] = starts[i % 3], pa, pb
                    rows.append(o + _axis_dir(axis, sign, zero))
    return _rays(rows)


def class_b(p: S.PackedScene) -> np.ndarray:
    """Directions with one zero component and along (1,1,0) / (1,1,1), from voxel corners and edge midpoints just above
    the ground (so that the rays run into the terrain along voxel edges and faces), and from the same points moved 1 ulp."""
    n = 1 << p.octree_depth
    dirs = [(1, 1, 0), (1, 1, 1), (-1, -1, 0), (-1, -1, -1), (1, -1, 1), (1, -1, 0), (0, -1, 1), (-1, 0, 1), (0, -1, -1),
            (0.6, -0.8, 0), (0, -0.8, -0.6), (-0.8, 0, 0.6)]
    cols = [c for c in k_values(p.octree_depth) if c < n - 1][:6] + [n // 2 - 1]
    pts = []
    for i, x in enumerate(cols):
        z = cols[(i + 2) % len(cols)]
        h = column_top(p, x, z) + 1
        h = min(max(h, 0), n - 1)
        pts += [(F(x), F(h), F(z)), (F(x), F(h + 1), F(z + 0.5)), (F(x + 0.5), F(h), F(z)),
                (up(x), F(h), F(z)), (F(x), down(h), F(z)), (F(x), F(h), up(z))]
    rows = []
    for i, o in enumerate(pts):
        for j in range(4):
            rows.append(list(o) + list(dirs[(3 * i + j) % len(dirs)]))
    return _rays(rows)


def class_c(p: S.PackedScene) -> np.ndarray:
    """Origins outside the cube: beyond each of the 6 faces, 12 edges and 8 corners a ray that enters (towards the
    centre), one that misses (towards a point beside the cube) and one that points away; grazing rays in the plane of
    each face (and 1 ulp outside and inside it) parallel to the face; origins at 1e4 and +-3e9."""
    n = 1 << p.octree_depth
    m = n / 4 + 0.37
    centre = np.array([n / 2 + 0.13, n / 2 - 0.29, n / 2 + 0.41])
    rows = []
    for cx in (-1, 0, 1):
        for cy in (-1, 0, 1):
            for cz in (-1, 0, 1):
                c = np.array([cx, cy, cz])
                if not c.any():
                    continue
                o = np.where(c < 0, -m, np.where(c > 0, n + m, centre))
                to_c = centre - o
                miss = centre + 2.0 * n * np.roll(np.where(c == 0, 1.0, c), 1) - o
                rows += [list(o) + list(to_c), list(o) + list(miss), list(o) + list(-to_c)]
    for axis in range(3):
        a, b = [c for c in range(3) if c != axis]
        for plane in (F(0), F(n)):
            for coord in (plane, up(plane), down(plane)):
                for (u, v) in ((1.0, 0.3), (-0.7, 1.0), (1.0, 0.0)):
                    o = [0.0, 0.0, 0.0]
                    o[axis], o[a], o[b] = coord, F(-m), F(n / 2 + 0.5)
                    d = [0.0, 0.0, 0.0]
                    d[a], d[b] = u if u > 0 else -u, v        # towards the cube along the face
                    rows.append(o + d)
    for far in (1e4, 3e9, -3e9):
        for axis in range(3):
            o = list(centre)
            o[axis] = far
            d = [0.0, 0.0, 0.0]
            d[axis] = -1.0 if far > 0 else 1.0
            rows.append(o + d)
            rows.append([far, far, far] + [-np.sign(far)] * 3)
    return _rays(rows)


def class_d(p: S.PackedScene) -> np.ndarray:
    """Origins on or inside solid blocks: exactly on a block's top face, inside stone, at (0,0,0) and at the far
    corner - 1 ulp, each with axis-aligned, diagonal and upward directions."""
    n = 1 << p.octree_depth
    dirs = [(0, -1, 0), (0, 1, 0), (1, 0, 0), (0, 0, -1), (0.6, -0.8, 0), (0.5, 0.5, 0.7071), (-1, -1, -1), (1, 1, 1)]
    m = min(n, 128)                      # the terrain of deep13 fills only the low 128^3 corner
    pts = []
    for x, z in ((m // 2, m // 4), (1, m - 2), (m // 4 + 1, m // 2 + 1)):
        h = column_top(p, x, z)
        if h >= 0:
            pts += [(x + 0.5, h + 1, z + 0.5), (x, h + 1, z), (x + 0.25, max(h - 2.5, 0.5), z + 0.75)]
    far = down(n)
    pts += [(0, 0, 0), (far, far, far), (0.5, 0.5, 0.5)]
    return _rays([list(o) + list(d) for o in pts for d in dirs])


def class_e(p: S.PackedScene) -> np.ndarray:
    """Extreme directions from two origins in the air (the scene camera's position, and one above the ground)."""
    n = 1 << p.octree_depth
    cam = [float(c) for c in p.camera[0:3]]
    lead = [20.3, 60.2, 20.7] if n == 64 else [n * 0.3 + 0.3, max(column_top(p, int(n * 0.3), int(n * 0.3)) + 20.2, 1.2),
                                                n * 0.3 + 0.7]
    e = 1e-40
    dirs = [(0, 0, 0), (-0.0, -0.0, -0.0), (e, -0.8, 0.3), (-e, -0.8, -e), (e, -e, e), (1e30, -1, 0.3), (0.2, -1e30, 0.1),
            (0.48e-3, -0.8e-3, 0.36e-3), (0.48e3, -0.8e3, 0.36e3), (np.inf, -0.8, 0.3), (0.2, -np.inf, 0.3),
            (np.inf, -np.inf, 0.1), (-np.inf, -np.inf, np.inf), (np.inf, 0, 0), (np.nan, -0.8, 0.3), (0.2, np.nan, 0.3),
            (np.nan, np.nan, -0.3), (np.nan, np.nan, np.nan), (np.nan, -np.inf, 0.3), (0.3, -0.8, np.nan)]
    rows = [o + list(d) for o in (lead, cam) for d in dirs]
    for o in ([np.nan, cam[1], cam[2]], [cam[0], np.nan, cam[2]], [np.nan, lead[1], np.nan]):
        for d in ((0.3, -0.8, 0.5), (-0.3, -0.8, -0.5), (0, -1, 0), (-0.0, -1, 0)):
            rows.append(o + list(d))
    return _rays(rows)


def _bvh_nodes(bvh: np.ndarray) -> np.ndarray:
    return np.asarray(bvh, np.int32).reshape(-1, 7)


def class_f(p: S.PackedScene) -> np.ndarray:
    """Axis-aligned rays onto triangle vertices and onto the midpoints of edges (shared by neighbouring triangles of
    a mesh), read from the packed triangles the BVH leaves point to; rays from the planes of BVH node boxes."""
    rows = []
    trigs = np.asarray(p.bvh_trigs, np.int32)
    tf = trigs.view(np.float32)
    for bvh in (p.world_bvh, p.actor_bvh):
        nodes = _bvh_nodes(bvh)
        leaves = [int(-w) for w in nodes[:, 0] if w <= 0][:6]
        for ptr in leaves:
            for t in range(min(int(trigs[ptr]), 2)):
                base = ptr + 1 + 20 * t
                e1, e2, o = tf[base + 1:base + 4], tf[base + 4:base + 7], tf[base + 7:base + 10]
                v1, v2 = (o + e2).astype(np.float32), (o + e1).astype(np.float32)
                for v in (o, v1, (o + v1) * F(0.5)):
                    rows.append([v[0], v[1] + 6, v[2]] + [0.0, -1.0, 0.0])
                    rows.append([v[0] - 6, v[1], v[2]] + [1.0, -0.0, 0.0])
                    rows.append([v[0], v[1], v[2] + 6] + [-0.0, 0.0, -1.0])
        for node in nodes[:8]:
            b = node[1:7].view(np.float32)
            if not np.isfinite(b).all():
                continue
            mid = [(b[0] + b[1]) / 2, (b[2] + b[3]) / 2, (b[4] + b[5]) / 2]
            rows.append([b[0], mid[1], mid[2], 1.0, 0.0, 0.0])
            rows.append([b[1], mid[1], mid[2], -1.0, -0.2, 0.0])
            rows.append([mid[0], b[3], mid[2], 0.0, -1.0, 0.0])
            rows.append([mid[0], b[3], b[4], 0.3, 0.0, 1.0])               # in the box's top plane, along its edge
    return _rays(rows)


BUILDERS = {"A": class_a, "B": class_b, "C": class_c, "D": class_d, "E": class_e, "F": class_f}


def _has_bvh(p: S.PackedScene) -> bool:
    return any(np.asarray(b).size > 7 or int(np.asarray(b)[0]) != 0 for b in (p.world_bvh, p.actor_bvh))


def catalogue_scene(name: str) -> S.PackedScene:
    """The base scene `name` with projectorType -1 and the catalogue's rays, 64 per row; meta["rows"][cls] = (first
    row, end row) of each class (a class's last row is padded with its first ray)."""
    p = BASES[name]()
    blocks, rows = [], {}
    row = 0
    for cls in CLASSES:
        if cls == "F" and not _has_bvh(p):
            continue
        r = BUILDERS[cls](p)
        nrow = -(-r.shape[0] // WIDTH)
        pad = nrow * WIDTH - r.shape[0]
        blocks.append(np.concatenate([r, np.repeat(r[:1], pad, axis=0)]))
        rows[cls] = (row, row + nrow)
        row += nrow
    rays = np.ascontiguousarray(np.concatenate(blocks).reshape(-1), dtype=np.float32)
    meta = dict(p.meta, rows=rows, base=name)
    return dataclasses.replace(p, projector_type=-1, camera=rays, width=WIDTH, height=row, name=f"edge_{name}", meta=meta)


def class_rays(p: S.PackedScene, cls: str) -> Tuple[np.ndarray, np.ndarray]:
    """(pixel indices, float32[n, 6] rays) of class `cls` in catalogue scene `p`."""
    r0, r1 = p.meta["rows"][cls]
    idx = np.arange(r0 * WIDTH, r1 * WIDTH)
    return idx, p.camera.reshape(-1, 6)[idx]


# ---------------------------------------------------------------------------------------------------------
# G: the sun at its switches
# ---------------------------------------------------------------------------------------------------------
DEFAULT_ALTITUDE, DEFAULT_AZIMUTH = 0.1745, 1.2566      # scenes.pack_sun


def switch_azimuths(altitude: float = DEFAULT_ALTITUDE) -> Tuple[float, float]:
    """The two adjacent float32 azimuths around acos(0.1 / cos(altitude)) on either side of Sun_new's
    `fabs(sw.x) > 0.1f` (sky.h:31), with sw.x = cos(azimuth) * fabs(cos(altitude)) in float32 and the oracle's cos (the
    device's dm_cos).  Returns (a, b), b = nextafter(a, +inf): |sw.x| > 0.1 at a, not at b."""
    import oracle
    r = np.abs(oracle.math_fn("cos", np.array([altitude], F)))[0]

    def above(theta):
        return abs(F(oracle.math_fn("cos", np.array([theta], F))[0] * r)) > F(0.1)

    lo, hi = F(1.3), F(1.6)
    assert above(lo) and not above(hi)
    while up(lo) != hi:
        mid = F((float(lo) + float(hi)) / 2)
        if mid in (lo, hi):
            mid = up(lo)
        if above(mid):
            lo = mid
        else:
            hi = mid
    return float(lo), float(hi)


def sun_variants() -> Dict[str, Tuple[float, float]]:
    """name -> (altitude, azimuth) as float32 values"""
    a, b = switch_azimuths()
    hp = float(F(math.pi / 2))
    out = {"alt+pi/2": (hp, DEFAULT_AZIMUTH), "alt-pi/2": (-hp, DEFAULT_AZIMUTH), "alt0": (0.0, DEFAULT_AZIMUTH),
           "alt-0.3": (-0.3, DEFAULT_AZIMUTH), "az0": (DEFAULT_ALTITUDE, 0.0), "az_pi/2": (DEFAULT_ALTITUDE, float(F(math.pi / 2))),
           "az_pi": (DEFAULT_ALTITUDE, float(F(math.pi))), "az_switch_above": (DEFAULT_ALTITUDE, a),
           "az_switch_below": (DEFAULT_ALTITUDE, b)}
    return {k: (float(F(x)), float(F(y))) for k, (x, y) in out.items()}


def sun_scene(base: str, variant: str) -> S.PackedScene:
    """terrain64 or mixed at 32 x 18 with the sun of `variant` (pinhole camera as in the parity scenes)."""
    p = BASES[base]()
    alt, az = sun_variants()[variant]
    sun = p.sun.copy()
    sun[4], sun[5] = S.f2i([alt, az])
    return dataclasses.replace(p, sun=sun, width=32, height=18, name=f"sun_{base}_{variant}")


SUN_BASES = ("terrain64", "mixed")


def scenes() -> Dict[str, S.PackedScene]:
    """Every catalogue scene and every sun scene, by name."""
    out = {f"edge_{n}": catalogue_scene(n) for n in BASES}
    for b in SUN_BASES:
        for v in sun_variants():
            out[f"sun_{b}_{v}"] = sun_scene(b, v)
    return out


def without_sun(p: S.PackedScene) -> S.PackedScene:
    sun = p.sun.copy()
    sun[0] &= ~1
    return dataclasses.replace(p, sun=sun)


# ---------------------------------------------------------------------------------------------------------
# comparisons shared by the CPU and GPU tests
# ---------------------------------------------------------------------------------------------------------
def same_bits_or_nan(a, b) -> np.ndarray:
    """Elementwise: the same float32 bits, or both NaN (whatever their sign and payload: the CPU's default NaN has the
    sign bit set, the GPU's canonical NaN does not)."""
    a = np.ascontiguousarray(a, np.float32)
    b = np.ascontiguousarray(b, np.float32)
    return (a.view(np.uint32) == b.view(np.uint32)) | (np.isnan(a) & np.isnan(b))


def sky_lookup_differs(rays: np.ndarray) -> np.ndarray:
    """Rays whose sky lookup (sky.h:97-106) the oracle, and with it the device, does not reproduce: theta =
    atan2(d.z, d.x) / 2pi is NaN (a NaN d.x or d.z), where the reference's texture unit still returns a texel; or
    atan2 is one of the IEEE special cases that detmath's atan2 does not implement: (+-0, -0), which is +-pi for the
    reference and 0 for detmath, and (+-inf, +-inf), which is an odd multiple of pi/4 for the reference and NaN for
    detmath.  Only a primary ray that misses looks up the sky in such a direction."""
    d = np.asarray(rays, np.float32).reshape(-1, 6)[:, 3:]
    nan_theta = np.isnan(d[:, 0]) | np.isnan(d[:, 2])
    both_inf = np.isinf(d[:, 0]) & np.isinf(d[:, 2])
    neg_zero = (d[:, 0] == 0) & np.signbit(d[:, 0]) & (d[:, 2] == 0)
    return nan_theta | both_inf | neg_zero


def axis_hits(p: S.PackedScene):
    """The independent geometric check for a full-cube scene: the class-A rays whose perpendicular coordinates are
    both k + 0.5.  Yields (pixel, expected) with expected = None for a ray that meets no non-air voxel, else
    (t, normal) for one whose first non-air voxel after the origin's is an opaque full cube: t is the fp64 distance
    to the face it enters, normal = -direction.  Rays that start in a non-air voxel, or whose first non-air voxel is
    not an opaque full cube, are left out."""
    n = 1 << p.octree_depth
    opaque = opaque_full_cubes(p)
    idx, rays = class_rays(p, "A")
    seen = set()
    for gid, r in zip(idx, rays):
        o, d = r[:3], r[3:]
        axis = int(np.nonzero(np.abs(d) == 1)[0][0])
        perp = [c for c in range(3) if c != axis]
        if not all(F(o[c]) - np.floor(o[c]) == F(0.5) for c in perp) or gid in seen:
            continue
        seen.add(gid)
        s = float(d[axis])
        c = float(o[axis])
        q = F(F(o[axis]) + F(d[axis]) * OFFSET)         # the voxel the march looks at first (octree.h:73-78)
        first = int(np.floor(q))
        cells = np.arange(first, n) if s > 0 else np.arange(first, -1, -1)
        cells = cells[(cells >= 0) & (cells < n)]
        if cells.size == 0:
            continue
        xyz = np.zeros((cells.size, 3), np.int64)
        xyz[:, axis] = cells
        for k in perp:
            xyz[:, k] = int(np.floor(o[k]))
        v = leaf_values(p, xyz)
        inside = 0 <= first < n
        if inside and v[0] != 0:
            continue
        nz = np.nonzero(v)[0]
        if nz.size == 0:
            yield int(gid), None
            continue
        j = int(cells[nz[0]])
        if int(v[nz[0]]) not in opaque:
            continue
        t = (j - c) if s > 0 else (c - (j + 1))
        normal = np.zeros(3)
        normal[axis] = -s
        yield int(gid), (t, normal)
