"""Synthetic scene generators that emit the reference's packed device layouts.

Nothing here renders.  These functions stand in for Chunky + the reference's
``common/export`` packers (which need a JVM and chunky-core, neither present): they
produce exactly the ``int[]`` / RGBA8 blobs the reference uploads, so the same bytes
feed the CPU oracle, the CUDA library and the reference's own OpenCL kernel.

Layouts (all ``int32`` words, floats bit-cast) follow:

* octree      ``PackedOctree.treeData`` after the leaf remap of ClSceneLoader.java:56-58 -
              node > 0: index of the first of 8 contiguous children, child order
              ``(x<<2)|(y<<1)|z`` (octree.h:84-86); node <= 0: ``-(block palette pointer)``.
* block       2 ints ``(modelType, modelPointer)``, PackedBlock.java:79-85.
* material    6 ints, PackedMaterial.java:74-100.
* aabb model  ``count`` + n x 13 ints, PackedAabb.java:75-102 / PackedAabbModel.java:40-47.
* quad model  ``count`` + n x 15 ints, PackedQuad.java:41-66 / PackedQuadModel.java.
* triangles   ``count`` + n x 20 ints, PackedTriangle.java:46-78.
* bvh         7 ints per node, PackedBvhNode.java:16-31 / AbstractSceneLoader.java:172-182.
* sun         6 ints, PackedSun.java:23-41.
* texture ref ``size = w<<16|h``, ``location = x<<22|y<<13|layer`` on a 16-px tile grid,
              ClTextureLoader.java:123-132.
* camera      ``float[15]`` = pos(3), row-major 3x3 transform(9), aperture,
              subjectDistance, fovTan, ClCamera.java:39-52.
"""
from __future__ import annotations

import dataclasses
import math
from typing import Callable, Dict, List, Optional, Tuple

import numpy as np

ANY_TYPE = 0x7FFFFFFE          # block.h:32
NAN_BITS = 0x7FC00000          # PackedBvhNode.java:19-21

# block "types" of the synthetic palette; palette pointer = 2 * type (ClPackedResourcePalette.put)
AIR, STONE, DIRT, GRASS, SAND, GLOWSTONE, GLASS, SLAB, CROSS = range(9)


def f2i(x) -> np.ndarray:
    """Float.floatToIntBits"""
    return np.asarray(x, dtype=np.float32).view(np.int32)


# --------------------------------------------------------------------------------------
# scene container
# --------------------------------------------------------------------------------------
@dataclasses.dataclass
class PackedScene:
    """Everything ``render`` binds (rayTracer.cl:11-38, SURVEY Appendix C)."""
    octree: np.ndarray            # int32[N]
    octree_depth: int
    block_palette: np.ndarray     # int32[2*nBlocks]
    quad_models: np.ndarray       # int32[]
    aabb_models: np.ndarray       # int32[]
    world_bvh: np.ndarray         # int32[7*n]
    actor_bvh: np.ndarray         # int32[7*n]
    bvh_trigs: np.ndarray         # int32[]
    atlas: np.ndarray             # uint8[layers, H, W, 4]
    mat_palette: np.ndarray       # int32[6*nMat]
    sky: np.ndarray               # uint8[res, res, 4]   (row j = phi index, col i = theta index)
    sky_intensity: float
    sun: np.ndarray               # int32[6]
    projector_type: int           # 0 pinhole, -1 pre-generated rays
    camera: np.ndarray            # float32[15] or float32[6*W*H]
    width: int
    height: int
    name: str = "scene"
    meta: dict = dataclasses.field(default_factory=dict)
    # biome colours for CCU_RENDER_BIOME_TINT: (chunks int32[n, 2] {cx, cz}, rgb float32[n, 3, 256, 3]) as
    # ccu_scene_set_biome_colors takes them (planes foliage, grass, water; texel (z & 15) * 16 + (x & 15)), or None
    biome: Optional[Tuple[np.ndarray, np.ndarray]] = None
    # fog for CCU_RENDER_FOG: (sigma, sky density, (r, g, b), fast) as ccu_scene_set_fog takes them (DESIGN.md §14), or None
    fog: Optional[Tuple[float, float, Tuple[float, float, float], bool]] = None
    # cloud layer for CCU_RENDER_CLOUDS: (mask uint8[256, 256] indexed [k, i], size, y0, y1, u0, v0) as ccu_scene_set_clouds takes
    # them (DESIGN.md §15), or None
    clouds: Optional[Tuple[np.ndarray, float, float, float, float, float]] = None

    def arrays(self) -> Dict[str, np.ndarray]:
        return {k: getattr(self, k) for k in (
            "octree", "block_palette", "quad_models", "aabb_models", "world_bvh",
            "actor_bvh", "bvh_trigs", "atlas", "mat_palette", "sky", "sun", "camera")}

    def with_resolution(self, width: int, height: int) -> "PackedScene":
        return dataclasses.replace(self, width=width, height=height)

    def nbytes(self) -> int:
        return int(sum(a.nbytes for a in self.arrays().values()))


# --------------------------------------------------------------------------------------
# integer-hash noise
# --------------------------------------------------------------------------------------
def hash_u32(*keys) -> np.ndarray:
    """Deterministic avalanche hash of integer arrays (uint32 wrap-around arithmetic)."""
    h = np.uint32(0x9E3779B9)
    with np.errstate(over="ignore"):
        for k in keys:
            k = np.asarray(k).astype(np.uint32)
            h = (h ^ k) * np.uint32(0x85EBCA6B)
            h = (h ^ (h >> np.uint32(13))) * np.uint32(0xC2B2AE35)
            h = h ^ (h >> np.uint32(16))
    return h


def value_noise(x: np.ndarray, z: np.ndarray, period: int, seed: int, octave: int) -> np.ndarray:
    """Smooth value noise in [0,1) on an integer lattice of the given period (float64)."""
    fx = x / period
    fz = z / period
    x0 = np.floor(fx).astype(np.int64)
    z0 = np.floor(fz).astype(np.int64)
    tx = fx - x0
    tz = fz - z0
    tx = tx * tx * (3 - 2 * tx)
    tz = tz * tz * (3 - 2 * tz)

    def lat(ix, iz):
        return hash_u32(ix & 0xFFFFFFFF, iz & 0xFFFFFFFF, seed, octave).astype(np.float64) / 4294967296.0

    a = lat(x0, z0)
    b = lat(x0 + 1, z0)
    c = lat(x0, z0 + 1)
    d = lat(x0 + 1, z0 + 1)
    return (a * (1 - tx) + b * tx) * (1 - tz) + (c * (1 - tx) + d * tx) * tz


def terrain_height(x: np.ndarray, z: np.ndarray, seed: int = 1337, base: int = 64, amp: int = 48) -> np.ndarray:
    """h(x,z) = base + fBm, 4 octaves (SURVEY 8d config 1)."""
    n = np.zeros(np.broadcast(x, z).shape, dtype=np.float64)
    norm = 0.0
    for o in range(4):
        w = 0.5 ** o
        n = n + w * value_noise(x, z, 64 >> o, seed, o)
        norm += w
    n = n / norm                       # [0,1)
    return (base + np.floor((n - 0.5) * 2 * amp)).astype(np.int32)


# --------------------------------------------------------------------------------------
# packed octree builder
# --------------------------------------------------------------------------------------
_MIXED = -1


def _merge_levels(types: np.ndarray) -> List[np.ndarray]:
    """U[l][x,y,z] = uniform block type of the 2^l cell, or _MIXED."""
    levels = [types.astype(np.int32)]
    cur = levels[0]
    while cur.shape[0] > 1:
        n = cur.shape[0] // 2
        c = cur.reshape(n, 2, n, 2, n, 2)
        first = c[:, 0, :, 0, :, 0]
        same = np.ones(first.shape, dtype=bool)
        for dx in (0, 1):
            for dy in (0, 1):
                for dz in (0, 1):
                    same &= c[:, dx, :, dy, :, dz] == first
        same &= first != _MIXED
        cur = np.where(same, first, _MIXED).astype(np.int32)
        levels.append(cur)
    return levels


def _subtree_blocks(levels: List[np.ndarray], leaf_value: Callable[[np.ndarray], np.ndarray]) -> Tuple[int, np.ndarray]:
    """Breadth-first child blocks of a cube whose per-level uniformity is ``levels``.

    Returns ``(root, blocks)``: ``root`` is the leaf value (<= 0) if the cube is uniform, else 1;
    ``blocks`` is int32[8*k] where a positive entry is the *block number + 1* of the child's
    own children block (caller converts to absolute indices)."""
    top = len(levels) - 1
    if levels[top][0, 0, 0] != _MIXED:
        return int(leaf_value(levels[top][0, 0, 0:1])[0]), np.zeros(0, dtype=np.int32)
    out = []
    cells = np.zeros((1, 3), dtype=np.int64)
    next_block = 1                       # block 0 = root's children
    offs = np.array([[(i >> 2) & 1, (i >> 1) & 1, i & 1] for i in range(8)], dtype=np.int64)
    for l in range(top, 0, -1):
        child = (cells[:, None, :] * 2 + offs[None, :, :]).reshape(-1, 3)
        vals = levels[l - 1][child[:, 0], child[:, 1], child[:, 2]]
        mixed = vals == _MIXED
        ent = leaf_value(vals)
        nm = int(mixed.sum())
        ent = ent.copy()
        ent[mixed] = next_block + np.arange(nm, dtype=np.int64) + 1     # block number + 1
        next_block += nm
        out.append(ent.astype(np.int32))
        cells = child[mixed]
        if nm == 0:
            break
    return 1, np.concatenate(out)


def build_octree(types: np.ndarray, block_mapping: np.ndarray) -> Tuple[np.ndarray, int]:
    """Dense ``types[x,y,z]`` (cube, power-of-two edge) -> (treeData, depth).

    Leaves hold ``-block_mapping[type]`` as after ClSceneLoader.java:56-58."""
    n = types.shape[0]
    assert types.shape == (n, n, n) and n & (n - 1) == 0
    depth = n.bit_length() - 1
    bm = np.asarray(block_mapping, dtype=np.int64)
    leaf = lambda v: -bm[np.maximum(v, 0)]
    root, blocks = _subtree_blocks(_merge_levels(types), leaf)
    if blocks.size == 0:
        return np.array([root], dtype=np.int32), depth
    pos = blocks > 0
    blocks = blocks.astype(np.int64)
    blocks[pos] = 1 + 8 * (blocks[pos] - 1)
    tree = np.concatenate([[1], blocks]).astype(np.int32)
    return tree, depth


def build_octree_tiled(tile_fn: Callable[[int, int, int], Optional[np.ndarray]], depth: int, tile_depth: int,
                       block_mapping: np.ndarray) -> Tuple[np.ndarray, int]:
    """Large worlds: ``tile_fn(tx,ty,tz)`` returns a dense 2^tile_depth cube of types or None (all air)."""
    bm = np.asarray(block_mapping, dtype=np.int64)
    leaf = lambda v: -bm[np.maximum(v, 0)]
    g = 1 << (depth - tile_depth)
    subs: Dict[Tuple[int, int, int], Tuple[int, np.ndarray]] = {}
    top0 = np.zeros((g, g, g), dtype=np.int32)
    for tx in range(g):
        for ty in range(g):
            for tz in range(g):
                t = tile_fn(tx, ty, tz)
                if t is None:
                    top0[tx, ty, tz] = AIR
                    continue
                lv = _merge_levels(t)
                u = lv[-1][0, 0, 0]
                top0[tx, ty, tz] = u
                if u == _MIXED:
                    subs[(tx, ty, tz)] = _subtree_blocks(lv, leaf)
    # top levels: reuse the BFS builder, with tiles as "voxels"; mixed tiles get a marker type
    marker_base = 1 << 20
    keys = list(subs.keys())
    top_types = top0.copy()
    for i, k in enumerate(keys):
        top_types[k] = marker_base + i
    lv = _merge_levels(top_types)

    def top_leaf(v):
        out = np.where(v >= marker_base, -(v.astype(np.int64)), -bm[np.clip(v, 0, len(bm) - 1)])
        return out
    root, blocks = _subtree_blocks(lv, top_leaf)
    if blocks.size == 0 and not keys:
        return np.array([root], dtype=np.int32), depth
    if blocks.size == 0:            # single tile world
        assert g == 1
        _, b = subs[keys[0]]
        b = b.astype(np.int64)
        p = b > 0
        b[p] = 1 + 8 * (b[p] - 1)
        return np.concatenate([[1], b]).astype(np.int32), depth
    blocks = blocks.astype(np.int64)
    pos = blocks > 0
    blocks[pos] = 1 + 8 * (blocks[pos] - 1)
    parts = [np.array([1], dtype=np.int64), blocks]
    base = 1 + blocks.size
    # splice tile subtrees
    flat = parts[1]
    for i, k in enumerate(keys):
        _, b = subs[k]
        b = b.astype(np.int64)
        p = b > 0
        b[p] = base + 8 * (b[p] - 1)
        where = np.nonzero(flat == -(marker_base + i))[0]
        assert where.size == 1
        flat[where[0]] = base
        parts.append(b)
        base += b.size
    tree = np.concatenate(parts)
    assert tree.max() < 2 ** 31
    return tree.astype(np.int32), depth


def octree_get(tree: np.ndarray, depth: int, x: int, y: int, z: int) -> Tuple[int, int, int]:
    """Point query as octree.h:23-39; returns (leaf value -data, level, node index)."""
    level = depth
    idx = 0
    data = int(tree[0])
    while data > 0:
        level -= 1
        idx = data + ((((x >> level) & 1) << 2) | (((y >> level) & 1) << 1) | ((z >> level) & 1))
        data = int(tree[idx])
    return -data, level, idx


# --------------------------------------------------------------------------------------
# textures / materials / atlas
# --------------------------------------------------------------------------------------
_BLOCK_RGB = {
    STONE: (125, 125, 125), DIRT: (134, 96, 67), GRASS: (95, 159, 53), SAND: (219, 207, 163),
    GLOWSTONE: (250, 217, 129), GLASS: (200, 230, 255), SLAB: (160, 130, 90), CROSS: (60, 170, 60),
}


def block_texture(btype: int, size: int = 16, seed: int = 7) -> np.ndarray:
    """16x16 procedural RGBA8 texture, alpha 255 (GLASS/CROSS carry alpha-0 texels)."""
    y, x = np.mgrid[0:size, 0:size]
    h = hash_u32(x, y, btype, seed)
    jitter = ((h & 0x3F).astype(np.int32) - 32)
    rgb = np.array(_BLOCK_RGB[btype], dtype=np.int32)
    tex = np.clip(rgb[None, None, :] + jitter[:, :, None], 0, 255).astype(np.uint8)
    a = np.full((size, size, 1), 255, dtype=np.uint8)
    if btype == GLASS:
        a[2:-2, 2:-2, 0] = 0                      # frame only
    if btype == CROSS:
        a[:, :, 0] = np.where(((h >> 8) & 3) == 0, 0, 255)
    return np.concatenate([tex, a], axis=2)


def sun_texture(size: int = 32) -> np.ndarray:
    y, x = np.mgrid[0:size, 0:size]
    r = np.hypot(x - (size - 1) / 2, y - (size - 1) / 2) / (size / 2)
    v = np.clip(1.2 - r, 0, 1)
    tex = np.zeros((size, size, 4), dtype=np.uint8)
    tex[..., 0] = (255 * v).astype(np.uint8)
    tex[..., 1] = (240 * v).astype(np.uint8)
    tex[..., 2] = (200 * v * v).astype(np.uint8)
    tex[..., 3] = 255
    return tex


class AtlasBuilder:
    """First-fit placement on the 16-px tile grid (ClTextureLoader.java:32-112), small canvas."""

    def __init__(self, width: int = 256, height: int = 256):
        assert width % 16 == 0 and height % 16 == 0
        self.w, self.h = width, height
        self.layers: List[np.ndarray] = [np.zeros((height, width, 4), dtype=np.uint8)]
        self.used: List[np.ndarray] = [np.zeros((width // 16, height // 16), dtype=bool)]

    def add(self, tex: np.ndarray) -> Tuple[int, int]:
        th, tw = tex.shape[:2]
        cw, ch = (tw + 15) // 16, (th + 15) // 16
        for l in range(len(self.layers) + 1):
            if l == len(self.layers):
                self.layers.append(np.zeros((self.h, self.w, 4), dtype=np.uint8))
                self.used.append(np.zeros((self.w // 16, self.h // 16), dtype=bool))
            u = self.used[l]
            for x in range(u.shape[0] - cw + 1):
                for y in range(u.shape[1] - ch + 1):
                    if not u[x:x + cw, y:y + ch].any():
                        u[x:x + cw, y:y + ch] = True
                        self.layers[l][y * 16:y * 16 + th, x * 16:x * 16 + tw] = tex
                        size = (tw << 16) | th
                        loc = (x << 22) | (y << 13) | l
                        return size, loc
        raise RuntimeError("atlas full")

    def build(self) -> np.ndarray:
        return np.stack(self.layers, axis=0)


def specular_word(specular: float = 0.0, metalness: float = 0.0, roughness: float = 0.0) -> int:
    """Word 5 of a packed material (PackedMaterial.java:69-71): specular, metalness, roughness bytes."""
    return int(specular * 255.0) | (int(metalness * 255.0) << 8) | (int(roughness * 255.0) << 16)


def pack_material(size: int, loc: int, emittance: float = 0.0, tint: int = 0, textured: bool = True,
                  argb: int = 0xFFFFFFFF, specular: float = 0.0, metalness: float = 0.0, roughness: float = 0.0) -> List[int]:
    """PackedMaterial.pack (PackedMaterial.java:88-100)."""
    flags = 4 if textured else 0
    w2, w3 = (size, loc) if textured else (-1 if argb & 0x80000000 else 0, argb)
    return [flags, tint, w2, w3, int(emittance * 255.0), specular_word(specular, metalness, roughness)]


def _i32(words) -> np.ndarray:
    return np.array([(int(w) + 2 ** 31) % 2 ** 32 - 2 ** 31 for w in words], dtype=np.int32)


# --------------------------------------------------------------------------------------
# sky / sun / camera
# --------------------------------------------------------------------------------------
def gradient_sky(res: int = 128) -> np.ndarray:
    """res x res RGBA8 equirect table; row j <-> phi (ClSky.java:41-58 loop order)."""
    j = np.arange(res, dtype=np.float64) / res                  # 0 = straight down, 1 = up
    horizon = np.array([0.80, 0.88, 1.00])
    zenith = np.array([0.25, 0.45, 0.95])
    ground = np.array([0.30, 0.28, 0.25])
    t = np.clip((j - 0.5) * 2, 0, 1)[:, None]
    up = horizon * (1 - t) + zenith * t
    g = np.clip((0.5 - j) * 2, 0, 1)[:, None]
    dn = horizon * (1 - g) + ground * g
    col = np.where((j >= 0.5)[:, None], up, dn)
    row = np.concatenate([(col * 255).astype(np.uint8), np.full((res, 1), 255, np.uint8)], axis=1)
    sky = np.repeat(row[:, None, :], res, axis=1)
    # slight azimuthal variation so theta is exercised too
    i = np.arange(res)
    sky[:, :, 0] = np.clip(sky[:, :, 0].astype(np.int32) + ((i * 8 // res) - 4)[None, :], 0, 255).astype(np.uint8)
    return np.ascontiguousarray(sky)


def pack_sun(size: int, loc: int, intensity: float = 1.25, altitude: float = 0.1745, azimuth: float = 1.2566,
             draw: bool = True) -> np.ndarray:
    """PackedSun.pack (PackedSun.java:31-41). altitude -> word 4 (phi), azimuth -> word 5 (theta)."""
    f = f2i([intensity, altitude, azimuth])
    return _i32([1 if draw else 0, size, loc, f[0], f[1], f[2]])


def pinhole_camera(pos, yaw_deg: float, pitch_deg: float, fov_deg: float = 70.0, aperture: float = 0.0,
                   subject_distance: float = 2.0) -> np.ndarray:
    """float[15] camera settings (ClCamera.java:39-52).  Image row 0 looks up (y = -0.5 -> world +y)."""
    yaw, pitch = math.radians(yaw_deg), math.radians(pitch_deg)
    fwd = np.array([math.sin(yaw) * math.cos(pitch), math.sin(pitch), math.cos(yaw) * math.cos(pitch)])
    right = np.array([math.cos(yaw), 0.0, -math.sin(yaw)])
    down = np.cross(fwd, right)
    down /= np.linalg.norm(down)
    if down[1] > 0:
        down = -down
    m = np.stack([right, down, fwd], axis=1)         # columns -> d' = M d
    fov_tan = 2.0 * math.tan(math.radians(fov_deg) / 2.0)
    out = np.concatenate([np.asarray(pos, dtype=np.float64), m.reshape(-1), [aperture, subject_distance, fov_tan]])
    return out.astype(np.float32)


def pregenerated_rays(cam15: np.ndarray, width: int, height: int, jitter: Optional[np.random.Generator] = None) -> np.ndarray:
    """float[6*W*H] (o,d) per pixel - the projectorType -1 path (ClCamera.java:72-105): pixel centres, or a fresh
    sub-pixel offset per pixel when a generator is given (the reference's jitter, ClCamera.java:83-87)."""
    pos = cam15[0:3].astype(np.float64)
    m = cam15[3:12].astype(np.float64).reshape(3, 3)
    fov_tan = float(cam15[14])
    half_w = width / (2.0 * height)
    inv_h = 1.0 / height
    px, py = np.meshgrid(np.arange(width), np.arange(height))
    ox = jitter.random((height, width), dtype=np.float32) if jitter is not None else 0.5
    oy = jitter.random((height, width), dtype=np.float32) if jitter is not None else 0.5
    x = -half_w + (px + ox) * inv_h
    y = -0.5 + (py + oy) * inv_h
    d = np.stack([fov_tan * x, fov_tan * y, np.ones_like(x)], axis=-1)
    d = d / np.linalg.norm(d, axis=-1, keepdims=True)
    d = d @ m.T
    rays = np.concatenate([np.broadcast_to(pos, d.shape), d], axis=-1)
    return np.ascontiguousarray(rays.reshape(-1).astype(np.float32))


EMPTY_BVH = _i32([0] + [NAN_BITS] * 6)


# --------------------------------------------------------------------------------------
# palette assembly
# --------------------------------------------------------------------------------------
class Palettes:
    """Block / material / model palettes for the synthetic block set."""

    def __init__(self, with_models: bool = False, atlas_wh: int = 256):
        self.atlas = AtlasBuilder(atlas_wh, atlas_wh)
        self.mat: List[int] = []
        self.blocks: List[int] = []
        self.aabb: List[int] = []
        self.quad: List[int] = []
        self.mat_ptr: Dict[int, int] = {}
        tex = {}
        for b in (STONE, DIRT, GRASS, SAND, GLOWSTONE, GLASS, SLAB, CROSS):
            tex[b] = self.atlas.add(block_texture(b))
        self.sun_tex = self.atlas.add(sun_texture())
        # block 0: air, invisible
        self.blocks += [0, 0]
        for b in (STONE, DIRT, GRASS, SAND, GLOWSTONE, GLASS):
            emit = 1.0 if b == GLOWSTONE else 0.0
            tint = (2 << 24) if b == GRASS else 0                  # biome-grass tint path (material.h:66-69)
            ptr = self.put_material(pack_material(*tex[b], emittance=emit, tint=tint))
            self.mat_ptr[b] = ptr
            self.blocks += [1, ptr]
        if with_models:
            # SLAB: AABB model, lower half cube; +z ("south" slot unreachable, SURVEY Q10) face disabled via flag 8
            m = self.put_material(pack_material(*tex[SLAB], tint=_s32(0xFF000000 | 0xE0C0A0)))
            flags = 0
            for i in range(6):
                flags |= (0b0000) << (4 * i)
            box = list(f2i([0.0, 1.0, 0.0, 0.5, 0.0, 1.0])) + [flags] + [m] * 6
            aptr = len(self.aabb)
            self.aabb += [1] + box
            self.blocks += [2, aptr]
            # CROSS: quad model, two crossed double-listed quads with alpha-tested texture
            mq = self.put_material(pack_material(*tex[CROSS], tint=(1 << 24)))
            quads = []
            for (o, xv, yv) in (((0, 0, 0), (1, 0, 1), (0, 1, 0)), ((1, 0, 1), (-1, 0, -1), (0, 1, 0)),
                                ((1, 0, 0), (-1, 0, 1), (0, 1, 0)), ((0, 0, 1), (1, 0, -1), (0, 1, 0))):
                quads += list(f2i(list(o) + list(xv) + list(yv) + [0.0, 1.0, 0.0, 1.0])) + [mq, 1]
            qptr = len(self.quad)
            self.quad += [len(quads) // 15] + quads
            self.blocks += [3, qptr]
        else:
            self.blocks += [0, 0, 0, 0]         # SLAB / CROSS unused -> invisible

    def put_material(self, words: List[int]) -> int:
        ptr = len(self.mat)
        self.mat += words
        return ptr

    @property
    def block_mapping(self) -> np.ndarray:
        return np.arange(len(self.blocks) // 2, dtype=np.int64) * 2


def _s32(v: int) -> int:
    return (v + 2 ** 31) % 2 ** 32 - 2 ** 31


# --------------------------------------------------------------------------------------
# terrain voxels
# --------------------------------------------------------------------------------------
def terrain_voxels(x0: int, z0: int, nx: int, ny: int, nz: int, seed: int = 1337, decorate: bool = False) -> np.ndarray:
    """types[x,y,z] for the column block [x0,x0+nx) x [0,ny) x [z0,z0+nz)."""
    xs = np.arange(x0, x0 + nx)
    zs = np.arange(z0, z0 + nz)
    X, Z = np.meshgrid(xs, zs, indexing="ij")
    h = terrain_height(X, Z, seed=seed)
    y = np.arange(ny)[None, :, None]
    H = h[:, None, :]
    t = np.zeros((nx, ny, nz), dtype=np.int32)
    t[y < H - 4] = STONE
    t[(y >= H - 4) & (y < H)] = DIRT
    t[np.broadcast_to(y == H, t.shape)] = GRASS
    sandy = (h <= 52)[:, None, :]
    t[np.broadcast_to((y >= H - 2) & (y <= H) & sandy, t.shape)] = SAND
    if decorate:
        r = hash_u32(X & 0xFFFFFFFF, Z & 0xFFFFFFFF, seed, 99)
        above = np.broadcast_to(y == H + 1, t.shape)
        for btype, sel in ((CROSS, (r % 11) == 0), (SLAB, (r % 37) == 1), (GLASS, (r % 53) == 2),
                           (GLOWSTONE, (r % 97) == 3)):
            t[above & np.broadcast_to(sel[:, None, :], t.shape)] = btype
    return t


def _finish(name, tree, depth, pal: Palettes, cam, width, height, world_bvh=None, actor_bvh=None, trigs=None,
            sun_draw=True, meta=None) -> PackedScene:
    return PackedScene(
        octree=tree, octree_depth=depth,
        block_palette=_i32(pal.blocks),
        quad_models=_i32(pal.quad) if pal.quad else np.zeros(1, np.int32),        # ClIntBuffer.java:15-18
        aabb_models=_i32(pal.aabb) if pal.aabb else np.zeros(1, np.int32),
        world_bvh=EMPTY_BVH.copy() if world_bvh is None else world_bvh,
        actor_bvh=EMPTY_BVH.copy() if actor_bvh is None else actor_bvh,
        bvh_trigs=np.zeros(1, np.int32) if trigs is None else trigs,
        atlas=pal.atlas.build(), mat_palette=_i32(pal.mat),
        sky=gradient_sky(128), sky_intensity=1.25,
        sun=pack_sun(*pal.sun_tex, draw=sun_draw),
        projector_type=0, camera=cam, width=width, height=height, name=name, meta=meta or {})


def terrain_scene(size: int = 256, width: int = 1920, height: int = 1080, seed: int = 1337, decorate: bool = False,
                  sun: bool = True, name: Optional[str] = None) -> PackedScene:
    """BASELINE config 1/2: size^3 procedural terrain, sun + sky, no entities."""
    assert size & (size - 1) == 0
    pal = Palettes(with_models=decorate)
    ny = min(size, 256)
    vox = np.zeros((size, size, size), dtype=np.int32)
    vox[:, :ny, :] = terrain_voxels(0, 0, size, ny, size, seed=seed, decorate=decorate)
    if size < 128:                                          # small test worlds: lower the terrain into the cube
        vox = np.zeros((size, size, size), dtype=np.int32)
        full = terrain_voxels(0, 0, size, 256, size, seed=seed, decorate=decorate)
        shift = 64 - size // 3
        vox[:, :size, :] = full[:, shift:shift + size, :]
    tree, depth = build_octree(vox, pal.block_mapping)
    hc = int(np.nonzero(vox[size // 2, :, size // 16] != AIR)[0].max(initial=0))
    cam = pinhole_camera((size / 2 + 0.37, hc + 40 * size / 256 + 0.21, size / 16 + 0.11), 0.0, -30.0, 70.0)
    return _finish(name or f"terrain{size}", tree, depth, pal, cam, width, height, sun_draw=sun,
                   meta={"size": size, "seed": seed, "decorate": decorate})


def indoor_scene(size: int = 256, width: int = 1920, height: int = 1080, seed: int = 4242) -> PackedScene:
    """BASELINE config 3: solid stone with carved rooms/corridors, glowstone on ceilings, sun flag off."""
    pal = Palettes()
    vox, cam = _indoor_voxels(size, seed)
    tree, depth = build_octree(vox, pal.block_mapping)
    return _finish(f"indoor{size}", tree, depth, pal, cam, width, height, sun_draw=False,
                   meta={"size": size, "seed": seed})


def _indoor_voxels(size: int, seed: int):
    """indoor_scene's types[x, y, z] and camera"""
    vox = np.full((size, size, size), STONE, dtype=np.int32)
    cell = 16
    n = size // cell
    cx, cy, cz = np.mgrid[0:n, 0:n, 0:n]
    r = hash_u32(cx, cy, cz, seed)
    room = (r % 3) != 0
    for ix in range(n):
        for iy in range(n):
            for iz in range(n):
                x0, y0, z0 = ix * cell, iy * cell, iz * cell
                if room[ix, iy, iz]:
                    vox[x0 + 1:x0 + cell - 1, y0 + 1:y0 + cell - 3, z0 + 1:z0 + cell - 1] = AIR
                # corridors along +x and +z through the walls
                hh = int(r[ix, iy, iz] >> 8)
                if hh & 1:
                    vox[x0 + cell - 2:x0 + cell + 2, y0 + 1:y0 + 5, z0 + 6:z0 + 10] = AIR
                if hh & 2:
                    vox[x0 + 6:x0 + 10, y0 + 1:y0 + 5, z0 + cell - 2:z0 + cell + 2] = AIR
                if hh & 4:
                    vox[x0 + 6:x0 + 10, y0 + cell - 4:y0 + cell + 2, z0 + 6:z0 + 10] = AIR
    vox = vox[:size, :size, :size]
    # glowstone with probability 1/64 on ceilings (stone voxel with air directly below)
    ceil = (vox[:, 1:, :] == STONE) & (vox[:, :-1, :] == AIR)
    X, Y, Z = np.mgrid[0:size, 1:size, 0:size]
    pick = (hash_u32(X, Y, Z, seed + 1) % 64) == 0
    sel = np.zeros_like(vox, dtype=bool)
    sel[:, 1:, :] = ceil & pick
    vox[sel] = GLOWSTONE
    # camera inside a room near the centre
    ix = iy = iz = n // 2
    found = None
    for d in range(n):
        for (a, b, c) in ((ix + d, iy, iz), (ix, iy + d, iz), (ix, iy, iz + d), (ix - d, iy, iz)):
            if 0 <= a < n and 0 <= b < n and 0 <= c < n and room[a, b, c]:
                found = (a, b, c)
                break
        if found:
            break
    a, b, c = found
    cam = pinhole_camera((a * cell + 3.3, b * cell + 4.2, c * cell + 2.6), 35.0, -8.0, 90.0)
    return vox, cam


def large_world_scene(sx: int = 2048, sy: int = 256, sz: int = 2048, width: int = 3840, height: int = 2160,
                      seed: int = 1337) -> PackedScene:
    """BASELINE config 5: sx x sy x sz terrain inside a power-of-two cube (depth 11 for 2048)."""
    pal = Palettes()
    edge = max(sx, sy, sz)
    depth = edge.bit_length() - 1
    td = min(8, depth)
    ts = 1 << td

    def tile(tx, ty, tz):
        if ty * ts >= sy or tx * ts >= sx or tz * ts >= sz:
            return None
        t = np.zeros((ts, ts, ts), dtype=np.int32)
        ny = min(ts, sy - ty * ts)
        full = terrain_voxels(tx * ts, tz * ts, ts, sy, ts, seed=seed)
        t[:, :ny, :] = full[:, ty * ts:ty * ts + ny, :]
        return t

    tree, depth = build_octree_tiled(tile, depth, td, pal.block_mapping)
    h = int(terrain_height(np.array([sx // 2]), np.array([sz // 16]), seed=seed)[0])
    cam = pinhole_camera((sx / 2 + 0.37, h + 60.21, sz / 16 + 0.11), 0.0, -25.0, 70.0)
    return _finish(f"large{sx}x{sy}x{sz}", tree, depth, pal, cam, width, height,
                   meta={"size": (sx, sy, sz), "seed": seed})


# --------------------------------------------------------------------------------------
# entities: triangle meshes + binary BVH in Chunky's packed layout
# --------------------------------------------------------------------------------------
def _icosphere(subdiv: int = 2) -> Tuple[np.ndarray, np.ndarray]:
    t = (1 + 5 ** 0.5) / 2
    v = np.array([[-1, t, 0], [1, t, 0], [-1, -t, 0], [1, -t, 0], [0, -1, t], [0, 1, t], [0, -1, -t], [0, 1, -t],
                  [t, 0, -1], [t, 0, 1], [-t, 0, -1], [-t, 0, 1]], dtype=np.float64)
    v /= np.linalg.norm(v, axis=1, keepdims=True)
    f = np.array([[0, 11, 5], [0, 5, 1], [0, 1, 7], [0, 7, 10], [0, 10, 11], [1, 5, 9], [5, 11, 4], [11, 10, 2],
                  [10, 7, 6], [7, 1, 8], [3, 9, 4], [3, 4, 2], [3, 2, 6], [3, 6, 8], [3, 8, 9], [4, 9, 5], [2, 4, 11],
                  [6, 2, 10], [8, 6, 7], [9, 8, 1]], dtype=np.int64)
    for _ in range(subdiv):
        verts = list(map(tuple, v))
        cache: Dict[Tuple[int, int], int] = {}

        def mid(a, b):
            k = (min(a, b), max(a, b))
            if k not in cache:
                m = (np.array(verts[a]) + np.array(verts[b])) / 2
                m /= np.linalg.norm(m)
                verts.append(tuple(m))
                cache[k] = len(verts) - 1
            return cache[k]
        nf = []
        for a, b, c in f:
            ab, bc, ca = mid(a, b), mid(b, c), mid(c, a)
            nf += [[a, ab, ca], [b, bc, ab], [c, ca, bc], [ab, bc, ca]]
        v = np.array(verts)
        f = np.array(nf, dtype=np.int64)
    return v, f            # counter-clockwise seen from outside


def _box_mesh() -> Tuple[np.ndarray, np.ndarray]:
    v = np.array([[x, y, z] for x in (0, 1) for y in (0, 1) for z in (0, 1)], dtype=np.float64) - 0.5
    q = [(0, 1, 3, 2), (4, 6, 7, 5), (0, 4, 5, 1), (2, 3, 7, 6), (0, 2, 6, 4), (1, 5, 7, 3)]
    f = []
    for a, b, c, d in q:
        f += [[a, b, c], [a, c, d]]
    f = np.array(f, dtype=np.int64)
    # orient outward (ccw from outside)
    tri = v[f]
    n = np.cross(tri[:, 1] - tri[:, 0], tri[:, 2] - tri[:, 0])
    flip = (n * tri.mean(axis=1)).sum(axis=1) < 0
    f[flip] = f[flip][:, ::-1]
    return v, f


def pack_triangles(tris: np.ndarray, material: np.ndarray, double_sided: np.ndarray) -> np.ndarray:
    """tris float64[n,3,3] with outward ccw winding -> int32[n,20] (PackedTriangle.java:71-78).

    Triangle_intersect (primitives.h:368-409) accepts a single-sided triangle only when
    ``dot(e1, cross(dir, e2)) <= -EPS``, i.e. when the ray travels along e1 x e2; so for a
    triangle visible from outside e1 x e2 must point inward: o = v0, e1 = v2 - v0, e2 = v1 - v0."""
    n = tris.shape[0]
    v0, v1, v2 = tris[:, 0], tris[:, 1], tris[:, 2]
    e1 = v2 - v0
    e2 = v1 - v0
    nrm = np.cross(v1 - v0, v2 - v0)
    nrm /= np.maximum(np.linalg.norm(nrm, axis=1, keepdims=True), 1e-30)
    out = np.zeros((n, 20), dtype=np.int32)
    out[:, 0] = 1 | (double_sided.astype(np.int32) << 8)
    out[:, 1:4] = f2i(e1)
    out[:, 4:7] = f2i(e2)
    out[:, 7:10] = f2i(v0)
    out[:, 10:13] = f2i(nrm)
    uv = np.array([1.0, 0.0, 0.0, 1.0, 0.0, 0.0])            # t1 (at o+e1), t2 (at o+e2), t3 (at o)
    out[:, 13:19] = f2i(np.broadcast_to(uv, (n, 6)))
    out[:, 19] = material
    return out


def build_bvh(tris: np.ndarray, packed: np.ndarray, trig_palette: List[np.ndarray], trig_base: int,
              leaf_size: int = 4) -> Tuple[np.ndarray, int]:
    """Median-split binary BVH in the BinaryBVH.packed layout the reference consumes (bvh.h:47-110):
    node = 7 ints {child, xmin,xmax,ymin,ymax,zmin,zmax}; inner: word0 > 0 = index of 2nd child, 1st child
    directly follows; leaf: word0 <= 0 = -(pointer into the triangle palette).  Appends leaf triangle models
    (count + n x 20 ints) to ``trig_palette``; returns (nodes, new_trig_base)."""
    lo = tris.min(axis=1)
    hi = tris.max(axis=1)
    cen = (lo + hi) * 0.5
    lo32 = lo.astype(np.float32)
    hi32 = hi.astype(np.float32)
    # conservative float32 bounds
    lo32 = np.where(lo32.astype(np.float64) > lo, np.nextafter(lo32, np.float32(-np.inf)), lo32)
    hi32 = np.where(hi32.astype(np.float64) < hi, np.nextafter(hi32, np.float32(np.inf)), hi32)
    nodes: List[List[int]] = []
    ptr = trig_base

    # iterative DFS; each stack item: (index array, slot of parent's "second child" field or None)
    order = np.arange(tris.shape[0])
    stack = [(order, None)]
    while stack:
        idx, fix = stack.pop()
        me = len(nodes)
        if fix is not None:
            nodes[fix][0] = me * 7
        b = [lo32[idx, 0].min(), hi32[idx, 0].max(), lo32[idx, 1].min(), hi32[idx, 1].max(),
             lo32[idx, 2].min(), hi32[idx, 2].max()]
        bw = list(f2i(b))
        if idx.size <= leaf_size:
            nodes.append([-ptr] + bw)
            trig_palette.append(np.concatenate([[idx.size], packed[idx].reshape(-1)]).astype(np.int32))
            ptr += 1 + 20 * idx.size
            continue
        ext = cen[idx].max(axis=0) - cen[idx].min(axis=0)
        ax = int(np.argmax(ext))
        half = idx.size // 2
        part = np.argpartition(cen[idx, ax], half)
        left, right = idx[part[:half]], idx[part[half:]]
        nodes.append([0] + bw)
        # first child must directly follow -> push right first (with fix-up), then left
        stack.append((right, me))
        stack.append((left, None))
    return _i32(np.array(nodes, dtype=np.int64).reshape(-1)), ptr


def entity_scene(size: int = 256, width: int = 1920, height: int = 1080, n_world: int = 2048, n_actor: int = 64,
                 seed: int = 1337, subdiv: int = 2) -> PackedScene:
    """BASELINE config 4: terrain + synthetic meshes (icospheres + boxes) in world / actor BVHs."""
    base = terrain_scene(size, width, height, seed=seed)
    pal = Palettes()
    sv, sf = _icosphere(subdiv)
    bv, bf = _box_mesh()
    mats = [pal.put_material(pack_material(*pal.atlas.add(block_texture(b, seed=seed + 11)), emittance=e))
            for b, e in ((SAND, 0.0), (GLASS, 0.0), (GLOWSTONE, 0.5), (STONE, 0.0))]
    trig_palette: List[np.ndarray] = []

    def meshes(count: int, salt: int):
        i = np.arange(count)
        px = (hash_u32(i, salt, 1) % (size * 16)).astype(np.float64) / 16.0
        pz = (hash_u32(i, salt, 2) % (size * 16)).astype(np.float64) / 16.0
        h = terrain_height(np.floor(px).astype(np.int64), np.floor(pz).astype(np.int64), seed=seed)
        py = h + 2.0 + (hash_u32(i, salt, 3) % 256).astype(np.float64) / 16.0
        rad = 0.5 + (hash_u32(i, salt, 4) % 64).astype(np.float64) / 32.0
        kind = hash_u32(i, salt, 5) % 4
        T, M, D = [], [], []
        for k in range(count):
            v, f = (bv, bf) if kind[k] == 0 else (sv, sf)
            w = v * rad[k] * (2.0 if kind[k] == 0 else 1.0) + np.array([px[k], py[k], pz[k]])
            T.append(w[f])
            M.append(np.full(f.shape[0], mats[int(kind[k])], dtype=np.int64))
            D.append(np.full(f.shape[0], kind[k] == 0))
        return np.concatenate(T), np.concatenate(M), np.concatenate(D)

    tw, mw, dw = meshes(n_world, 101)
    ta, ma, da = meshes(n_actor, 202)
    wb, nxt = build_bvh(tw, pack_triangles(tw, mw, dw), trig_palette, 0)
    ab, nxt = build_bvh(ta, pack_triangles(ta, ma, da), trig_palette, nxt)
    trigs = np.concatenate(trig_palette).astype(np.int32)
    assert trigs.size == nxt
    # re-use terrain octree; palettes must be the ones with the extra materials
    tree = base.octree
    return _finish(f"entities{size}", tree, base.octree_depth, pal, base.camera, width, height,
                   world_bvh=wb, actor_bvh=ab, trigs=trigs,
                   meta={"size": size, "world_tris": int(tw.shape[0]), "actor_tris": int(ta.shape[0])})


# (specular, metalness, roughness) that glossy() hands out in turn: specular only, metal only, specular + rough, zero,
# metal + specular + rough
GLOSS = ((0.8, 0.0, 0.0), (0.0, 0.9, 0.0), (0.7, 0.0, 0.5), (0.0, 0.0, 0.0), (0.3, 0.6, 0.25))


def glossy(p: PackedScene) -> PackedScene:
    """The scene with word 5 of its materials set (CCU_RENDER_SPECULAR): materials take the GLOSS entries in turn, emitters
    become emissive-specular.  Full cubes, model blocks and entity triangles of the scene thereby get a mix of materials."""
    mp = p.mat_palette.copy()
    for i in range(mp.size // 6):
        emissive = (mp[6 * i] & 2) or (mp[6 * i + 4] & 0xFF)
        mp[6 * i + 5] = specular_word(0.5) if emissive else specular_word(*GLOSS[i % len(GLOSS)])
    return dataclasses.replace(p, mat_palette=mp, name=p.name + "_glossy")


def mixed_test_scene(size: int = 64, width: int = 96, height: int = 54, seed: int = 99) -> PackedScene:
    """Small scene that exercises every branch: model blocks, alpha tests, tints, emitters, both BVHs, DoF."""
    base = terrain_scene(size, width, height, seed=seed, decorate=True)
    pal = Palettes(with_models=True)
    sv, sf = _icosphere(1)
    bv, bf = _box_mesh()
    m0 = pal.put_material(pack_material(0, 0, textured=False, argb=_s32(0xFFC08040)))
    m1 = pal.put_material(pack_material(*pal.atlas.add(block_texture(GLASS, seed=5)), emittance=0.25))
    trig_palette: List[np.ndarray] = []
    c = np.array([size / 2, size * 0.55, size / 2])
    tw = np.concatenate([(sv * 4 + c + [6, 3, 8])[sf], (bv * 5 + c + [-7, 2, 10])[bf]])
    mw = np.concatenate([np.full(sf.shape[0], m0), np.full(bf.shape[0], m1)])
    dw = np.concatenate([np.zeros(sf.shape[0], bool), np.ones(bf.shape[0], bool)])
    ta = (sv * 2.5 + c + [0, 6, 14])[sf]
    wb, nxt = build_bvh(tw, pack_triangles(tw, mw, dw), trig_palette, 0, leaf_size=3)
    ab, nxt = build_bvh(ta, pack_triangles(ta, np.full(sf.shape[0], m1), np.ones(sf.shape[0], bool)), trig_palette, nxt, leaf_size=2)
    trigs = np.concatenate(trig_palette).astype(np.int32)
    cam = base.camera.copy()
    cam[12] = 0.05          # aperture > 0 -> DoF draws (camera.h:21-31)
    cam[13] = 20.0
    s = _finish(f"mixed{size}", base.octree, base.octree_depth, pal, cam, width, height,
                world_bvh=wb, actor_bvh=ab, trigs=trigs, meta={"size": size})
    return s


# --------------------------------------------------------------------------------------
# model-block lights (CCU_RENDER_EMITTER_MODELS, DESIGN.md §12): torches and lanterns
# --------------------------------------------------------------------------------------
TORCH, LANTERN = 9, 10          # type indices of Palettes.block_mapping after add_model_lights


def torch_texture(size: int = 16, seed: int = 7) -> np.ndarray:
    """A 2-texel-wide stick (columns 7, 8) with a flame in its top three rows; every other texel, and two texels of the flame
    tip, are alpha 0 (the alpha test cuts them)."""
    y, x = np.mgrid[0:size, 0:size]
    h = hash_u32(x, y, 101, seed)
    tex = np.zeros((size, size, 4), np.uint8)
    stick = (x >= 7) & (x <= 8)
    flame = stick & (y < 3)
    tex[stick] = [120, 85, 45, 255]
    tex[flame] = [255, 210, 90, 255]
    tex[..., 0] = np.clip(tex[..., 0].astype(np.int32) + ((h & 15).astype(np.int32) - 8) * stick, 0, 255).astype(np.uint8)
    tex[0, 7, 3] = tex[0, 8, 3] = 0
    return tex


def _torch_quads(mat: int) -> List[int]:
    """Four one-sided outward quads around the stick [7/16, 9/16] x [0, 10/16] x [7/16, 9/16] and one on its top, the sides
    mapped to the stick's texels and the top to the flame; packed as PackedQuad words (PackedQuad.java:41-66)."""
    a, b, t = 7 / 16, 9 / 16, 10 / 16
    w = b - a
    quads = []
    for o, xv, yv in (((a, 0, a), (0, 0, w), (0, t, 0)),      # -x
                      ((b, 0, b), (0, 0, -w), (0, t, 0)),     # +x
                      ((b, 0, a), (-w, 0, 0), (0, t, 0)),     # -z
                      ((a, 0, b), (w, 0, 0), (0, t, 0)),      # +z
                      ((a, t, a), (0, 0, w), (w, 0, 0))):     # +y
        uv = [a, w, 0.0, t] if yv[1] else [a, w, 1 - 3 / 16, 2 / 16]
        quads += list(f2i(list(o) + list(xv) + list(yv) + uv)) + [mat, 0]
    return [len(quads) // 15] + quads


def _lantern_boxes(body: int, cap: int) -> List[int]:
    """An emitting body box whose bottom (-y) face is disabled and whose +x face is flipped in u (its +z face reads material
    0, SURVEY Q10), under a non-emitting cap box; packed as PackedAabb words (PackedAabb.java:75-102)."""
    flags = (0b1000 << 20) | (0b0100 << 4)
    out = [2]
    for box, m, fl in (((5 / 16, 11 / 16, 1 / 16, 8 / 16, 5 / 16, 11 / 16), body, flags), ((6 / 16, 10 / 16, 8 / 16, 10 / 16, 6 / 16, 10 / 16), cap, 0)):
        out += list(f2i(list(box))) + [fl] + [m] * 6
    return out


def add_model_lights(pal: Palettes, emittance: float = 1.0) -> Tuple[int, int]:
    """Appends a torch (quad model, alpha-tested textured emitter) and a lantern (AABB model mixing emitting and non-emitting
    faces) to the palettes; returns their block palette positions (type indices TORCH, LANTERN)."""
    assert len(pal.blocks) == 2 * TORCH
    torch = pal.put_material(pack_material(*pal.atlas.add(torch_texture()), emittance=emittance))
    body = pal.put_material(pack_material(*pal.atlas.add(block_texture(GLOWSTONE, seed=11)), emittance=emittance))
    cap = pal.put_material(pack_material(0, 0, textured=False, argb=_s32(0xFF404048)))
    qptr = len(pal.quad)
    pal.quad += _torch_quads(torch)
    aptr = len(pal.aabb)
    pal.aabb += _lantern_boxes(body, cap)
    b_torch = len(pal.blocks)
    pal.blocks += [3, qptr]
    b_lantern = len(pal.blocks)
    pal.blocks += [2, aptr]
    return b_torch, b_lantern


def indoor_models_scene(size: int = 256, width: int = 1920, height: int = 1080, seed: int = 4242) -> PackedScene:
    """BASELINE config 3 lit only by model blocks: the rooms, corridors and camera of indoor_scene, no glowstone; a lantern
    hangs under each ceiling voxel that indoor_scene turns into glowstone, and torches stand on 1 in 64 floor voxels."""
    pal = Palettes()
    add_model_lights(pal)
    vox, cam = _indoor_voxels(size, seed)
    X, Y, Z = np.mgrid[0:size, 0:size, 0:size]
    lamp = vox == GLOWSTONE
    vox[lamp] = STONE
    below = np.zeros_like(lamp)
    below[:, :-1, :] = lamp[:, 1:, :]
    vox[below & (vox == AIR)] = LANTERN
    floor = np.zeros_like(lamp)
    floor[:, 1:, :] = (vox[:, :-1, :] == STONE) & (vox[:, 1:, :] == AIR)
    vox[floor & ((hash_u32(X, Y, Z, seed + 2) % 64) == 0)] = TORCH
    tree, depth = build_octree(vox, pal.block_mapping)
    return _finish(f"indoor_models{size}", tree, depth, pal, cam, width, height, sun_draw=False,
                   meta={"size": size, "seed": seed})


def emissive_models(p: PackedScene, emittance: float = 1.0) -> PackedScene:
    """p with every material that a quad or AABB model of its block palette references made emissive (emittance byte), the
    rest unchanged: config 1 decorated with its CROSS and SLAB blocks lit."""
    bp = np.asarray(p.block_palette, np.int64)
    mp = np.array(p.mat_palette, np.int32)
    mats = set()
    for b in range(0, bp.size - 1, 2):
        if bp[b] == 3:
            q = int(bp[b + 1])
            mats.update(int(p.quad_models[q + 1 + 15 * i + 13]) for i in range(int(p.quad_models[q])))
        elif bp[b] == 2:
            a = int(bp[b + 1])
            mats.update(int(p.aabb_models[a + 1 + 13 * i + k]) for i in range(int(p.aabb_models[a])) for k in range(7, 13))
    for m in mats:
        mp[m + 4] = int(emittance * 255.0)
    return dataclasses.replace(p, mat_palette=mp, name=p.name + "_litmodels")


# --------------------------------------------------------------------------------------
# biome colours (CCU_RENDER_BIOME_TINT, DESIGN.md §13)
# --------------------------------------------------------------------------------------
def biome_field(chunks: np.ndarray, seed: int = 1) -> np.ndarray:
    """float32[n, 3, 256, 3] linear colours of the chunks {cx, cz}: per plane a field that runs at different rates along x and z
    (so that a swapped axis, a wrong chunk or a wrong texel shows), offset by a hash of the chunk."""
    chunks = np.asarray(chunks, np.int64).reshape(-1, 2)
    t = np.arange(256)
    x = chunks[:, 0:1] * 16 + (t & 15)[None, :]          # [n, 256] voxel x of every texel
    z = chunks[:, 1:2] * 16 + (t >> 4)[None, :]
    out = np.empty((chunks.shape[0], 3, 256, 3), np.float32)
    for plane in range(3):
        h = hash_u32(chunks[:, 0], chunks[:, 1], seed, plane).astype(np.float64)[:, None] / 2.0 ** 32
        for c, (fx, fz) in enumerate(((0.031, 0.007), (0.005, 0.043), (0.019, 0.013))):
            f = (x * fx + z * (fz * (plane + 1)) + h * (c + 1)) % 1.0
            out[:, plane, :, c] = 0.05 + 0.9 * f
    return out


def with_biomes(p: PackedScene, seed: int = 1, holes: float = 0.125) -> PackedScene:
    """p with biome colours over the octree's max(1, 2^depth / 16)^2 chunks (biome_field); a hash of the chunk leaves out about
    the fraction `holes` of them."""
    g = max(1, (1 << p.octree_depth) // 16)
    cx, cz = np.meshgrid(np.arange(g), np.arange(g), indexing="ij")
    chunks = np.stack([cx.reshape(-1), cz.reshape(-1)], 1)
    keep = hash_u32(chunks[:, 0], chunks[:, 1], seed, 7).astype(np.float64) / 2.0 ** 32 >= holes
    chunks = chunks[keep].astype(np.int32)
    return dataclasses.replace(p, biome=(chunks, biome_field(chunks, seed)), name=p.name + "_biomes")


def water_tinted(p: PackedScene) -> PackedScene:
    """p with every second untinted full-cube material given the water tint (tint type 3)."""
    bp = np.asarray(p.block_palette, np.int64)
    mp = np.array(p.mat_palette, np.int32)
    mats = sorted({int(bp[b + 1]) for b in range(0, bp.size - 1, 2) if bp[b] == 1 and mp[int(bp[b + 1]) + 1] == 0})
    for m in mats[::2]:
        mp[m + 1] = 3 << 24
    return dataclasses.replace(p, mat_palette=mp, name=p.name + "_water")


# --------------------------------------------------------------------------------------
# cloud layer (CCU_RENDER_CLOUDS, DESIGN.md §15)
# --------------------------------------------------------------------------------------
def cloud_mask(seed: int = 1, cover: float = 0.5) -> np.ndarray:
    """uint8[256, 256] (indexed [k, i]): cell (i, k) is set where a hash of the cell falls below `cover`."""
    k, i = np.meshgrid(np.arange(256), np.arange(256), indexing="ij")
    h = hash_u32(i.reshape(-1), k.reshape(-1), seed, 11).astype(np.float64) / 2.0 ** 32
    return (h < cover).astype(np.uint8).reshape(256, 256)


def with_clouds(p: PackedScene, mask: np.ndarray, size: float = 4.0, y0: float = None, y1: float = None, u0: float = 0.0,
                v0: float = 0.0) -> PackedScene:
    """p with a cloud layer of `mask` (uint8[256, 256] indexed [k, i]), cells of `size` blocks; the slab defaults to
    [3/4, 7/8] of the octree's height."""
    h = float(1 << p.octree_depth)
    y0 = 0.75 * h if y0 is None else y0
    y1 = 0.875 * h if y1 is None else y1
    m = np.ascontiguousarray(mask, np.uint8).reshape(256, 256)
    return dataclasses.replace(p, clouds=(m, float(size), float(y0), float(y1), float(u0), float(v0)), name=p.name + "_clouds")
