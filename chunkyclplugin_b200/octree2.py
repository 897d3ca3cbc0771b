"""Loader for Chunky's ``.octree2`` scene files (SURVEY 8f #4), so that a saved Chunky scene - e.g. the reference's own
benchmark scene ``benchmark/OpenCL_test/OpenCL_test.octree2`` - renders through the C ABI without Chunky.

File layout (gzip stream, big-endian; version 6 as written by chunky-core 2.5.0-SNAPSHOT, the version the reference builds
against, build.gradle:22): ``int version``, ``int paletteVersion``, ``int nBlocks`` followed by one NBT compound body per
block (``Name`` string + optional ``Properties`` compound), then the world octree and the water octree, each ``int depth``
+ nodes in pre-order (``-1`` = branch followed by its 8 children, anything else = leaf holding a palette index; the child
order is the kernel's ``x<<2 | y<<1 | z``, octree.h:84-86), then - optionally - Chunky's three biome colour textures in the
order grass, foliage, water: each ``int count`` followed by ``count`` tiles of ``int x, int z`` (chunk coordinates in octree
space) and 256 x 3 floats, texel (z & 15) * 16 + (x & 15), linear RGB.  A file that ends after the water octree has none.

The packed node array produced is the layout the reference uploads (``PackedOctree.treeData`` after the leaf remap of
ClSceneLoader.java:52-63): root at 0, a branch holds the index of its first child, its 8 children are contiguous, a leaf
holds ``-(block palette pointer)``; ANY_TYPE leaves are kept verbatim (ClSceneLoader.java:57).

Chunky's real block models and textures live in chunky-core and Minecraft's assets (absent here), so blocks become full
cubes with a flat colour derived from the block name (a small table for the common blocks, a hash otherwise); ``air``,
``cave_air`` and ``void_air`` map to the invisible block 0.
"""
from __future__ import annotations

import gzip
import struct
import zlib
from dataclasses import dataclass
from typing import Dict, List, Optional, Tuple

import numpy as np

from . import scenes as S

BRANCH = -1
ANY_TYPE = 0x7FFFFFFE


# ------------------------------------------------------------------------------------------------------
# NBT (the subset block palettes use)
# ------------------------------------------------------------------------------------------------------
def _nbt_payload(buf: bytes, pos: int, tag: int):
    if tag == 1:
        return buf[pos], pos + 1
    if tag == 2:
        return struct.unpack_from(">h", buf, pos)[0], pos + 2
    if tag == 3:
        return struct.unpack_from(">i", buf, pos)[0], pos + 4
    if tag == 4:
        return struct.unpack_from(">q", buf, pos)[0], pos + 8
    if tag == 5:
        return struct.unpack_from(">f", buf, pos)[0], pos + 4
    if tag == 6:
        return struct.unpack_from(">d", buf, pos)[0], pos + 8
    if tag == 7:
        n = struct.unpack_from(">i", buf, pos)[0]
        return buf[pos + 4:pos + 4 + n], pos + 4 + n
    if tag == 8:
        n = struct.unpack_from(">H", buf, pos)[0]
        return buf[pos + 2:pos + 2 + n].decode("utf-8", errors="replace"), pos + 2 + n
    if tag == 9:
        et = buf[pos]
        n = struct.unpack_from(">i", buf, pos + 1)[0]
        pos += 5
        out = []
        for _ in range(n):
            v, pos = _nbt_payload(buf, pos, et)
            out.append(v)
        return out, pos
    if tag == 10:
        return _nbt_compound_body(buf, pos)
    if tag == 11:
        n = struct.unpack_from(">i", buf, pos)[0]
        return list(struct.unpack_from(f">{n}i", buf, pos + 4)), pos + 4 + 4 * n
    if tag == 12:
        n = struct.unpack_from(">i", buf, pos)[0]
        return list(struct.unpack_from(f">{n}q", buf, pos + 4)), pos + 4 + 8 * n
    raise ValueError(f"unknown NBT tag {tag} at {pos}")


def _nbt_compound_body(buf: bytes, pos: int) -> Tuple[Dict[str, object], int]:
    """Named tags up to TAG_End."""
    out: Dict[str, object] = {}
    while True:
        tag = buf[pos]
        pos += 1
        if tag == 0:
            return out, pos
        n = struct.unpack_from(">H", buf, pos)[0]
        name = buf[pos + 2:pos + 2 + n].decode("utf-8", errors="replace")
        out[name], pos = _nbt_payload(buf, pos + 2 + n, tag)


# ------------------------------------------------------------------------------------------------------
# octree stream -> packed node array
# ------------------------------------------------------------------------------------------------------
def pack_preorder(stream: np.ndarray, start: int = 0) -> Tuple[np.ndarray, int]:
    """Pre-order node stream (-1 = branch) -> (packed tree with leaves as -type, index after the last node read)."""
    tree: List[int] = [0]
    todo = [0]                     # slots still to fill; children are pushed in reverse so child 0 is read first
    i = start
    n = stream.size
    while todo:
        if i >= n:
            raise ValueError("octree stream ends inside a node")
        slot = todo.pop()
        v = int(stream[i])
        i += 1
        if v == BRANCH:
            base = len(tree)
            tree.extend((0, 0, 0, 0, 0, 0, 0, 0))
            tree[slot] = base
            todo.extend((base + 7, base + 6, base + 5, base + 4, base + 3, base + 2, base + 1, base))
        else:
            tree[slot] = -v
    return np.asarray(tree, dtype=np.int64), i


def write_preorder(tree: np.ndarray) -> List[int]:
    """Inverse of pack_preorder for a packed tree whose leaves hold -type (used by the tests' fixture writer)."""
    out: List[int] = []
    todo = [0]
    while todo:
        at = todo.pop()
        w = int(tree[at])
        if w > 0:
            out.append(BRANCH)
            todo.extend(range(w + 7, w - 1, -1))
        else:
            out.append(-w)
    return out


# ------------------------------------------------------------------------------------------------------
# file
# ------------------------------------------------------------------------------------------------------
@dataclass
class Octree2:
    version: int
    palette_version: int
    blocks: List[Dict[str, object]]       # NBT of every palette entry ({"Name": ..., "Properties": {...}})
    world_depth: int
    world: np.ndarray                     # packed nodes, leaves = -(palette index), ANY_TYPE leaves = -0x7FFFFFFE
    water_depth: int
    water: np.ndarray
    biomes: Optional[Dict[str, Tuple[np.ndarray, np.ndarray]]] = None   # name -> (chunks int32[n, 2], rgb float32[n, 256, 3])

    def stats(self) -> Dict[str, int]:
        w = self.world
        leaves = w[w <= 0]
        return {"nodes": int(w.size), "branches": int((w > 0).sum()), "any_type_leaves": int((leaves == -ANY_TYPE).sum()),
                "leaf_types": int(np.unique(leaves).size), "depth": self.world_depth,
                "water_nodes": int(self.water.size), "water_depth": self.water_depth}


def _read_stream(path: str) -> bytes:
    raw = open(path, "rb").read()
    if raw[:2] == b"\x1f\x8b":
        return gzip.decompress(raw)
    try:
        return zlib.decompress(raw)
    except zlib.error:
        return raw


def load(path: str) -> Octree2:
    buf = _read_stream(path)
    version, palette_version, n_blocks = struct.unpack_from(">iii", buf, 0)
    if version < 5 or version > 6:
        raise ValueError(f"unsupported octree file version {version} (this loader reads the palette-based formats 5 and 6)")
    pos = 12
    blocks = []
    for _ in range(n_blocks):
        b, pos = _nbt_compound_body(buf, pos)
        blocks.append(b)
    # the node streams are 4-byte ints but start at an arbitrary byte offset
    world_depth = struct.unpack_from(">i", buf, pos)[0]
    stream = np.frombuffer(buf, dtype=">i4", offset=pos + 4, count=(len(buf) - pos - 4) // 4)
    world, used = pack_preorder(stream)
    pos2 = pos + 4 + 4 * used
    water_depth = struct.unpack_from(">i", buf, pos2)[0]
    stream2 = np.frombuffer(buf, dtype=">i4", offset=pos2 + 4, count=(len(buf) - pos2 - 4) // 4)
    water, used2 = pack_preorder(stream2)
    biomes = read_biomes(buf, pos2 + 4 + 4 * used2)
    return Octree2(version, palette_version, blocks, world_depth, world, water_depth, water, biomes)


BIOME_TEXTURES = ("grass", "foliage", "water")   # file order
_TILE_BYTES = 8 + 256 * 3 * 4


def read_biomes(buf: bytes, pos: int) -> Optional[Dict[str, Tuple[np.ndarray, np.ndarray]]]:
    """The biome colour section that starts at ``pos``: None when the stream ends there; ValueError when it is truncated."""
    if pos == len(buf):
        return None
    out = {}
    for name in BIOME_TEXTURES:
        if pos + 4 > len(buf):
            raise ValueError(f"biome section ends before the {name} texture")
        n = struct.unpack_from(">i", buf, pos)[0]
        pos += 4
        if n < 0 or pos + n * _TILE_BYTES > len(buf):
            raise ValueError(f"biome {name} texture: {n} tiles do not fit the {len(buf) - pos} bytes left")
        raw = np.frombuffer(buf, dtype=np.uint8, count=n * _TILE_BYTES, offset=pos).reshape(n, _TILE_BYTES)
        chunks = raw[:, :8].copy().view(">i4").astype(np.int32)
        rgb = raw[:, 8:].copy().view(">f4").astype(np.float32).reshape(n, 256, 3)
        out[name] = (chunks, rgb)
        pos += n * _TILE_BYTES
    return out


def write_biomes(biomes: Dict[str, Tuple[np.ndarray, np.ndarray]]) -> bytes:
    """The biome colour section of ``biomes`` (inverse of read_biomes)."""
    out = bytearray()
    for name in BIOME_TEXTURES:
        chunks, rgb = biomes[name]
        chunks = np.asarray(chunks, dtype=">i4").reshape(-1, 2)
        rgb = np.asarray(rgb, dtype=">f4").reshape(-1, 256 * 3)
        out += struct.pack(">i", chunks.shape[0])
        for c, t in zip(chunks, rgb):
            out += c.tobytes() + t.tobytes()
    return bytes(out)


def save(path: str, blocks: List[Dict[str, object]], world_depth: int, world: np.ndarray, water_depth: int = 0,
         water: np.ndarray = None, biomes: Optional[Dict[str, Tuple[np.ndarray, np.ndarray]]] = None) -> None:
    """Writes the subset of the format ``load`` reads (string-valued block NBT only, biome colours when given); for fixtures."""
    out = bytearray(struct.pack(">iii", 6, 4, len(blocks)))

    def put_str(s: str):
        b = s.encode()
        out.extend(struct.pack(">H", len(b)) + b)

    for blk in blocks:
        for k, v in blk.items():
            if isinstance(v, dict):
                out.append(10); put_str(k)
                for pk, pv in v.items():
                    out.append(8); put_str(pk); put_str(str(pv))
                out.append(0)
            else:
                out.append(8); put_str(k); put_str(str(v))
        out.append(0)
    for depth, tree in ((world_depth, world), (water_depth, np.zeros(1, np.int64) if water is None else water)):
        nodes = write_preorder(np.asarray(tree))
        out.extend(struct.pack(">i", depth))
        out.extend(np.asarray(nodes, dtype=">i4").tobytes())
    if biomes is not None:
        out.extend(write_biomes(biomes))
    with gzip.open(path, "wb") as f:
        f.write(bytes(out))


# ------------------------------------------------------------------------------------------------------
# scene
# ------------------------------------------------------------------------------------------------------
_INVISIBLE = {"minecraft:air", "minecraft:cave_air", "minecraft:void_air"}
_COLOURS = {
    "stone": (125, 125, 125), "dirt": (134, 96, 67), "grass_block": (100, 150, 70), "sand": (219, 207, 163), "water": (50, 90, 200),
    "bedrock": (60, 60, 60), "gravel": (130, 125, 120), "oak_log": (110, 85, 50), "oak_leaves": (60, 120, 40),
    "oak_planks": (160, 130, 80), "cobblestone": (120, 120, 120), "stone_bricks": (122, 122, 122), "glass": (200, 220, 230),
    "bricks": (150, 90, 75), "snow": (245, 250, 250), "glowstone": (250, 215, 120), "sea_lantern": (220, 235, 230),
    "white_concrete": (207, 213, 214), "gray_concrete": (55, 58, 62), "black_concrete": (8, 10, 15), "iron_block": (220, 220, 220),
    "quartz_block": (235, 230, 224), "smooth_stone": (160, 160, 160), "andesite": (135, 136, 136), "diorite": (190, 190, 192),
    "granite": (150, 105, 85), "lava": (210, 90, 20), "sandstone": (216, 203, 155), "terracotta": (152, 94, 68),
}
_EMITTERS = {"glowstone": 1.0, "sea_lantern": 1.0, "lava": 1.0, "torch": 0.9, "lantern": 0.9, "redstone_lamp": 0.0, "jack_o_lantern": 1.0,
             "shroomlight": 1.0, "beacon": 1.0, "end_rod": 0.9, "fire": 1.0, "magma_block": 0.6}


def block_colour(name: str) -> Tuple[int, int, int]:
    short = name.split(":", 1)[-1]
    if short in _COLOURS:
        return _COLOURS[short]
    for key, rgb in _COLOURS.items():
        if key in short:
            return rgb
    h = zlib.crc32(short.encode())
    return 64 + (h & 0x7F), 64 + ((h >> 8) & 0x7F), 64 + ((h >> 16) & 0x7F)


# Chunky's biome-tinted blocks (PackedMaterial.java:79 tint types): 1 foliage, 2 grass, 3 water
_TINT_TYPES = {"grass_block": 2, "grass": 2, "short_grass": 2, "tall_grass": 2, "fern": 2, "large_fern": 2, "sugar_cane": 2,
               "oak_leaves": 1, "jungle_leaves": 1, "acacia_leaves": 1, "dark_oak_leaves": 1, "mangrove_leaves": 1, "vine": 1,
               "water": 3}
_TINT_BASE = (200, 200, 200)   # the light grey a tinted block's texture has before its tint


_FIXED_TINTS = {"foliage": 0x71A74D, "grass": 0x8EB971, "water": 0x3F76E4}   # material.h:61-72, tint types 1, 2, 3


def biome_planes(biomes: Dict[str, Tuple[np.ndarray, np.ndarray]]) -> Tuple[np.ndarray, np.ndarray]:
    """The file's three textures as ccu_scene_set_biome_colors takes them: (chunks int32[n, 2], rgb float32[n, 3, 256, 3]) with
    the planes in tint-type order (foliage, grass, water), over every chunk any texture has (in file order: grass, foliage,
    water).  Chunky writes the textures independently; a chunk missing from one texture gets that plane filled with the fixed
    tint's own floats (byte / 256), which renders exactly as the fixed tint does (DESIGN.md section 13)."""
    order: Dict[Tuple[int, int], int] = {}
    for name in BIOME_TEXTURES:
        for x, z in biomes[name][0]:
            order.setdefault((int(x), int(z)), len(order))
    rgb = np.empty((len(order), 3, 256, 3), np.float32)
    for k, name in enumerate(("foliage", "grass", "water")):
        t = _FIXED_TINTS[name]
        rgb[:, k] = np.array([(t >> 16) & 0xFF, (t >> 8) & 0xFF, t & 0xFF], np.float32) / np.float32(256)
        c, tex = biomes[name]
        if c.shape[0]:
            rgb[[order[(int(x), int(z))] for x, z in c], k] = tex
    chunks = np.array(list(order), np.int32).reshape(-1, 2)
    return chunks, rgb


def to_scene(o: Octree2, width: int = 1920, height: int = 1080, camera=None, sun: bool = True,
             biome_tints: bool = False) -> S.PackedScene:
    """Packed scene in the reference's layouts: one full-cube block (type 1, block.h:48-65) with a flat-colour material
    (PackedMaterial.java:88-100, untextured) per palette entry; leaves remapped as ClSceneLoader.java:56-58 does.
    biome_tints: grass, foliage and water blocks get their tint type and a light-grey base colour, and the file's biome
    colours (if any) become the scene's (PackedScene.biome, for CCU_RENDER_BIOME_TINT)."""
    pal = S.Palettes()
    pal.blocks = [0, 0]                                   # pointer 0: invisible (block.h:39-41)
    mapping = np.zeros(len(o.blocks), dtype=np.int64)
    for i, blk in enumerate(o.blocks):
        name = str(blk.get("Name", "minecraft:air"))
        if name in _INVISIBLE:
            mapping[i] = 0
            continue
        r, g, b = block_colour(name)
        emit = next((e for k, e in _EMITTERS.items() if k in name), 0.0)
        tint = _TINT_TYPES.get(name.split(":", 1)[-1], 0) if biome_tints else 0
        if tint:
            r, g, b = _TINT_BASE
        ptr = pal.put_material(S.pack_material(0, 0, emittance=emit, tint=tint << 24, textured=False,
                                               argb=(0xFF << 24) | (r << 16) | (g << 8) | b))
        mapping[i] = len(pal.blocks)
        pal.blocks += [1, ptr]
    tree = o.world.copy()
    leaf = tree <= 0
    types = -tree[leaf]
    in_range = types < len(mapping)
    remapped = types.copy()
    remapped[in_range] = mapping[types[in_range]]          # out-of-range types (ANY_TYPE) stay verbatim
    tree[leaf] = -remapped
    edge = 1 << o.world_depth
    if camera is None:
        camera = S.pinhole_camera((edge / 2 + 0.37, edge * 0.55 + 0.21, edge / 8 + 0.11), 0.0, -35.0, 70.0)
    p = S._finish("octree2", tree.astype(np.int32), o.world_depth, pal, camera, width, height, sun_draw=sun,
                  meta={"blocks": len(o.blocks), **o.stats()})
    if biome_tints and o.biomes is not None:
        p.biome = biome_planes(o.biomes)
    return p


def scene_origin(d: dict) -> Tuple[int, int, int]:
    """The world position of the octree origin in a parsed Chunky scene description: the low corner of the loaded chunk
    rectangle in x and z, yMin in y (see camera_from_json).  The plugin's frame is world minus this."""
    chunks = np.asarray(d["chunkList"], dtype=np.int64)
    return int(chunks[:, 0].min()) * 16, int(d.get("yMin", 0)), int(chunks[:, 1].min()) * 16


def camera_from_json(json_path: str) -> np.ndarray:
    """float[15] camera settings (ClCamera.java:39-52) from a Chunky scene description.

    The octree origin is the corner of the loaded chunk rectangle (Chunky places the chunks at the low corner of the cube:
    checked against the benchmark scene, whose non-air leaves span exactly [0, 16*chunks) in x and z).  chunky-core's
    ``Camera.transform`` is not available here, so the orientation is an approximation (Chunky's pitch -90 deg = horizon,
    0 = straight down); it places the reference's benchmark camera at street level inside the city, which is all the
    traversal statistics need."""
    import json
    import math
    d = json.loads(open(json_path, "rb").read().decode("latin-1"))
    ox, oy, oz = scene_origin(d)
    cam = d["camera"]
    pos = (cam["position"]["x"] - ox, cam["position"]["y"] - oy, cam["position"]["z"] - oz)
    yaw, pitch = cam["orientation"]["yaw"], cam["orientation"]["pitch"]
    return S.pinhole_camera(pos, 270.0 + math.degrees(yaw), -(90.0 + math.degrees(pitch)), float(cam.get("fov", 70.0)))


# Chunky's extinction per block for a fog density of 1 (Fog.EXTINCTION_FACTOR).  chunky-core is not available here, so the value
# is unverified: 0.04 is what it is believed to be.
FOG_EXTINCTION_FACTOR = 0.04


def fog_from_json(json_path: str) -> Tuple[float, float, Tuple[float, float, float], bool]:
    """The fog of a Chunky scene description as ccu_scene_set_fog takes it (DESIGN.md §14): (sigma, sky density, linear RGB
    colour, fast).  sigma = fogDensity * FOG_EXTINCTION_FACTOR, the only place that converts Chunky's density; a density of 0
    gives sigma = 0, no fog.  fogColor is taken as linear RGB, and a missing key takes a default (fogDensity 0, skyFogDensity 1,
    a white fogColor, fastFog true); like the extinction factor, neither is checked against chunky-core, which is not
    available here."""
    import json
    d = json.loads(open(json_path, "rb").read().decode("latin-1"))
    c = d.get("fogColor", {"red": 1.0, "green": 1.0, "blue": 1.0})
    color = (float(c["red"]), float(c["green"]), float(c["blue"]))
    return (float(d.get("fogDensity", 0.0)) * FOG_EXTINCTION_FACTOR, float(d.get("skyFogDensity", 1.0)), color,
            bool(d.get("fastFog", True)))


# The cloud layer's thickness in blocks.  chunky-core is not available here, so the value is unverified: Minecraft's fancy clouds
# are 4 blocks thick, and that is what Chunky's layer is believed to be.
CLOUD_THICKNESS = 4.0
# How cloudOffset x / z move the cells: +1 = the mask cell of world point (x, z) is floor((x + offset.x) / cloudSize),
# floor((z + offset.z) / cloudSize), and the layer starts at y = offset.y.  Like the thickness it is not checked against
# chunky-core.
CLOUD_OFFSET_SIGN = 1.0


def clouds_from_json(json_path: str, mask) -> Optional[Tuple[np.ndarray, float, float, float, float, float]]:
    """The cloud layer of a Chunky scene description as ccu_scene_set_clouds takes it (DESIGN.md §15): (mask, size, y0, y1, u0, v0)
    in the plugin's frame (world minus the scene origin of camera_from_json), or None when sky.cloudsEnabled is false or missing.
    `mask` is Minecraft's cloud texture as uint8[256, 256] indexed [k, i] (non-zero = cloud): it is not part of the scene
    description.  The layer spans CLOUD_THICKNESS blocks from cloudOffset.y; cloudOffset x / z shift the cells by
    CLOUD_OFFSET_SIGN."""
    import json
    d = json.loads(open(json_path, "rb").read().decode("latin-1"))
    sky = d.get("sky", {})
    if not sky.get("cloudsEnabled", False):
        return None
    m = np.ascontiguousarray(mask, np.uint8)
    if m.shape != (256, 256):
        raise ValueError("the cloud mask needs 256 x 256 cells")
    ox, oy, oz = scene_origin(d)
    size = float(sky.get("cloudSize", 64.0))
    off = sky.get("cloudOffset", {})
    y0 = float(off.get("y", 128.0)) - oy
    u0 = (ox + CLOUD_OFFSET_SIGN * float(off.get("x", 0.0))) / size
    v0 = (oz + CLOUD_OFFSET_SIGN * float(off.get("z", 0.0))) / size
    return m, size, y0, y0 + CLOUD_THICKNESS, u0, v0


def load_scene(octree_path: str, json_path: str = None, width: int = 1920, height: int = 1080,
               cloud_mask=None) -> S.PackedScene:
    """The scene of an .octree2 file, with the camera and fog of a Chunky scene description when one is given, and its clouds
    when a cloud mask is given too (clouds_from_json)."""
    o = load(octree_path)
    p = to_scene(o, width, height, camera=camera_from_json(json_path) if json_path else None)
    if json_path:
        p.fog = fog_from_json(json_path)
        if cloud_mask is not None:
            p.clouds = clouds_from_json(json_path, cloud_mask)
    return p
