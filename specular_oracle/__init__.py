"""ctypes binding of the CPU restatement of CCU_RENDER_SPECULAR, CCU_RENDER_EMITTER_SAMPLING, CCU_RENDER_EMITTER_NEAR_FIELD,
CCU_RENDER_EMITTER_MODELS, CCU_RENDER_BIOME_TINT, CCU_RENDER_FOG and CCU_RENDER_CLOUDS (specular_oracle.c).  TEST INFRASTRUCTURE
ONLY.

``SpecularOracle`` is the parity oracle (``oracle.Oracle``) with the specular events of DESIGN.md section 9 in its path
loop; ``FlagsOracle`` takes the render flags and adds the emitter sampling of sections 10 to 12, with the emitter table that
``emitter_grid`` builds from the packed arrays (``model_emitters`` adds the model emitters of section 12), and its ``features``
restates the denoiser's feature buffers of section 16; ``denoise`` restates the denoiser of section 17.  Everything else - first hit, preview, counters - is the oracle's.  Like the
oracle, only tests/ and scripts use it.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess
from typing import Optional, Sequence

import numpy as np

import oracle

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB_PATH = os.path.join(_HERE, "_build", "libspecular_oracle.so")
_SOURCES = (os.path.join(_HERE, "specular_oracle.c"), os.path.join(os.path.dirname(_HERE), "oracle", "chunky_oracle.c"))
_lib = None


def build(force: bool = False) -> str:
    if force or not os.path.exists(_LIB_PATH) or any(os.path.getmtime(_LIB_PATH) < os.path.getmtime(s) for s in _SOURCES):
        subprocess.run(["make", "-C", _HERE, "CC=gcc"], check=True, capture_output=True)
    return _LIB_PATH


def lib():
    global _lib
    if _lib is None:
        build()
        _lib = C.CDLL(_LIB_PATH)
        assert _lib.oracle_scene_struct_size() == C.sizeof(oracle._Scene), "OracleScene layout mismatch"
        assert _lib.emitter_grid_struct_size() == C.sizeof(_Grid), "EmitterGrid layout mismatch"
        assert _lib.biome_tiles_struct_size() == C.sizeof(_Biome), "BiomeTiles layout mismatch"
        assert _lib.fog_params_struct_size() == C.sizeof(_Fog), "FogParams layout mismatch"
        assert _lib.cloud_layer_struct_size() == C.sizeof(_Clouds), "CloudLayer layout mismatch"
        _lib.fog_expf_test.restype = C.c_float
        _lib.fog_expf_test.argtypes = [C.c_float]
    return _lib


class _Grid(C.Structure):
    _fields_ = [("emit", C.c_void_p), ("off", C.c_void_p), ("list", C.c_void_p),
                ("g0", C.c_int32 * 3), ("dim", C.c_int32 * 3), ("shift", C.c_int32), ("mhead", C.c_void_p), ("mprim", C.c_void_p)]


class _Fog(C.Structure):
    _fields_ = [("sigma", C.c_float), ("sky", C.c_float), ("color", C.c_float * 3), ("fast", C.c_int32)]


class _Clouds(C.Structure):
    _fields_ = [("bits", C.c_void_p), ("inv", C.c_float), ("y0", C.c_float), ("y1", C.c_float), ("u0", C.c_float),
                ("v0", C.c_float)]


def cloud_bits(mask) -> np.ndarray:
    """The mask uint8[256, 256] (indexed [k, i]) bit-packed as the library holds it: uint32[2048], cell (i, k) at bit
    (k & 255) * 256 + (i & 255)."""
    m = np.ascontiguousarray(mask, np.uint8).reshape(-1) != 0
    return np.packbits(m, bitorder="little").view("<u4").astype(np.uint32)


def _cloud_layer(clouds, keep: dict) -> "_Clouds":
    mask, size, y0, y1, u0, v0 = clouds
    bits = cloud_bits(mask)
    keep["cloud_bits"] = bits
    inv = np.float32(1.0) / np.float32(size)    # ccu_scene_set_clouds: 1.0f / size
    return _Clouds(bits.ctypes.data, float(inv), float(np.float32(y0)), float(np.float32(y1)), float(np.float32(u0)),
                   float(np.float32(v0)))


def cloud_hit(clouds, o, d, limit=None):
    """DESIGN.md section 15.2 for N rays (o, d float32[N, 3], limit float32[N], default unbounded) against the cloud layer
    clouds = (mask, size, y0, y1, u0, v0): (t float32[N], NaN for a miss; normal float32[N, 3]; cells the walk tested int32[N])."""
    keep = {}
    cl = _cloud_layer(clouds, keep)
    o = np.ascontiguousarray(o, np.float32).reshape(-1, 3)
    d = np.ascontiguousarray(d, np.float32).reshape(-1, 3)
    n = o.shape[0]
    lim = np.full(n, np.inf, np.float32) if limit is None else np.ascontiguousarray(np.broadcast_to(limit, (n,)), np.float32)
    out = np.zeros((n, 4), np.float32)
    visited = np.zeros(n, np.int32)
    lib().cloud_hit_batch(C.byref(cl), C.c_int64(n), o.ctypes.data_as(C.c_void_p), d.ctypes.data_as(C.c_void_p),
                          lim.ctypes.data_as(C.c_void_p), out.ctypes.data_as(C.c_void_p), visited.ctypes.data_as(C.c_void_p))
    return out[:, 0], out[:, 1:], visited


def dm_expf(x: float) -> float:
    """The fog's transmittance kernel (DESIGN.md section 14), as the restatement and the kernels evaluate it."""
    return float(np.float32(lib().fog_expf_test(float(x))))


def denoise(color, albedo, normal, iterations: int, sigma_l: float, width: Optional[int] = None,
            height: Optional[int] = None) -> np.ndarray:
    """DESIGN.md section 17: the guided a-trous filter of a sample buffer, as the restatement evaluates it.  color: float64
    (H, W, 3) or flat with width and height given; albedo, normal: float32 of the same layout.  Returns float64[3*W*H]."""
    c = np.ascontiguousarray(color, np.float64)
    if width is None or height is None:
        height, width = c.shape[0], c.shape[1]
    c = c.reshape(-1)
    a = np.ascontiguousarray(albedo, np.float32).reshape(-1)
    nrm = np.ascontiguousarray(normal, np.float32).reshape(-1)
    assert c.size == a.size == nrm.size == 3 * width * height
    out = np.empty_like(c)
    rc = lib().denoise(C.c_int32(width), C.c_int32(height), c.ctypes.data_as(C.c_void_p), a.ctypes.data_as(C.c_void_p),
                       nrm.ctypes.data_as(C.c_void_p), C.c_int32(iterations), C.c_float(sigma_l), out.ctypes.data_as(C.c_void_p))
    if rc != 0:
        raise MemoryError("specular_oracle.denoise: out of memory")
    return out


class _Biome(C.Structure):
    _fields_ = [("grid", C.c_void_p), ("tiles", C.c_void_p), ("x0", C.c_int32), ("z0", C.c_int32), ("gx", C.c_int32),
                ("gz", C.c_int32)]


CCU_RENDER_SPECULAR, CCU_RENDER_EMITTER_SAMPLING, CCU_RENDER_EMITTER_NEAR_FIELD, CCU_RENDER_EMITTER_MODELS = 4, 8, 128, 256
CCU_RENDER_BIOME_TINT = 512
CCU_RENDER_FOG = 1024
CCU_RENDER_CLOUDS = 2048
EMIT_SHIFT0, EMIT_CELL_BUDGET, EMIT_MAX = 3, 1 << 21, 1 << 18      # DESIGN.md section 10


def _leaves(tree: np.ndarray, depth: int):
    """Every leaf of the reference's node array: (x, y, z) of its low corner, level and value (-word), breadth first."""
    tree = np.asarray(tree, np.int64)
    node = np.zeros(1, np.int64)
    xyz = np.zeros((1, 3), np.int64)
    out = []
    for level in range(depth, -1, -1):
        data = tree[node]
        leaf = data <= 0
        out.append((xyz[leaf] << level, np.full(int(leaf.sum()), level), -data[leaf]))
        inner = ~leaf
        if level == 0 or not inner.any():
            break
        k = np.arange(8)
        node = (data[inner][:, None] + k[None, :]).reshape(-1)
        child = np.stack([k >> 2, (k >> 1) & 1, k & 1], axis=1)
        xyz = ((xyz[inner][:, None, :] << 1) | child[None, :, :]).reshape(-1, 3)
    return (np.concatenate([o[0] for o in out]), np.concatenate([o[1] for o in out]), np.concatenate([o[2] for o in out]))


def emitter_blocks(block_palette: np.ndarray, mat_palette: np.ndarray) -> np.ndarray:
    """bool per block palette position: a full cube (type 1) whose material has textured emittance or an emittance byte."""
    bp = np.asarray(block_palette, np.int64)
    mp = np.asarray(mat_palette, np.int64)
    out = np.zeros(max(bp.size - 1, 0), bool)
    for b in range(out.size):
        ptr = bp[b + 1]
        if bp[b] == 1 and 0 <= ptr and ptr + 5 < mp.size:
            out[b] = bool((mp[ptr] & 2) or (mp[ptr + 4] & 0xFF))
    return out


def _f32(words) -> np.ndarray:
    return np.asarray(words, np.int32).view(np.float32)


def _material_emits(mp: np.ndarray, ptr: int) -> bool:
    return 0 <= ptr and ptr + 5 < mp.size and bool((mp[ptr] & 2) or (mp[ptr + 4] & 0xFF))


def model_emitters(p):
    """DESIGN.md section 12: (head, prim) of the model emitters, as native.debug_emitter_models returns them.  head[b] is the
    int4 index in prim of palette position b's emitting primitives, -1 for no model emitter; prim holds per model emitter the
    header {m, bounding box (float32 bits: xmin, xmax, ymin, ymax, zmin, zmax), 0} and m records of 16 words {kind, material,
    face flags, 13 words}: kind 6 a quad and its 13 words, kind axis * 2 + (1 for +) a box face and the box's 6 words."""
    bp = np.asarray(p.block_palette, np.int64)
    mp = np.asarray(p.mat_palette, np.int64)
    quads, aabbs = np.asarray(p.quad_models, np.int32), np.asarray(p.aabb_models, np.int32)
    n_pos = max(bp.size - 1, 1)
    head = np.full(n_pos, -1, np.int32)
    prim = []
    for b in range(bp.size - 1):
        typ, ptr = int(bp[b]), int(bp[b + 1])
        if typ not in (2, 3):
            continue
        src, words = (aabbs, 13) if typ == 2 else (quads, 15)
        if ptr < 0 or ptr >= src.size or src[ptr] < 0 or ptr + 1 + int(src[ptr]) * words > src.size:
            continue
        recs, pts = [], []
        for i in range(int(src[ptr])):
            w = src[ptr + 1 + i * words:ptr + 1 + (i + 1) * words]
            if typ == 3:
                if not _material_emits(mp, int(w[13])):
                    continue
                recs.append([6, int(w[13]), 0] + [int(v) for v in w[:13]])
                o, x, y = _f32(w[0:3]), _f32(w[3:6]), _f32(w[6:9])
                pts += [o, o + x, o + y, (o + x) + y]
                continue
            box = _f32(w[0:6])
            for f, (mat, sh) in enumerate(((w[10], 12), (w[8], 4), (w[12], 20), (w[11], 16), (w[9], 8), (0, None))):
                fl = 0 if sh is None else (int(w[6]) >> sh) & 15
                if fl & 8 or not _material_emits(mp, int(mat)):
                    continue
                recs.append([f, int(mat), fl] + [int(v) for v in w[:6]] + [0] * 7)
                axis = f >> 1
                lo, hi = box[0::2].copy(), box[1::2].copy()
                lo[axis] = hi[axis] = box[2 * axis + (f & 1)]
                pts += [lo, hi]
        if not recs:
            continue
        pts = np.stack(pts).astype(np.float32)
        bb = np.stack([pts.min(0), pts.max(0)], 1).reshape(-1).astype(np.float32).view(np.int32)
        head[b] = sum(len(r) for r in prim) // 4
        prim.append([len(recs)] + [int(v) for v in bb] + [0])
        prim += recs
    return head, np.array([v for r in prim for v in r], np.int32)


def emitter_grid(p, models: bool = False) -> dict:
    """The emitter table and cell lists of DESIGN.md section 10 for a packed scene (same keys as native.debug_emitter_grid).
    models: the wider table of section 12, with "head" / "prim" (model_emitters); it is empty unless it holds a model emitter."""
    empty = {"has_emitters": False, "g0": np.zeros(3, np.int32), "dim": np.zeros(3, np.int32), "shift": EMIT_SHIFT0,
             "emit": np.zeros((0, 4), np.int32), "off": np.zeros(0, np.int32), "list": np.zeros(0, np.int32)}
    emits = emitter_blocks(p.block_palette, p.mat_palette)
    if models:
        head, prim = model_emitters(p)
        empty.update(head=np.zeros(0, np.int32), prim=np.zeros(0, np.int32))
        emits = emits | (head[:emits.size] >= 0)
        if not (head >= 0).any():
            return empty
    corner, level, value = _leaves(p.octree, p.octree_depth)
    sel = (value >= 0) & (value < emits.size)
    sel[sel] = emits[value[sel]]
    corner, level, value = corner[sel], level[sel], value[sel]
    if corner.shape[0] == 0 or level.max() > 6 or int((8 ** level).sum()) > EMIT_MAX:
        return empty
    parts = []
    for c, l, v in zip(corner, level, value):
        s = 1 << int(l)
        g = np.stack(np.meshgrid(np.arange(s), np.arange(s), np.arange(s), indexing="ij"), -1).reshape(-1, 3) + c
        parts.append(np.concatenate([g, np.full((g.shape[0], 1), v)], axis=1))
    e = np.concatenate(parts)
    e = e[np.lexsort((e[:, 2], e[:, 1], e[:, 0]))]
    lo, hi = e[:, :3].min(0), e[:, :3].max(0)
    shift = EMIT_SHIFT0
    while True:
        c0, c1 = (lo >> shift) - 1, (hi >> shift) + 1
        dim = c1 - c0 + 1
        if int(np.prod(dim)) <= EMIT_CELL_BUDGET:
            break
        shift += 1
    g0 = c0 << shift
    cell = (e[:, :3] - g0) >> shift
    d = np.stack(np.meshgrid([-1, 0, 1], [-1, 0, 1], [-1, 0, 1], indexing="ij"), -1).reshape(-1, 3)
    nb = cell[:, None, :] + d[None, :, :]
    lin = ((nb[..., 0] * dim[1] + nb[..., 1]) * dim[2] + nb[..., 2]).reshape(-1)
    idx = np.repeat(np.arange(e.shape[0]), 27)
    order = np.lexsort((idx, lin))
    off = np.zeros(int(np.prod(dim)) + 1, np.int64)
    np.add.at(off, lin + 1, 1)
    out = {"has_emitters": True, "g0": g0.astype(np.int32), "dim": dim.astype(np.int32), "shift": shift,
           "emit": e.astype(np.int32), "off": np.cumsum(off).astype(np.int32), "list": idx[order].astype(np.int32)}
    if models:
        if not (head[e[:, 3]] >= 0).any():
            return empty
        out.update(head=head, prim=prim)
    return out


BIOME_GRID_MAX = 1 << 24    # DESIGN.md section 13: cells of the chunk grid


def biome_layout(chunks, rgb, depth: int) -> dict:
    """DESIGN.md section 13: the biome layout commit builds (as native.debug_biome_layout returns it): x0, z0 the low chunk of
    the chunks' bounding box, grid int32[gx, gz] indexed [cx - x0, cz - z0] holding the chunk's tile or -1, tiles
    float32[n, 3, 256, 4] with w = 0.  Raises ValueError for a chunk outside the octree's max(1, 2^depth / 16) chunks per axis,
    or a bounding box of more than BIOME_GRID_MAX chunks."""
    chunks = np.asarray(chunks, np.int64).reshape(-1, 2)
    rgb = np.asarray(rgb, np.float32).reshape(-1, 3, 256, 3)
    extent = 1 << max(depth - 4, 0)
    if chunks.size and (chunks.min() < 0 or chunks.max() >= extent):
        raise ValueError(f"a chunk lies outside the octree's {extent} x {extent} chunks")
    lo = chunks.min(0) if chunks.size else np.zeros(2, np.int64)
    dim = chunks.max(0) - lo + 1 if chunks.size else np.zeros(2, np.int64)
    if int(dim[0]) * int(dim[1]) > BIOME_GRID_MAX:
        raise ValueError(f"the chunks span more than {BIOME_GRID_MAX} chunks")
    grid = np.full((int(dim[0]), int(dim[1])), -1, np.int32)
    grid[chunks[:, 0] - lo[0], chunks[:, 1] - lo[1]] = np.arange(chunks.shape[0], dtype=np.int32)
    tiles = np.zeros((chunks.shape[0], 3, 256, 4), np.float32)
    tiles[..., :3] = rgb
    return {"x0": int(lo[0]), "z0": int(lo[1]), "grid": grid, "tiles": tiles}


class SpecularOracle(oracle.Oracle):
    """oracle.Oracle whose render() runs the path loop with CCU_RENDER_SPECULAR on."""

    def render(self, seeds: Sequence[int], start_spp: int = 0, res: Optional[np.ndarray] = None,
               gids: Optional[np.ndarray] = None, threads: int = 0) -> np.ndarray:
        n = self._s.width * self._s.height
        if res is None:
            res = np.zeros(n * 3, dtype=np.float32)
        assert res.dtype == np.float32 and res.size == n * 3 and res.flags.c_contiguous
        sd = np.ascontiguousarray(seeds, dtype=np.int32)
        cnt = oracle._Counters()
        gp, gn = None, 0
        if gids is not None:
            g = np.ascontiguousarray(gids, dtype=np.int32)
            gp, gn = g.ctypes.data_as(C.c_void_p), g.size
        lib().specular_render(C.byref(self._s), sd.ctypes.data_as(C.c_void_p), C.c_int(sd.size), C.c_int(start_spp),
                              res.ctypes.data_as(C.c_void_p), gp, C.c_int64(gn), C.c_int(threads), C.byref(cnt))
        self._counters(cnt)
        return res


class FlagsOracle(oracle.Oracle):
    """oracle.Oracle whose render() runs the path loop with the given CCU_RENDER_SPECULAR / CCU_RENDER_EMITTER_SAMPLING /
    CCU_RENDER_EMITTER_NEAR_FIELD / CCU_RENDER_EMITTER_MODELS / CCU_RENDER_BIOME_TINT bits (the other flags act on the scene:
    oracle.edge_rays.without_sun, or empty BVHs for CCU_RENDER_NO_ENTITIES).  With CCU_RENDER_EMITTER_MODELS the wider table
    of section 12 is sampled when the scene has one, else the table of section 10.  With CCU_RENDER_BIOME_TINT the biome
    colours are `biome` = (chunks, rgb) as ccu_scene_set_biome_colors takes them, by default the scene's own (scene.biome).
    With CCU_RENDER_FOG the fog of section 14 is `fog` = (sigma, sky density, colour, fast) as ccu_scene_set_fog takes it,
    by default the scene's own (scene.fog); sigma = 0 is no fog.  With CCU_RENDER_CLOUDS the cloud layer of section 15 is `clouds`
    = (mask, size, y0, y1, u0, v0) as ccu_scene_set_clouds takes it, by default the scene's own (scene.clouds); a mask without a
    set cell is no cloud layer."""

    def __init__(self, scene, flags: int = 0, biome=None, fog=None, clouds=None, **kw):
        super().__init__(scene, **kw)
        self.flags = flags
        if clouds is None:
            clouds = getattr(scene, "clouds", None)
        self._clouds = None
        if flags & CCU_RENDER_CLOUDS and clouds is not None and np.asarray(clouds[0]).any():
            self._clouds = _cloud_layer(clouds, self._keep)
        if fog is None:
            fog = getattr(scene, "fog", None)
        self._fog = None
        if flags & CCU_RENDER_FOG and fog is not None and fog[0] > 0:
            self._fog = _Fog(fog[0], fog[1], (C.c_float * 3)(*fog[2]), int(fog[3]))
        if biome is None:
            biome = getattr(scene, "biome", None)
        self._biome = None
        if flags & CCU_RENDER_BIOME_TINT and biome is not None and np.asarray(biome[0]).size > 0:
            b = biome_layout(biome[0], biome[1], scene.octree_depth)
            grid, tiles = b["grid"], b["tiles"]
            self._keep["biome_grid"], self._keep["biome_tiles"] = grid, tiles
            self._biome = _Biome(grid.ctypes.data, tiles.ctypes.data, b["x0"], b["z0"], grid.shape[0], grid.shape[1])
        self.grid = emitter_grid(scene, models=True) if flags & CCU_RENDER_EMITTER_MODELS else None
        if not (self.grid and self.grid["has_emitters"]):
            self.grid = emitter_grid(scene)
        g = _Grid()
        for k in ("emit", "off", "list", "head", "prim"):
            if k not in self.grid:
                continue
            a = np.ascontiguousarray(self.grid[k], dtype=np.int32)
            self._keep["grid_" + k] = a
            setattr(g, {"head": "mhead", "prim": "mprim"}.get(k, k), a.ctypes.data)
        g.g0[:] = [int(v) for v in self.grid["g0"]]
        g.dim[:] = [int(v) for v in self.grid["dim"]]
        g.shift = self.grid["shift"]
        self._grid = g

    def render(self, seeds: Sequence[int], start_spp: int = 0, res: Optional[np.ndarray] = None,
               gids: Optional[np.ndarray] = None, threads: int = 0) -> np.ndarray:
        n = self._s.width * self._s.height
        if res is None:
            res = np.zeros(n * 3, dtype=np.float32)
        assert res.dtype == np.float32 and res.size == n * 3 and res.flags.c_contiguous
        sd = np.ascontiguousarray(seeds, dtype=np.int32)
        cnt = oracle._Counters()
        gp, gn = None, 0
        if gids is not None:
            g = np.ascontiguousarray(gids, dtype=np.int32)
            gp, gn = g.ctypes.data_as(C.c_void_p), g.size
        nee = (self.flags & CCU_RENDER_EMITTER_SAMPLING) and self.grid["has_emitters"]
        lib().flags_render(C.byref(self._s), sd.ctypes.data_as(C.c_void_p), C.c_int(sd.size), C.c_int(start_spp),
                           res.ctypes.data_as(C.c_void_p), gp, C.c_int64(gn), C.c_int(threads), C.byref(cnt),
                           C.c_int(1 if self.flags & CCU_RENDER_SPECULAR else 0), C.byref(self._grid) if nee else None,
                           C.c_int(1 if self.flags & CCU_RENDER_EMITTER_NEAR_FIELD else 0),
                           C.byref(self._biome) if self._biome is not None else None,
                           C.byref(self._fog) if self._fog is not None else None,
                           C.byref(self._clouds) if self._clouds is not None else None)
        self._counters(cnt)
        return res

    def features(self, seeds: Sequence[int], rays: Optional[np.ndarray] = None, threads: int = 0):
        """DESIGN.md section 16: the feature buffers (albedo, normal), float32[H*W*3] each, of the passes with these seeds under
        this oracle's flags: of them only CCU_RENDER_BIOME_TINT and CCU_RENDER_CLOUDS act (with the scene's biome colours and
        cloud layer); CCU_RENDER_NO_ENTITIES acts on the scene (empty BVHs).  rays: pre-generated camera rays (float32[H*W*6])
        in place of the scene's camera, as ccu_camera_set with projector -1 takes them."""
        n = self._s.width * self._s.height
        s = self._s
        keep = None
        if rays is not None:
            keep = np.ascontiguousarray(rays, np.float32).reshape(-1)
            assert keep.size == n * 6
            s = oracle._Scene.from_buffer_copy(self._s)
            s.projector_type = -1
            s.camera = keep.ctypes.data
        sd = np.ascontiguousarray(seeds, dtype=np.int32)
        albedo = np.zeros(n * 3, np.float32)
        normal = np.zeros(n * 3, np.float32)
        lib().features_render(C.byref(s), sd.ctypes.data_as(C.c_void_p), C.c_int(sd.size), albedo.ctypes.data_as(C.c_void_p),
                              normal.ctypes.data_as(C.c_void_p), C.byref(self._biome) if self._biome is not None else None,
                              C.byref(self._clouds) if self._clouds is not None else None, C.c_int(threads))
        return albedo, normal
