"""ctypes binding of libchunkycu.so (include/chunkycu.h) - the same symbols a JNI/FFM shim binds.

There is no fallback: if the library is missing or no B200 is present the calls raise.
"""
from __future__ import annotations

import ctypes as C
import os
from typing import Optional

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
# CHUNKYCU_LIB: load another build of the same library (kernel tuning sweeps build variants next to each other)
LIB_PATH = os.environ.get("CHUNKYCU_LIB") or os.path.join(_HERE, "libchunkycu.so")

CCU_RENDER_NO_ENTITIES, CCU_RENDER_NO_SUN, CCU_RENDER_SPECULAR, CCU_RENDER_EMITTER_SAMPLING = 1, 2, 4, 8
CCU_RENDER_EMITTER_NEAR_FIELD = 128
CCU_RENDER_EMITTER_MODELS = 256
CCU_RENDER_BIOME_TINT = 512
CCU_RENDER_FOG = 1024
CCU_RENDER_CLOUDS = 2048
CCU_UNIQUE_ID_BYTES = 128

CCU_OK, CCU_ENODEVICE, CCU_EINVAL, CCU_ECUDA, CCU_ENOMEM, CCU_ESTATE = 0, -1, -2, -3, -4, -5


class ChunkyCuError(RuntimeError):
    """Non-zero status from the C ABI (the Java shim throws RuntimeException, as JOCL's CLException did)."""

    def __init__(self, code: int, message: str):
        super().__init__(f"[{code}] {message}")
        self.code = code


class RenderParams(C.Structure):
    _fields_ = [("draw_depth", C.c_int32), ("max_depth", C.c_int32), ("emitter_scale", C.c_float), ("kernel", C.c_int32), ("flags", C.c_int32)]


# every symbol include/chunkycu.h declares: name -> (restype, argtypes)
_vp, _i32, _i64, _f = C.c_void_p, C.c_int32, C.c_int64, C.c_float
_pi32 = C.POINTER(C.c_int32)
SYMBOLS = {
    "ccu_device_count": (C.c_int, [C.POINTER(C.c_int)]),
    "ccu_device_info": (C.c_int, [C.c_int, C.c_char_p, C.c_int, C.POINTER(C.c_int), C.POINTER(C.c_int), C.POINTER(C.c_uint64)]),
    "ccu_ctx_create": (C.c_int, [C.c_int, C.POINTER(_vp)]),
    "ccu_ctx_destroy": (C.c_int, [_vp]),
    "ccu_last_error": (C.c_char_p, []),
    "ccu_version": (C.c_char_p, []),
    "ccu_scene_begin": (C.c_int, [_vp]),
    "ccu_scene_set_octree": (C.c_int, [_vp, _vp, _i64, _i32]),
    "ccu_scene_set_block_palette": (C.c_int, [_vp, _vp, _i64]),
    "ccu_scene_set_quad_models": (C.c_int, [_vp, _vp, _i64]),
    "ccu_scene_set_aabb_models": (C.c_int, [_vp, _vp, _i64]),
    "ccu_scene_set_material_palette": (C.c_int, [_vp, _vp, _i64]),
    "ccu_scene_set_triangles": (C.c_int, [_vp, _vp, _i64]),
    "ccu_scene_set_world_bvh": (C.c_int, [_vp, _vp, _i64]),
    "ccu_scene_set_actor_bvh": (C.c_int, [_vp, _vp, _i64]),
    "ccu_scene_set_biome_colors": (C.c_int, [_vp, _vp, _vp, _i64]),
    "ccu_scene_set_fog": (C.c_int, [_vp, _f, _f, _vp, _i32]),
    "ccu_scene_set_clouds": (C.c_int, [_vp, _vp, _f, _f, _f, _f, _f]),
    "ccu_scene_atlas_create": (C.c_int, [_vp, _i32, _i32, _i32]),
    "ccu_scene_atlas_write": (C.c_int, [_vp, _i32, _i32, _i32, _i32, _i32, _vp]),
    "ccu_scene_set_atlas": (C.c_int, [_vp, _vp, _i32, _i32, _i32]),
    "ccu_scene_set_sky": (C.c_int, [_vp, _vp, _i32, _f]),
    "ccu_scene_set_sun": (C.c_int, [_vp, _vp]),
    "ccu_scene_commit": (C.c_int, [_vp]),
    "ccu_camera_set": (C.c_int, [_vp, _i32, _vp, _i64]),
    "ccu_render_begin": (C.c_int, [_vp, _i32, _i32]),
    "ccu_render_set_params": (C.c_int, [_vp, C.POINTER(RenderParams)]),
    "ccu_render_passes": (C.c_int, [_vp, _vp, _i32]),
    "ccu_render_passes_async": (C.c_int, [_vp, _vp, _i32]),
    "ccu_render_sync": (C.c_int, [_vp]),
    "ccu_render_read": (C.c_int, [_vp, _vp, _pi32]),
    "ccu_render_merge": (C.c_int, [_vp, _vp, _i32, _pi32]),
    "ccu_render_merge_async": (C.c_int, [_vp, _vp, _i32, _pi32]),
    "ccu_render_merge_wait": (C.c_int, [_vp]),
    "ccu_render_window_close": (C.c_int, [_vp, _pi32]),
    "ccu_render_window_merge": (C.c_int, [_vp, _vp, _i32]),
    "ccu_render_reset_window": (C.c_int, [_vp]),
    "ccu_render_set_window_spp": (C.c_int, [_vp, _i32]),
    "ccu_render_end": (C.c_int, [_vp]),
    "ccu_render_device_buffer": (C.c_int, [_vp, C.POINTER(_vp), C.POINTER(_i64)]),
    "ccu_render_scale": (C.c_int, [_vp, _f]),
    "ccu_stream_handle": (C.c_int, [_vp, C.POINTER(_vp)]),
    "ccu_first_hit": (C.c_int, [_vp, _i32, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "ccu_preview": (C.c_int, [_vp, _vp]),
    "ccu_last_kernel_ms": (C.c_int, [_vp, C.POINTER(_f)]),
    "ccu_launch_count": (C.c_int, [_vp, C.POINTER(_i64)]),
    "ccu_debug_last_render": (C.c_int, [_vp, _vp]),
    "ccu_debug_last_render_n": (C.c_int, [_vp, _vp, _i32]),
    "ccu_scene_device_bytes": (C.c_int, [_vp, C.POINTER(_i64)]),
    "ccu_scene_commit_ms": (C.c_int, [_vp, C.POINTER(C.c_double)]),
    "ccu_tonemap": (C.c_int, [_vp, _i32, _i32, _f, _vp, _i32, _vp]),
    "ccu_bench_gather": (C.c_int, [_vp, _i64, _i32, C.POINTER(_f), C.POINTER(_f)]),
    "ccu_debug_layout_lookup": (C.c_int, [_vp, _i64, _i32, _vp, _i64, _vp, _vp, _vp, _vp]),
    "ccu_debug_bvh_layout": (C.c_int, [_vp, _i64, _vp, _i64, _vp, _i64, _vp, _i64, C.POINTER(_i64), C.POINTER(_i64), _pi32, _pi32]),
    "ccu_debug_emitter_grid": (C.c_int, [_vp, _i64, _i32, _vp, _i64, _vp, _i64, _vp, _vp, _vp, _vp]),
    "ccu_debug_emitter_models": (C.c_int, [_vp, _i64, _i32, _vp, _i64, _vp, _i64, _vp, _i64, _vp, _i64, _vp, _vp, _vp, _vp, _vp, _vp]),
    "ccu_debug_biome_layout": (C.c_int, [_vp, _vp, _i64, _i32, _vp, _vp, _vp]),
    # multi-GPU
    "ccu_group_create": (C.c_int, [_vp, _i32, C.POINTER(_vp)]),
    "ccu_group_unique_id": (C.c_int, [_vp]),
    "ccu_group_join": (C.c_int, [_vp, _vp, _i32, _i32, C.POINTER(_vp)]),
    "ccu_group_destroy": (C.c_int, [_vp]),
    "ccu_group_size": (C.c_int, [_vp, _pi32, _pi32]),
    "ccu_group_member": (C.c_int, [_vp, _i32, C.POINTER(_vp)]),
    "ccu_group_replicate_scene": (C.c_int, [_vp]),
    "ccu_group_camera_set": (C.c_int, [_vp, _i32, _vp, _i64]),
    "ccu_group_render_begin": (C.c_int, [_vp, _i32, _i32]),
    "ccu_group_render_set_params": (C.c_int, [_vp, C.POINTER(RenderParams)]),
    "ccu_group_render_passes": (C.c_int, [_vp, _vp, _i32]),
    "ccu_group_render_sync": (C.c_int, [_vp]),
    "ccu_group_render_merge": (C.c_int, [_vp, _vp, _i32, _pi32]),
    "ccu_group_render_merge_async": (C.c_int, [_vp, _vp, _i32, _pi32]),
    "ccu_group_render_merge_wait": (C.c_int, [_vp]),
    "ccu_group_render_reduce": (C.c_int, [_vp, _pi32]),
    "ccu_group_render_end": (C.c_int, [_vp]),
    "ccu_group_last_ms": (C.c_int, [_vp, C.POINTER(_f), C.POINTER(_f)]),
}

_lib = None


def _prefer_bundled_nccl():
    """The multi-GPU entry points bind NCCL at run time (dlopen "libnccl.so.2").  A process shares ONE object of that soname,
    whichever user loads it first; torch needs the (newer) copy it ships with, so point the library at that copy when it exists."""
    if os.environ.get("CCU_NCCL_LIB"):
        return
    try:
        import importlib.util
        spec = importlib.util.find_spec("nvidia.nccl")
        for loc in (spec.submodule_search_locations if spec else []):
            cand = os.path.join(loc, "lib", "libnccl.so.2")
            if os.path.exists(cand):
                os.environ["CCU_NCCL_LIB"] = cand
                return
    except Exception:
        pass


def load():
    """Load libchunkycu.so; raises OSError when it has not been built (the UnsatisfiedLinkError path)."""
    global _lib
    if _lib is None:
        _prefer_bundled_nccl()
        if not os.path.exists(LIB_PATH):
            raise OSError(f"{LIB_PATH} not built - run `python -m chunkyclplugin_b200.build` (needs nvcc); there is no CPU fallback")
        lib = C.CDLL(LIB_PATH)
        for name, (res, args) in SYMBOLS.items():
            fn = getattr(lib, name)
            fn.restype = res
            fn.argtypes = args
        _lib = lib
    return _lib


def check(rc: int):
    if rc != CCU_OK:
        raise ChunkyCuError(rc, load().ccu_last_error().decode(errors="replace"))


def _ptr(a: Optional[np.ndarray]):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


def layout_lookup(tree: np.ndarray, depth: int, xyz: np.ndarray):
    """Host-only: what the commit-time traversal layouts answer for the voxels `xyz` (count x 3).  Returns a dict with
    wide_value / wide_level (value-carrying layout) and air_solid / air_level (march layout)."""
    tree = np.ascontiguousarray(tree, dtype=np.int32)
    xyz = np.ascontiguousarray(xyz, dtype=np.int32).reshape(-1, 3)
    n = xyz.shape[0]
    out = {k: np.empty(n, dtype=np.int32) for k in ("wide_value", "wide_level", "air_solid", "air_level")}
    check(load().ccu_debug_layout_lookup(_ptr(tree), tree.size, depth, _ptr(xyz), n, _ptr(out["wide_value"]), _ptr(out["wide_level"]),
                                         _ptr(out["air_solid"]), _ptr(out["air_level"])))
    return out


def debug_bvh_layout(bvh: np.ndarray, trigs: np.ndarray):
    """The BVH stage layout the library builds at commit for a packed BVH node array + triangle palette (host only).
    Returns (rec int32[n, 16], tris int32[...], root, ok)."""
    bvh = np.ascontiguousarray(bvh, dtype=np.int32)
    trigs = np.ascontiguousarray(trigs, dtype=np.int32)
    nr, nt, root, ok = _i64(), _i64(), _i32(), _i32()
    lib = load()
    check(lib.ccu_debug_bvh_layout(_ptr(bvh), bvh.size, _ptr(trigs), trigs.size, None, 0, None, 0, C.byref(nr), C.byref(nt), C.byref(root), C.byref(ok)))
    rec = np.zeros(max(nr.value, 1), dtype=np.int32)
    tris = np.zeros(max(nt.value, 1), dtype=np.int32)
    check(lib.ccu_debug_bvh_layout(_ptr(bvh), bvh.size, _ptr(trigs), trigs.size, _ptr(rec), rec.size, _ptr(tris), tris.size,
                                   C.byref(nr), C.byref(nt), C.byref(root), C.byref(ok)))
    return rec[:nr.value].reshape(-1, 16), tris[:nt.value], root.value, bool(ok.value)


def debug_emitter_grid(tree: np.ndarray, depth: int, block_palette: np.ndarray, mat_palette: np.ndarray):
    """The emitter table of CCU_RENDER_EMITTER_SAMPLING the library builds at commit (host only).  Returns a dict:
    has_emitters, g0 / dim (int[3]: grid origin in voxels, size in cells), shift (log2 of the cell edge), emit (int32[n, 4]:
    x, y, z, block palette position), off (int32[cells + 1]) and list (int32[...])."""
    tree, bp, mp = (np.ascontiguousarray(a, dtype=np.int32) for a in (tree, block_palette, mat_palette))
    info = np.zeros(10, dtype=np.int32)
    lib = load()
    args = (_ptr(tree), tree.size, depth, _ptr(bp), bp.size, _ptr(mp), mp.size, _ptr(info))
    check(lib.ccu_debug_emitter_grid(*args, None, None, None))
    cells = int(np.prod(info[4:7].astype(np.int64)))
    emit = np.zeros(max(int(info[8]) * 4, 1), dtype=np.int32)
    off = np.zeros(cells + 1, dtype=np.int32)
    lst = np.zeros(max(int(info[9]), 1), dtype=np.int32)
    check(lib.ccu_debug_emitter_grid(*args, _ptr(emit), _ptr(off), _ptr(lst)))
    return {"has_emitters": bool(info[0]), "g0": info[1:4].copy(), "dim": info[4:7].copy(), "shift": int(info[7]),
            "emit": emit[:info[8] * 4].reshape(-1, 4), "off": off if info[0] else off[:0], "list": lst[:info[9]]}


def debug_emitter_models(p):
    """The wider emitter table of CCU_RENDER_EMITTER_MODELS the library builds at commit for the packed scene p (host only):
    the keys of debug_emitter_grid plus head (int32 per block palette position: int4 index of its primitive list in prim, -1
    for no model emitter) and prim (int32 headers and primitive records, DESIGN.md §12); all empty without a model emitter."""
    arrs = [np.ascontiguousarray(a, dtype=np.int32) for a in (p.octree, p.block_palette, p.mat_palette, p.quad_models, p.aabb_models)]
    tree, bp, mp, qm, am = arrs
    info = np.zeros(12, dtype=np.int32)
    lib = load()
    args = (_ptr(tree), tree.size, p.octree_depth, _ptr(bp), bp.size, _ptr(mp), mp.size, _ptr(qm), qm.size, _ptr(am), am.size, _ptr(info))
    check(lib.ccu_debug_emitter_models(*args, None, None, None, None, None))
    cells = int(np.prod(info[4:7].astype(np.int64)))
    emit = np.zeros(max(int(info[8]) * 4, 1), dtype=np.int32)
    off = np.zeros(cells + 1, dtype=np.int32)
    lst = np.zeros(max(int(info[9]), 1), dtype=np.int32)
    head = np.zeros(max(int(info[10]), 1), dtype=np.int32)
    prim = np.zeros(max(int(info[11]), 1), dtype=np.int32)
    check(lib.ccu_debug_emitter_models(*args, _ptr(emit), _ptr(off), _ptr(lst), _ptr(head), _ptr(prim)))
    return {"has_emitters": bool(info[0]), "g0": info[1:4].copy(), "dim": info[4:7].copy(), "shift": int(info[7]),
            "emit": emit[:info[8] * 4].reshape(-1, 4), "off": off if info[0] else off[:0], "list": lst[:info[9]],
            "head": head[:info[10]], "prim": prim[:info[11]]}


def _biome_arrays(chunks, rgb):
    chunks = np.ascontiguousarray(chunks, dtype=np.int32).reshape(-1, 2)
    rgb = np.ascontiguousarray(rgb, dtype=np.float32).reshape(-1, 3, 256, 3)
    if rgb.shape[0] != chunks.shape[0]:
        raise ValueError(f"{chunks.shape[0]} chunks but {rgb.shape[0]} colour tiles")
    return chunks, rgb


def debug_biome_layout(chunks, rgb, depth: int):
    """The biome layout of CCU_RENDER_BIOME_TINT the library builds at commit for an octree of `depth` (host only): a dict with
    x0, z0 (the low chunk of the chunks' bounding box), grid (int32[gx, gz], indexed [cx - x0, cz - z0], -1 = no tile) and tiles
    (float32[n, 3, 256, 4])."""
    chunks, rgb = _biome_arrays(chunks, rgb)
    n = chunks.shape[0]
    info = np.zeros(5, dtype=np.int32)
    lib = load()
    check(lib.ccu_debug_biome_layout(_ptr(chunks), _ptr(rgb), n, depth, _ptr(info), None, None))
    grid = np.zeros((int(info[2]), int(info[3])), dtype=np.int32)
    tiles = np.zeros((n, 3, 256, 4), dtype=np.float32)
    check(lib.ccu_debug_biome_layout(_ptr(chunks), _ptr(rgb), n, depth, _ptr(info), _ptr(grid), _ptr(tiles)))
    return {"x0": int(info[0]), "z0": int(info[1]), "grid": grid, "tiles": tiles}


def device_count() -> int:
    n = C.c_int()
    check(load().ccu_device_count(C.byref(n)))
    return n.value


def device_info(index: int) -> dict:
    name = C.create_string_buffer(256)
    sms, khz, mem = C.c_int(), C.c_int(), C.c_uint64()
    check(load().ccu_device_info(index, name, 256, C.byref(sms), C.byref(khz), C.byref(mem)))
    return {"name": name.value.decode(), "sm_count": sms.value, "clock_khz": khz.value, "mem_bytes": mem.value}


class Context:
    """Owns one ccu_ctx (one CUDA device)."""

    def __init__(self, device_index: int = 0, _borrowed=None):
        self._lib = load()
        self._owned = _borrowed is None
        if _borrowed is None:
            h = C.c_void_p()
            check(self._lib.ccu_ctx_create(device_index, C.byref(h)))
        else:
            h = _borrowed          # a member context owned by a Group
        self._h = h
        self.device_index = device_index

    def close(self):
        if getattr(self, "_h", None):
            if self._owned:
                self._lib.ccu_ctx_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    # -- scene -------------------------------------------------------------------------------------
    def _words(self, fn, arr):
        a = np.ascontiguousarray(arr, dtype=np.int32)
        check(fn(self._h, _ptr(a), a.size))

    def scene_begin(self):
        check(self._lib.ccu_scene_begin(self._h))

    def set_octree(self, tree, depth: int):
        a = np.ascontiguousarray(tree, dtype=np.int32)
        check(self._lib.ccu_scene_set_octree(self._h, _ptr(a), a.size, depth))

    def set_block_palette(self, a): self._words(self._lib.ccu_scene_set_block_palette, a)
    def set_quad_models(self, a): self._words(self._lib.ccu_scene_set_quad_models, a)
    def set_aabb_models(self, a): self._words(self._lib.ccu_scene_set_aabb_models, a)
    def set_material_palette(self, a): self._words(self._lib.ccu_scene_set_material_palette, a)
    def set_triangles(self, a): self._words(self._lib.ccu_scene_set_triangles, a)
    def set_world_bvh(self, a): self._words(self._lib.ccu_scene_set_world_bvh, a)
    def set_actor_bvh(self, a): self._words(self._lib.ccu_scene_set_actor_bvh, a)

    def set_biome_colors(self, chunks, rgb):
        """chunks int[n, 2] {cx, cz}, rgb float[n, 3, 256, 3] (planes foliage, grass, water; texel (z & 15) * 16 + (x & 15))."""
        chunks, rgb = _biome_arrays(chunks, rgb)
        check(self._lib.ccu_scene_set_biome_colors(self._h, _ptr(chunks), _ptr(rgb), chunks.shape[0]))

    def set_fog(self, sigma: float, sky_density: float, color, fast: bool):
        """The scene's fog for CCU_RENDER_FOG (DESIGN.md §14): extinction per block, sky fog density in [0, 1], linear RGB
        colour, fast fog; sigma = 0 removes it."""
        col = np.ascontiguousarray(color, np.float32)
        if col.shape != (3,):
            raise ValueError("the fog colour needs 3 components")
        check(self._lib.ccu_scene_set_fog(self._h, float(sigma), float(sky_density), _ptr(col), int(fast)))

    def set_clouds(self, mask, size: float = 1.0, y0: float = 0.0, y1: float = 1.0, u0: float = 0.0, v0: float = 0.0):
        """The scene's cloud layer for CCU_RENDER_CLOUDS (DESIGN.md §15): mask uint8[256, 256] indexed [k, i] (non-zero = cloud),
        cell size, slab y0 < y1 and cell offsets, in the plugin's frame; mask None removes it."""
        if mask is None:
            check(self._lib.ccu_scene_set_clouds(self._h, None, float(size), float(y0), float(y1), float(u0), float(v0)))
            return
        m = np.ascontiguousarray(mask, np.uint8)
        if m.size != 256 * 256:
            raise ValueError("the cloud mask needs 256 x 256 cells")
        check(self._lib.ccu_scene_set_clouds(self._h, _ptr(m), float(size), float(y0), float(y1), float(u0), float(v0)))

    def atlas_create(self, width: int, height: int, layers: int):
        check(self._lib.ccu_scene_atlas_create(self._h, width, height, layers))

    def atlas_write(self, x: int, y: int, layer: int, rgba: np.ndarray):
        a = np.ascontiguousarray(rgba, dtype=np.uint8)
        h, w = a.shape[:2]
        check(self._lib.ccu_scene_atlas_write(self._h, x, y, layer, w, h, _ptr(a)))

    def set_atlas(self, rgba: np.ndarray):
        a = np.ascontiguousarray(rgba, dtype=np.uint8)
        layers, h, w = a.shape[:3]
        check(self._lib.ccu_scene_set_atlas(self._h, _ptr(a), w, h, layers))

    def set_sky(self, rgba: np.ndarray, intensity: float):
        a = np.ascontiguousarray(rgba, dtype=np.uint8)
        check(self._lib.ccu_scene_set_sky(self._h, _ptr(a), a.shape[0], float(intensity)))

    def set_sun(self, words):
        a = np.ascontiguousarray(words, dtype=np.int32)
        assert a.size == 6
        check(self._lib.ccu_scene_set_sun(self._h, _ptr(a)))

    def scene_commit(self):
        check(self._lib.ccu_scene_commit(self._h))

    def camera_set(self, projector_type: int, settings):
        a = np.ascontiguousarray(settings, dtype=np.float32)
        check(self._lib.ccu_camera_set(self._h, projector_type, _ptr(a), a.size))

    # -- rendering ---------------------------------------------------------------------------------
    def render_begin(self, width: int, height: int):
        check(self._lib.ccu_render_begin(self._h, width, height))
        self._wh = (width, height)

    def render_set_params(self, draw_depth=256, max_depth=5, emitter_scale=13.0, kernel=0, flags=0):
        p = RenderParams(draw_depth, max_depth, emitter_scale, kernel, flags)
        check(self._lib.ccu_render_set_params(self._h, C.byref(p)))

    def render_passes(self, seeds, block: bool = True):
        a = np.ascontiguousarray(seeds, dtype=np.int32)
        fn = self._lib.ccu_render_passes if block else self._lib.ccu_render_passes_async
        check(fn(self._h, _ptr(a), a.size))

    def render_sync(self):
        check(self._lib.ccu_render_sync(self._h))

    def render_read(self, out: Optional[np.ndarray] = None):
        w, h = self._wh
        if out is None:
            out = np.empty(w * h * 3, dtype=np.float32)
        spp = C.c_int32()
        check(self._lib.ccu_render_read(self._h, _ptr(out), C.byref(spp)))
        return out, spp.value

    def render_merge(self, sample_buffer: np.ndarray, sample_spp: int) -> int:
        assert sample_buffer.dtype == np.float64 and sample_buffer.flags.c_contiguous
        m = C.c_int32()
        check(self._lib.ccu_render_merge(self._h, _ptr(sample_buffer), sample_spp, C.byref(m)))
        return m.value

    def render_merge_async(self, sample_buffer: np.ndarray, sample_spp: int) -> int:
        """Closes the window and merges it in the background; ``sample_buffer`` must stay alive until render_merge_wait()."""
        assert sample_buffer.dtype == np.float64 and sample_buffer.flags.c_contiguous
        m = C.c_int32()
        check(self._lib.ccu_render_merge_async(self._h, _ptr(sample_buffer), sample_spp, C.byref(m)))
        self._merge_keepalive = sample_buffer
        return m.value

    def render_merge_wait(self):
        check(self._lib.ccu_render_merge_wait(self._h))
        self._merge_keepalive = None

    def render_window_close(self) -> int:
        """Closes the window and starts its read-back; returns the window's passes (merge it with render_window_merge)."""
        m = C.c_int32()
        check(self._lib.ccu_render_window_close(self._h, C.byref(m)))
        return m.value

    def render_window_merge(self, sample_buffer: np.ndarray, sample_spp: int):
        assert sample_buffer.dtype == np.float64 and sample_buffer.flags.c_contiguous
        check(self._lib.ccu_render_window_merge(self._h, _ptr(sample_buffer), sample_spp))

    def render_reset_window(self):
        check(self._lib.ccu_render_reset_window(self._h))

    def render_set_window_spp(self, window_spp: int):
        check(self._lib.ccu_render_set_window_spp(self._h, int(window_spp)))

    def render_end(self):
        check(self._lib.ccu_render_end(self._h))

    def render_device_buffer(self):
        p, n = C.c_void_p(), C.c_int64()
        check(self._lib.ccu_render_device_buffer(self._h, C.byref(p), C.byref(n)))
        return p.value, n.value

    def render_scale(self, factor: float):
        check(self._lib.ccu_render_scale(self._h, float(factor)))

    def stream_handle(self) -> int:
        p = C.c_void_p()
        check(self._lib.ccu_stream_handle(self._h, C.byref(p)))
        return p.value or 0

    def first_hit(self, seed: int) -> dict:
        w, h = self._wh
        n = w * h
        out = dict(block=np.empty(n, np.int32), face=np.empty(n, np.int32), node=np.empty(n, np.int32),
                   kind=np.empty(n, np.int32), t=np.empty(n, np.float32), normal=np.empty(n * 3, np.float32),
                   color=np.empty(n * 4, np.float32))
        check(self._lib.ccu_first_hit(self._h, seed, _ptr(out["block"]), _ptr(out["face"]), _ptr(out["node"]),
                                      _ptr(out["kind"]), _ptr(out["t"]), _ptr(out["normal"]), _ptr(out["color"])))
        return out

    def preview(self) -> np.ndarray:
        w, h = self._wh
        out = np.empty(w * h, np.int32)
        check(self._lib.ccu_preview(self._h, _ptr(out)))
        return out

    def tonemap(self, width: int, height: int, exposure: float, sample_buffer: np.ndarray, filter_type: int) -> np.ndarray:
        """GpuPostProcessingFilter.processFrame: double sample buffer -> ARGB int[W*H]."""
        inp = np.ascontiguousarray(sample_buffer, dtype=np.float64).reshape(-1)
        if inp.size != width * height * 3:
            raise ValueError("sample buffer must hold 3 doubles per pixel")
        out = np.empty(width * height, dtype=np.int32)
        check(self._lib.ccu_tonemap(self._h, width, height, C.c_float(exposure), _ptr(inp), filter_type, _ptr(out)))
        return out

    def bench_gather(self, array_bytes: int, dependent: bool = False):
        """Random 32-byte-sector gather microbenchmark: returns (GB/s of sectors, ns per load per thread)."""
        gbs, ns = C.c_float(), C.c_float()
        check(self._lib.ccu_bench_gather(self._h, int(array_bytes), 1 if dependent else 0, C.byref(gbs), C.byref(ns)))
        return float(gbs.value), float(ns.value)

    def last_kernel_ms(self) -> float:
        ms = C.c_float()
        check(self._lib.ccu_last_kernel_ms(self._h, C.byref(ms)))
        return ms.value

    def launch_count(self) -> int:
        n = C.c_int64()
        check(self._lib.ccu_launch_count(self._h, C.byref(n)))
        return n.value

    def last_render(self) -> tuple:
        """The render kernel instance of the last render_passes launch: (kernel, has_bvh, lay or mode, spec, nee, biome,
        staged sky texels), all zero before the first launch (ccu_debug_last_render)."""
        out = np.zeros(7, np.int32)
        check(self._lib.ccu_debug_last_render(self._h, _ptr(out)))
        return tuple(int(v) for v in out)

    def last_render_n(self, n: int = 9) -> tuple:
        """The first min(n, 9) entries of the last launch's instance: last_render()'s 7, then fog and clouds
        (ccu_debug_last_render_n)."""
        out = np.zeros(max(n, 0), np.int32)
        check(self._lib.ccu_debug_last_render_n(self._h, _ptr(out), n))
        return tuple(int(v) for v in out[:min(n, 9)])

    def scene_device_bytes(self) -> int:
        n = C.c_int64()
        check(self._lib.ccu_scene_device_bytes(self._h, C.byref(n)))
        return n.value

    def scene_commit_ms(self) -> float:
        ms = C.c_double()
        check(self._lib.ccu_scene_commit_ms(self._h, C.byref(ms)))
        return ms.value


def group_unique_id() -> bytes:
    """NCCL unique id for a one-process-per-GPU group: rank 0 calls this and the host distributes the 128 bytes."""
    buf = C.create_string_buffer(CCU_UNIQUE_ID_BYTES)
    check(load().ccu_group_unique_id(buf))
    return buf.raw


class Group:
    """N GPUs of one box rendering one image: ccu_group_* (include/chunkycu.h, "multi-GPU").

    ``Group(devices=[0, 1, ...])`` drives all GPUs from this process (what a JVM plugin does);
    ``Group(ctx=ctx, unique_id=..., rank=r, world=N)`` wraps this process's context in a one-process-per-GPU job."""

    def __init__(self, devices=None, ctx: Optional[Context] = None, unique_id: Optional[bytes] = None, rank: int = 0, world: int = 1):
        self._lib = load()
        h = C.c_void_p()
        if devices is not None:
            d = np.ascontiguousarray(devices, dtype=np.int32)
            check(self._lib.ccu_group_create(_ptr(d), d.size, C.byref(h)))
            self._ctx_keep = None
        else:
            assert ctx is not None
            uid = C.create_string_buffer(unique_id, CCU_UNIQUE_ID_BYTES) if unique_id is not None else None
            check(self._lib.ccu_group_join(ctx._h, uid, rank, world, C.byref(h)))
            self._ctx_keep = ctx
        self._h = h
        w, l = C.c_int32(), C.c_int32()
        check(self._lib.ccu_group_size(self._h, C.byref(w), C.byref(l)))
        self.world, self.local_members = w.value, l.value
        self.rank = rank if devices is None else 0
        self._wh = None

    def close(self):
        if getattr(self, "_h", None):
            self._lib.ccu_group_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def member(self, i: int) -> Context:
        h = C.c_void_p()
        check(self._lib.ccu_group_member(self._h, i, C.byref(h)))
        if self._ctx_keep is not None:
            return self._ctx_keep
        c = Context(_borrowed=h)
        return c

    def replicate_scene(self):
        check(self._lib.ccu_group_replicate_scene(self._h))

    def camera_set(self, projector_type: int, settings):
        a = np.ascontiguousarray(settings, dtype=np.float32)
        check(self._lib.ccu_group_camera_set(self._h, projector_type, _ptr(a), a.size))

    def render_begin(self, width: int, height: int):
        check(self._lib.ccu_group_render_begin(self._h, width, height))
        self._wh = (width, height)

    def render_set_params(self, draw_depth=256, max_depth=5, emitter_scale=13.0, kernel=0, flags=0):
        p = RenderParams(draw_depth, max_depth, emitter_scale, kernel, flags)
        check(self._lib.ccu_group_render_set_params(self._h, C.byref(p)))

    def render_passes(self, seeds):
        a = np.ascontiguousarray(seeds, dtype=np.int32)
        check(self._lib.ccu_group_render_passes(self._h, _ptr(a), a.size))

    def render_sync(self):
        check(self._lib.ccu_group_render_sync(self._h))

    def render_merge(self, sample_buffer: np.ndarray, sample_spp: int) -> int:
        assert sample_buffer.dtype == np.float64 and sample_buffer.flags.c_contiguous
        m = C.c_int32()
        check(self._lib.ccu_group_render_merge(self._h, _ptr(sample_buffer), sample_spp, C.byref(m)))
        return m.value

    def render_merge_async(self, sample_buffer: np.ndarray, sample_spp: int) -> int:
        assert sample_buffer.dtype == np.float64 and sample_buffer.flags.c_contiguous
        m = C.c_int32()
        check(self._lib.ccu_group_render_merge_async(self._h, _ptr(sample_buffer), sample_spp, C.byref(m)))
        self._merge_keepalive = sample_buffer
        return m.value

    def render_merge_wait(self):
        check(self._lib.ccu_group_render_merge_wait(self._h))
        self._merge_keepalive = None

    def reduce_only(self) -> int:
        """Reduce-scatter of the open window without the read-back (the sums stay on the GPUs); returns the window's passes."""
        m = C.c_int32()
        check(self._lib.ccu_group_render_reduce(self._h, C.byref(m)))
        return m.value

    def render_end(self):
        check(self._lib.ccu_group_render_end(self._h))

    def last_ms(self):
        a, b = C.c_float(), C.c_float()
        check(self._lib.ccu_group_last_ms(self._h, C.byref(a), C.byref(b)))
        return a.value, b.value
