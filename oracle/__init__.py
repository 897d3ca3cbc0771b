"""ctypes binding of the CPU oracle (oracle/chunky_oracle.c).  TEST INFRASTRUCTURE ONLY.

Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference legs may
import this package.  The product (chunkyclplugin_b200) never does.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess
from typing import Dict, Optional, Sequence

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB_PATH = os.path.join(_HERE, "_build", "liboracle.so")
_lib = None


def build(force: bool = False) -> str:
    src = os.path.join(_HERE, "chunky_oracle.c")
    if force or not os.path.exists(_LIB_PATH) or os.path.getmtime(_LIB_PATH) < os.path.getmtime(src):
        subprocess.run(["make", "-C", _HERE, "CC=gcc"], check=True, capture_output=True)
    return _LIB_PATH


class _Scene(C.Structure):
    _fields_ = [
        ("octree", C.c_void_p), ("octree_len", C.c_int64), ("octree_depth", C.c_int32),
        ("block_palette", C.c_void_p), ("quad_models", C.c_void_p), ("aabb_models", C.c_void_p),
        ("world_bvh", C.c_void_p), ("actor_bvh", C.c_void_p), ("bvh_trigs", C.c_void_p),
        ("atlas", C.c_void_p), ("atlas_w", C.c_int32), ("atlas_h", C.c_int32), ("atlas_layers", C.c_int32),
        ("mat_palette", C.c_void_p),
        ("sky", C.c_void_p), ("sky_res", C.c_int32), ("sky_intensity", C.c_float),
        ("sun", C.c_void_p),
        ("projector_type", C.c_int32), ("camera", C.c_void_p),
        ("width", C.c_int32), ("height", C.c_int32),
        ("draw_depth", C.c_int32), ("max_depth", C.c_int32), ("emitter_scale", C.c_float), ("math_mode", C.c_int32),
    ]


COUNTER_NAMES = ("samples", "rays", "march_steps", "descent_loads", "block_tests", "material_samples", "texel_reads",
                 "bvh_calls", "bvh_inner", "bvh_leaf", "triangles", "sky_lookups", "sun_texels", "aabb_boxes", "quads",
                 "segments")


class _Counters(C.Structure):
    _fields_ = [(n, C.c_uint64) for n in COUNTER_NAMES]


def lib():
    global _lib
    if _lib is None:
        build()
        _lib = C.CDLL(_LIB_PATH)
        assert _lib.oracle_scene_struct_size() == C.sizeof(_Scene), "OracleScene layout mismatch"
    return _lib


def algorithmic_bytes(counters: Dict[str, int]) -> int:
    """SURVEY.md 8(d): bytes the algorithm must touch, from the oracle's event counts."""
    c = counters
    return int(4 * c["descent_loads"] + 8 * c["block_tests"] + 24 * c["material_samples"] + 4 * c["texel_reads"]
               + 28 * c["bvh_calls"] + 60 * c["bvh_inner"] + 4 * c["bvh_leaf"] + 80 * c["triangles"]
               + 16 * c["sky_lookups"] + 52 * c["aabb_boxes"] + 60 * c["quads"] + 24 * c["samples"])


class Oracle:
    """Holds a scene (numpy arrays kept alive) and runs the restated kernels on the CPU."""

    def __init__(self, scene, draw_depth: int = 256, max_depth: int = 5, emitter_scale: float = 13.0,
                 math_mode: int = 0):
        self.scene = scene
        self._keep = {}
        s = _Scene()

        def ptr(name, arr, dtype):
            a = np.ascontiguousarray(arr, dtype=dtype)
            self._keep[name] = a
            return a.ctypes.data

        s.octree = ptr("octree", scene.octree, np.int32)
        s.octree_len = scene.octree.size
        s.octree_depth = scene.octree_depth
        s.block_palette = ptr("bp", scene.block_palette, np.int32)
        s.quad_models = ptr("qm", scene.quad_models, np.int32)
        s.aabb_models = ptr("am", scene.aabb_models, np.int32)
        s.world_bvh = ptr("wb", scene.world_bvh, np.int32)
        s.actor_bvh = ptr("ab", scene.actor_bvh, np.int32)
        s.bvh_trigs = ptr("tr", scene.bvh_trigs, np.int32)
        s.atlas = ptr("atlas", scene.atlas, np.uint8)
        s.atlas_layers, s.atlas_h, s.atlas_w = scene.atlas.shape[:3]
        s.mat_palette = ptr("mp", scene.mat_palette, np.int32)
        s.sky = ptr("sky", scene.sky, np.uint8)
        s.sky_res = scene.sky.shape[0]
        s.sky_intensity = scene.sky_intensity
        s.sun = ptr("sun", scene.sun, np.int32)
        s.projector_type = scene.projector_type
        s.camera = ptr("cam", scene.camera, np.float32)
        s.width, s.height = scene.width, scene.height
        s.draw_depth, s.max_depth, s.emitter_scale, s.math_mode = draw_depth, max_depth, emitter_scale, math_mode
        self._s = s
        self.last_counters: Dict[str, int] = {}

    def _counters(self, c: _Counters) -> Dict[str, int]:
        self.last_counters = {n: int(getattr(c, n)) for n in COUNTER_NAMES}
        return self.last_counters

    def render(self, seeds: Sequence[int], start_spp: int = 0, res: Optional[np.ndarray] = None,
               gids: Optional[np.ndarray] = None, threads: int = 0) -> np.ndarray:
        """Running mean over the passes (rayTracer.cl:109-112); returns float32[H*W*3]."""
        n = self._s.width * self._s.height
        if res is None:
            res = np.zeros(n * 3, dtype=np.float32)
        assert res.dtype == np.float32 and res.size == n * 3 and res.flags.c_contiguous
        sd = np.ascontiguousarray(seeds, dtype=np.int32)
        cnt = _Counters()
        gp, gn = None, 0
        if gids is not None:
            g = np.ascontiguousarray(gids, dtype=np.int32)
            gp, gn = g.ctypes.data_as(C.c_void_p), g.size
        lib().oracle_render(C.byref(self._s), sd.ctypes.data_as(C.c_void_p), C.c_int(sd.size), C.c_int(start_spp),
                            res.ctypes.data_as(C.c_void_p), gp, C.c_int64(gn), C.c_int(threads), C.byref(cnt))
        self._counters(cnt)
        return res

    def first_hit(self, seed: int, threads: int = 0) -> Dict[str, np.ndarray]:
        n = self._s.width * self._s.height
        out = dict(block=np.zeros(n, np.int32), face=np.zeros(n, np.int32), node=np.zeros(n, np.int32),
                   kind=np.zeros(n, np.int32), t=np.zeros(n, np.float32), normal=np.zeros(n * 3, np.float32),
                   color=np.zeros(n * 4, np.float32))
        cnt = _Counters()
        p = lambda a: a.ctypes.data_as(C.c_void_p)
        lib().oracle_first_hit(C.byref(self._s), C.c_int32(seed), p(out["block"]), p(out["face"]), p(out["node"]),
                               p(out["kind"]), p(out["t"]), p(out["normal"]), p(out["color"]), C.c_int(threads),
                               C.byref(cnt))
        self._counters(cnt)
        return out

    def preview(self, threads: int = 0) -> np.ndarray:
        n = self._s.width * self._s.height
        res = np.zeros(n, np.int32)
        lib().oracle_preview(C.byref(self._s), res.ctypes.data_as(C.c_void_p), C.c_int(threads))
        return res

    def sun_basis(self) -> np.ndarray:
        """float32[3, 3]: rows sw, su, sv of Sun_new (sky.h:19-40)."""
        out = np.zeros(9, np.float32)
        lib().oracle_sun_basis(C.byref(self._s), out.ctypes.data_as(C.c_void_p))
        return out.reshape(3, 3)

    def camera_rays(self, seed: int) -> np.ndarray:
        n = self._s.width * self._s.height
        rays = np.zeros(n * 6, np.float32)
        lib().oracle_camera_rays(C.byref(self._s), C.c_int32(seed), rays.ctypes.data_as(C.c_void_p))
        return rays.reshape(n, 6)


def rng_chain(state: int, n: int):
    st = np.zeros(n, np.uint32)
    fl = np.zeros(n, np.float32)
    lib().oracle_rng_chain(C.c_uint32(state), C.c_int(n), st.ctypes.data_as(C.c_void_p), fl.ctypes.data_as(C.c_void_p))
    return st, fl


def math_fn(fn: str, x: np.ndarray, y: Optional[np.ndarray] = None, libm: bool = False) -> np.ndarray:
    code = {"sin": 0, "cos": 1, "atan2": 2, "asin": 3, "acos": 4}[fn]
    x = np.ascontiguousarray(x, np.float32)
    y = np.ascontiguousarray(y if y is not None else np.zeros_like(x), np.float32)
    out = np.zeros_like(x)
    lib().oracle_math(C.c_int(code), C.c_int(int(libm)), x.ctypes.data_as(C.c_void_p), y.ctypes.data_as(C.c_void_p),
                      out.ctypes.data_as(C.c_void_p), C.c_int64(x.size))
    return out


def num_threads() -> int:
    return int(lib().oracle_num_threads())


def tonemap(width: int, height: int, exposure: float, sample_buffer: np.ndarray, filter_type: int, libm: bool = False,
            threads: int = 0) -> np.ndarray:
    """post_processing_filter.cl:5-51 on the CPU: double sample buffer -> ARGB int[W*H]."""
    inp = np.ascontiguousarray(sample_buffer, dtype=np.float64).reshape(-1)
    assert inp.size == width * height * 3
    out = np.empty(width * height, dtype=np.int32)
    rc = lib().oracle_tonemap(C.c_int(width), C.c_int(height), C.c_float(exposure), inp.ctypes.data_as(C.c_void_p), C.c_int(filter_type),
                              out.ctypes.data_as(C.c_void_p), C.c_int(1 if libm else 0), C.c_int(threads))
    if rc != 0:
        raise ValueError("oracle_tonemap: bad arguments")
    return out
