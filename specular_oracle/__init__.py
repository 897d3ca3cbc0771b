"""ctypes binding of the CPU restatement of CCU_RENDER_SPECULAR, CCU_RENDER_EMITTER_SAMPLING and CCU_RENDER_EMITTER_NEAR_FIELD
(specular_oracle.c).  TEST INFRASTRUCTURE ONLY.

``SpecularOracle`` is the parity oracle (``oracle.Oracle``) with the specular events of DESIGN.md section 9 in its path
loop; ``FlagsOracle`` takes the render flags and adds the emitter sampling of sections 10 and 11, with the emitter table that
``emitter_grid`` builds from the packed arrays.  Everything else - first hit, preview, counters - is the oracle's.  Like the
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
    return _lib


class _Grid(C.Structure):
    _fields_ = [("emit", C.c_void_p), ("off", C.c_void_p), ("list", C.c_void_p),
                ("g0", C.c_int32 * 3), ("dim", C.c_int32 * 3), ("shift", C.c_int32)]


CCU_RENDER_SPECULAR, CCU_RENDER_EMITTER_SAMPLING, CCU_RENDER_EMITTER_NEAR_FIELD = 4, 8, 128
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


def emitter_grid(p) -> dict:
    """The emitter table and cell lists of DESIGN.md section 10 for a packed scene (same keys as native.debug_emitter_grid)."""
    empty = {"has_emitters": False, "g0": np.zeros(3, np.int32), "dim": np.zeros(3, np.int32), "shift": EMIT_SHIFT0,
             "emit": np.zeros((0, 4), np.int32), "off": np.zeros(0, np.int32), "list": np.zeros(0, np.int32)}
    emits = emitter_blocks(p.block_palette, p.mat_palette)
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
    return {"has_emitters": True, "g0": g0.astype(np.int32), "dim": dim.astype(np.int32), "shift": shift,
            "emit": e.astype(np.int32), "off": np.cumsum(off).astype(np.int32), "list": idx[order].astype(np.int32)}


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
    CCU_RENDER_EMITTER_NEAR_FIELD bits (the other flags act on the scene: oracle.edge_rays.without_sun, or empty BVHs for
    CCU_RENDER_NO_ENTITIES)."""

    def __init__(self, scene, flags: int = 0, **kw):
        super().__init__(scene, **kw)
        self.flags = flags
        self.grid = emitter_grid(scene)
        g = _Grid()
        for k in ("emit", "off", "list"):
            a = np.ascontiguousarray(self.grid[k], dtype=np.int32)
            self._keep["grid_" + k] = a
            setattr(g, k, a.ctypes.data)
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
                           C.c_int(1 if self.flags & CCU_RENDER_EMITTER_NEAR_FIELD else 0))
        self._counters(cnt)
        return res
