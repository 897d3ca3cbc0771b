"""ctypes binding of the CPU restatement of CCU_RENDER_SPECULAR (specular_oracle.c).  TEST INFRASTRUCTURE ONLY.

``SpecularOracle`` is the parity oracle (``oracle.Oracle``) with the specular events of DESIGN.md section 9 in its path
loop; everything else - first hit, preview, counters - is the oracle's.  Like the oracle, only tests/ and scripts use it.
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
    return _lib


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
