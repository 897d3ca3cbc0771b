"""Stored outputs of the reference's OpenCL kernel at the BASELINE configurations' real sizes.  TEST INFRASTRUCTURE ONLY.

scripts/acceptance_golden.py runs the unmodified reference kernel (oracle/clref) on a B200 and writes
tests/golden/acceptance_reference.npz; tests/test_gpu_acceptance.py compares the CUDA path with it.  A full frame of
first-hit buffers or converged radiance is far too large to store, so the file holds
  * first hit (strict build, bit-exact comparison): SHA-256 digests of the full-frame buffers, plus the values at a
    strided pixel sample so that a mismatch can be located;
  * converged radiance (stock build, statistical comparison): the mean RGB at a strided pixel sample and the full-frame
    image mean.
"""
from __future__ import annotations

import hashlib
import os
from typing import Dict

import numpy as np

PATH = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests", "golden", "acceptance_reference.npz")
FIRST_HIT_SAMPLES = 1024
RADIANCE_SAMPLES = 2048


def sample_pixels(n_pixels: int, k: int) -> np.ndarray:
    """About k pixel indices spread over the frame (a stride that is not a multiple of the row length)."""
    stride = n_pixels // k
    return np.arange(stride // 2, n_pixels, stride, dtype=np.int64)


def first_hit_digests(hit: np.ndarray, block: np.ndarray, t: np.ndarray, normal: np.ndarray, color: np.ndarray) -> Dict[str, str]:
    """Digests of the hit mask and of every buffer at the hit pixels (what the reference defines for a hit)."""
    hit = np.asarray(hit, bool).reshape(-1)
    parts = {"hit": hit.astype(np.uint8), "block": np.asarray(block, "<i4").reshape(-1)[hit],
             "t": np.asarray(t, "<f4").reshape(-1)[hit], "normal": np.asarray(normal, "<f4").reshape(-1, 3)[hit],
             "color": np.asarray(color, "<f4").reshape(-1, 4)[hit]}
    return {k: hashlib.sha256(np.ascontiguousarray(v).tobytes()).hexdigest() for k, v in parts.items()}
