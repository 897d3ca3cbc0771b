"""Portable float maps (PFM), the image format Open Image Denoise's tools and the Chunky denoiser plugin read: the beauty image and
the feature buffers of ``CudaPathTracingRenderer.render_features`` (DESIGN.md §16) go to the denoiser as three such files."""
from __future__ import annotations

import numpy as np


def write_pfm(path: str, rgb, width: int, height: int) -> None:
    """Writes rgb (3 values per pixel, rows top to bottom as in Chunky's buffers) as a colour PFM: the header "PF", the size and
    the scale -1 (little-endian), then float32 rows from the bottom row up."""
    a = np.asarray(rgb, dtype=np.float32)
    if a.size != width * height * 3:
        raise ValueError(f"write_pfm: {a.size} values for a {width} x {height} RGB image")
    rows = a.reshape(height, width, 3)[::-1]
    with open(path, "wb") as f:
        f.write(b"PF\n%d %d\n-1\n" % (width, height))
        f.write(np.ascontiguousarray(rows, dtype="<f4").tobytes())
