#!/usr/bin/env python3
"""Writes tests/golden/clref_edge_rays.npz from the reference's unmodified OpenCL kernel (strict build: IEEE arithmetic,
see oracle/clref) on the scenes of oracle/edge_rays.py.

  python scripts/edge_rays_golden.py [out dir]      # default tests/golden; needs oracle/_ref and a GPU with OpenCL

Per catalogue scene (edge_*): the probe_first_hit buffers (hit, material, t, normal, colour) of every pixel, the 4-pass
radiance with the sun on and with it off, and the preview.  Per sun scene (sun_*): the 4-pass radiance.
"""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from chunkyclplugin_b200.javarandom import pass_seeds  # noqa: E402
from oracle import clref  # noqa: E402
from oracle import edge_rays as E  # noqa: E402

NAME = "clref_edge_rays.npz"
PASSES = 4


def main() -> int:
    out_dir = sys.argv[1] if len(sys.argv) > 1 else os.path.join(ROOT, "tests", "golden")
    why = clref.available()
    if why is not None:
        raise SystemExit(f"reference kernel not runnable: {why}")
    g = {}
    device = None
    seed = pass_seeds(1)[0]
    for name, p in E.scenes().items():
        variants = [("sun", p), ("nosun", E.without_sun(p))] if name.startswith("edge_") else [("sun", p)]
        for tag, q in variants:
            ref = clref.ClReference(q, strict=True)
            try:
                device = device or ref.device_name()
                img, _ = ref.render(pass_seeds(PASSES))
                g[f"{name}__rad_{tag}"] = img
                if tag == "sun" and name.startswith("edge_"):
                    fh = ref.first_hit(seed)
                    g[f"{name}__hit"] = fh["hit"].astype(np.int8)
                    g[f"{name}__block"] = fh["block"]
                    g[f"{name}__t"] = fh["t"]
                    g[f"{name}__normal"] = fh["normal"]
                    g[f"{name}__color"] = fh["color"]
                    assert E.same_bits_or_nan(fh["ray"], q.camera).all(), name
                    g[f"{name}__preview"] = ref.preview()[0]
                    print(name, "first hit:", int(fh["hit"].sum()), "of", q.width * q.height, flush=True)
            finally:
                ref.close()
    g["seed"] = np.int32(seed)
    g["passes"] = np.int32(PASSES)
    g["device"] = np.array(device)
    os.makedirs(out_dir, exist_ok=True)
    path = os.path.join(out_dir, NAME)
    np.savez_compressed(path, **g)
    print("wrote", path, os.path.getsize(path), "bytes")
    return 0


if __name__ == "__main__":
    sys.exit(main())
