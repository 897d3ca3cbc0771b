#!/usr/bin/env python3
"""Writes acceptance_reference.npz (see oracle/golden.py) from the reference's unmodified OpenCL kernel.

  python scripts/acceptance_golden.py [out dir]      # default tests/golden; needs oracle/_ref and a GPU with OpenCL

The scenes, seeds and spp are those of tests/test_gpu_acceptance.py.
"""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from chunkyclplugin_b200 import scenes as S  # noqa: E402
from chunkyclplugin_b200.javarandom import JavaRandom, pass_seeds  # noqa: E402
from oracle import clref, golden  # noqa: E402

SCENES = {"config1": lambda: S.terrain_scene(256, 1920, 1080), "config3": lambda: S.indoor_scene(256, 1920, 1080),
          "config4": lambda: S.entity_scene(256, 1920, 1080), "config5": lambda: S.large_world_scene(width=3840, height=2160)}
RADIANCE_SPP = {"config1": 256, "config4": 64, "config3": 1024}


def rel_rmse(a, b):
    a, b = a.astype(np.float64), b.astype(np.float64)
    return float(np.sqrt(np.mean((a - b) ** 2)) / b.mean())


def main() -> int:
    out_dir = sys.argv[1] if len(sys.argv) > 1 else os.path.dirname(golden.PATH)
    why = clref.available()
    if why is not None:
        raise SystemExit(f"reference kernel not runnable: {why}")
    g = {}
    for config, make in SCENES.items():
        p = make()
        n = p.width * p.height
        ref = clref.ClReference(p, strict=True)
        try:
            fh = ref.first_hit(pass_seeds(1)[0])
            device = ref.device_name()
        finally:
            ref.close()
        hit = fh["hit"] != 0
        for k, v in golden.first_hit_digests(hit, fh["block"], fh["t"], fh["normal"], fh["color"]).items():
            g[f"fh_{config}_digest_{k}"] = np.array(v)
        idx = golden.sample_pixels(n, golden.FIRST_HIT_SAMPLES)
        g[f"fh_{config}_hit"] = hit[idx].astype(np.uint8)
        g[f"fh_{config}_block"] = fh["block"][idx]
        g[f"fh_{config}_t"] = fh["t"][idx]
        g[f"fh_{config}_normal"] = fh["normal"].reshape(-1, 3)[idx]
        g[f"fh_{config}_color"] = fh["color"].reshape(-1, 4)[idx]
        print(config, "first hit:", int(hit.sum()), "of", n, "pixels hit", flush=True)
        if config not in RADIANCE_SPP:
            continue
        spp = RADIANCE_SPP[config]
        ref = clref.ClReference(p, strict=False)
        try:
            want, _ = ref.render(pass_seeds(spp))
            if config == "config3":             # the reference's own noise: the same spp on a disjoint seed stream
                r2 = JavaRandom(987654321)
                want2, _ = ref.render([r2.next_int() for _ in range(spp)])
        finally:
            ref.close()
        idx = golden.sample_pixels(n, golden.RADIANCE_SAMPLES)
        rgb = want.reshape(-1, 3)
        g[f"rad_{config}_rgb"] = rgb[idx]
        g[f"rad_{config}_mean"] = np.float64(want.mean())
        if config == "config3":
            g["rad_config3_noise_floor"] = np.float64(rel_rmse(want2.reshape(-1, 3)[idx], rgb[idx]))
            print(config, "noise floor: sample", float(g["rad_config3_noise_floor"]), "full frame", rel_rmse(want2, want))
        print(config, "radiance:", spp, "spp, mean", float(want.mean()), flush=True)
    g["device"] = np.array(device)
    os.makedirs(out_dir, exist_ok=True)
    path = os.path.join(out_dir, os.path.basename(golden.PATH))
    np.savez_compressed(path, **g)
    print("wrote", path, os.path.getsize(path), "bytes")
    return 0


if __name__ == "__main__":
    sys.exit(main())
