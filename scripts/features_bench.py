"""Cost of the denoiser's feature buffers (ccu_render_features, DESIGN §16) at 1920 x 1080 on config 1 (256^3 terrain, sun on) and
config 4 (config 1 terrain with entity BVHs).

Per config, three legs alternated window by window in one process, L2 flushed before each, on the same committed scene: `render`
= a 16-pass window of kernel 0 (the wavefront kernel, what bench.py times), `features` = one ccu_render_features call over the
same 16 seeds, and `first_hit` = one ccu_first_hit launch (the pass the feature kernel's march comes from).  Times are CUDA-event
device times (ccu_last_kernel_ms).  Prints one JSON line with the GPU's name, power limit and SM clock.

    python scripts/features_bench.py [--windows N] [--warmup W] [--out FILE]
"""
from __future__ import annotations

import argparse
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "scripts"))
PASSES = 16


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--windows", type=int, default=8, help="timed windows per leg")
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()

    import torch
    from chunkyclplugin_b200 import native, scenes as S
    from chunkyclplugin_b200.javarandom import JavaRandom
    from chunkyclplugin_b200.renderer import upload_scene
    from emitter_models_bench import gpu_info

    configs = {"config1_1080p": lambda: S.terrain_scene(256, 1920, 1080), "config4_1080p": lambda: S.entity_scene(256, 1920, 1080)}
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")      # > 126 MB L2
    result = dict(gpu_info(), windows=args.windows, warmup=args.warmup, passes_per_window=PASSES, render_kernel=0, configs={})
    for cname, make in configs.items():
        p = make()
        ctx = native.Context(0)
        upload_scene(ctx, p)
        ctx.camera_set(p.projector_type, p.camera)
        ctx.render_set_params(kernel=0)
        ctx.render_begin(p.width, p.height)
        rand = JavaRandom(0)
        ms = {"render": [], "features": [], "first_hit": []}
        for i in range(args.warmup + args.windows):
            seeds = np.asarray([rand.next_int() for _ in range(PASSES)], np.int32)
            for leg in ms:
                flush.fill_(i & 0xFF)
                torch.cuda.synchronize()
                if leg == "render":
                    ctx.render_reset_window()
                    ctx.render_passes(seeds)
                elif leg == "features":
                    ctx.render_features(seeds)
                else:
                    ctx.first_hit(int(seeds[0]))
                if i >= args.warmup:
                    ms[leg].append(ctx.last_kernel_ms())
        instance = ctx.last_features()
        ctx.render_end()
        ctx.close()
        per_pass = {"render": PASSES, "features": PASSES, "first_hit": 1}
        result["configs"][cname] = {
            "width": p.width, "height": p.height, "feature_instance": list(instance),
            "legs": {k: {"ms_per_call_mean": float(np.mean(v)), "ms_min": float(np.min(v)), "ms_max": float(np.max(v)),
                         "passes_per_call": per_pass[k], "ms_per_pass": float(np.mean(v)) / per_pass[k]} for k, v in ms.items()},
            "feature_pass_over_render_pass": float(np.mean(ms["features"]) / np.mean(ms["render"])),
            "feature_pass_over_first_hit": float(np.mean(ms["features"]) / PASSES / np.mean(ms["first_hit"])),
        }
    line = json.dumps(result)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")
    return 0


if __name__ == "__main__":
    sys.exit(main())
