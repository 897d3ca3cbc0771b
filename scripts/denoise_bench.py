"""Cost of the guided denoiser (ccu_denoise, DESIGN §17) at 1920 x 1080 and 3840 x 2160, for 1, 3 and 5 iterations.

The input is real: config 1 (256^3 terrain, sun on) rendered for 16 passes by kernel 0, with 16-pass feature buffers.  Per size,
legs alternated round by round in one process, L2 flushed (a 256 MB fill) before each: `render` = a 16-pass window of kernel 0
(what bench.py times), and `denoise_<k>` = one ccu_denoise call of k iterations on that window's image.  `device_ms` is the
CUDA-event time of the denoise launches (ccu_last_kernel_ms); `e2e_ms` is the host time of Context.denoise, host copies
included (pageable buffers, as a Java or numpy caller passes them).  Prints one JSON line with the GPU's name, power limit
and SM clock.

    python scripts/denoise_bench.py [--rounds N] [--warmup W] [--out FILE]
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "scripts"))
PASSES = 16
ITERATIONS = (1, 3, 5)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=10, help="timed rounds per leg")
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()

    import torch
    from chunkyclplugin_b200 import native, scenes as S
    from chunkyclplugin_b200.javarandom import JavaRandom, pass_seeds
    from chunkyclplugin_b200.renderer import upload_scene
    from emitter_models_bench import gpu_info

    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")      # > 126 MB L2
    result = dict(gpu_info(), rounds=args.rounds, warmup=args.warmup, passes_per_window=PASSES, render_kernel=0, sizes={})
    for w, h in ((1920, 1080), (3840, 2160)):
        p = S.terrain_scene(256, w, h)
        ctx = native.Context(0)
        upload_scene(ctx, p)
        ctx.camera_set(p.projector_type, p.camera)
        ctx.render_set_params(kernel=0)
        ctx.render_begin(w, h)
        albedo, normal = ctx.render_features(np.asarray(pass_seeds(PASSES), np.int32))
        rand = JavaRandom(0)
        legs = ["render"] + ["denoise_%d" % k for k in ITERATIONS]
        dev = {k: [] for k in legs}
        e2e = {k: [] for k in legs if k != "render"}
        img = None
        for i in range(args.warmup + args.rounds):
            seeds = np.asarray([rand.next_int() for _ in range(PASSES)], np.int32)
            for leg in legs:
                flush.fill_(i & 0xFF)
                torch.cuda.synchronize()
                if leg == "render":
                    ctx.render_reset_window()
                    ctx.render_passes(seeds)
                    t = None
                    img = ctx.render_read()[0].astype(np.float64)
                else:
                    t0 = time.perf_counter()
                    ctx.denoise(img, albedo, normal, int(leg.split("_")[1]), 4.0, width=w, height=h)
                    t = (time.perf_counter() - t0) * 1e3
                if i >= args.warmup:
                    dev[leg].append(ctx.last_kernel_ms())
                    if t is not None:
                        e2e[leg].append(t)
        ctx.render_end()
        ctx.close()
        stats = lambda v: {"mean": float(np.mean(v)), "min": float(np.min(v)), "max": float(np.max(v))}    # noqa: E731
        result["sizes"]["%dx%d" % (w, h)] = {
            "render_window_device_ms": stats(dev["render"]),
            "render_pass_device_ms": float(np.mean(dev["render"])) / PASSES,
            "denoise": {str(k): {"device_ms": stats(dev["denoise_%d" % k]), "e2e_ms": stats(e2e["denoise_%d" % k]),
                                 "over_render_pass": float(np.mean(dev["denoise_%d" % k]) / (np.mean(dev["render"]) / PASSES))}
                        for k in ITERATIONS},
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
