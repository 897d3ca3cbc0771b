"""Cost of CCU_RENDER_CLOUDS (DESIGN §15): config 1 at 1920 x 1080 and config 3 (the 256^3 carved rooms) at 1920 x 1080, both
with the sun on, under a Minecraft-like cloud layer: 12-block cells, about a third of them set, 4 blocks thick at y = 192.

Per config, two legs on kernel 0 (the wavefront kernel, what bench.py times) alternated window by window in one process
(16-pass windows, L2 flushed before each): `off` with the flags off and `on` with CCU_RENDER_CLOUDS, on the same committed scene
with clouds.  Then bench.py in the same session (--bench-steps, 0 = skip): its flag-off result, which shows the default path
unchanged.  Prints one JSON line with the GPU's name, power limit and SM clock, read before the legs and again after bench.py.

    python scripts/clouds_bench.py [--windows N] [--warmup W] [--bench-steps S] [--out FILE]
"""
from __future__ import annotations

import argparse
import dataclasses
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "scripts"))
PASSES = 16
LAYER = dict(size=12.0, y0=192.0, y1=196.0, u0=0.37, v0=-0.21)   # ccu_scene_set_clouds arguments after the mask
COVER = 0.35


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--windows", type=int, default=8, help="timed windows per leg")
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--bench-steps", type=int, default=20, help="steps of the bench.py run (0: no bench.py run)")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()

    import torch
    from chunkyclplugin_b200 import native, scenes as S
    from chunkyclplugin_b200.javarandom import JavaRandom
    from chunkyclplugin_b200.renderer import upload_scene
    from emitter_models_bench import gpu_info

    def sun_on(p):
        sun = p.sun.copy()
        sun[0] |= 1
        return dataclasses.replace(p, sun=sun)

    legs = {"off": 0, "on": native.CCU_RENDER_CLOUDS}
    configs = {"config1_1080p": lambda: S.terrain_scene(256, 1920, 1080), "config3_1080p": lambda: S.indoor_scene(256, 1920, 1080)}
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")      # > 126 MB L2
    result = dict(gpu_info(), windows=args.windows, warmup=args.warmup, passes_per_window=PASSES, kernel=0, layer=dict(LAYER, cover=COVER),
                  configs={})
    for cname, make in configs.items():
        p = S.with_clouds(sun_on(make()), S.cloud_mask(seed=1, cover=COVER), **LAYER)
        ctx = native.Context(0)
        upload_scene(ctx, p)
        ctx.camera_set(p.projector_type, p.camera)
        ctx.render_begin(p.width, p.height)
        rand = JavaRandom(0)
        ms = {k: [] for k in legs}
        ran = {}
        for i in range(args.warmup + args.windows):
            seeds = np.asarray([rand.next_int() for _ in range(PASSES)], np.int32)
            for name, flags in legs.items():
                ctx.render_set_params(kernel=0, flags=flags)
                flush.fill_(i & 0xFF)
                torch.cuda.synchronize()
                ctx.render_reset_window()
                ctx.render_passes(seeds)
                ran[name] = ctx.last_render_n(9)
                if i >= args.warmup:
                    ms[name].append(ctx.last_kernel_ms())
        ctx.render_end()
        ctx.close()
        result["configs"][cname] = {
            "width": p.width, "height": p.height,
            "instance": {k: list(v) for k, v in ran.items()},
            "legs": {k: {"ms_per_window_mean": float(np.mean(v)), "ms_min": float(np.min(v)), "ms_max": float(np.max(v)),
                         "ms_per_pass": float(np.mean(v)) / PASSES} for k, v in ms.items()},
            "on_over_off": float(np.mean(ms["on"]) / np.mean(ms["off"])),
        }
    if args.bench_steps > 0:
        del flush
        torch.cuda.empty_cache()
        cmd = [sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--steps", str(args.bench_steps), "--warmup", "3"]
        out = subprocess.run(cmd, capture_output=True, text=True, cwd=ROOT, check=True).stdout
        b = json.loads([l for l in out.splitlines() if l.startswith("{")][-1])
        result["bench_py"] = dict(gpu_info(), command=" ".join(["bench.py"] + cmd[2:]), ms_per_step=b["ms_per_step"],
                                  value=b["value"], unit=b["unit"], clocks=b.get("clocks"))
    line = json.dumps(result)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")
    return 0


if __name__ == "__main__":
    sys.exit(main())
