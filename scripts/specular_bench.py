"""Cost of CCU_RENDER_SPECULAR on BASELINE config 1 (256^3 terrain, 1920 x 1080, 16-pass windows, L2 flushed before each).

Three legs, alternated window by window in one process so that they see the same clocks and neighbours:
  a  config 1, flag off                       (what bench.py times)
  b  config 1, flag on: every word 5 is 0, so the launch picks the same kernel as (a)
  c  config 1 with glossy materials (scenes.glossy), flag on: the specular kernel
Prints one JSON line: the GPU's name and power limit, and per leg the mean / min / max device ms per window and G samples/s.

    python scripts/specular_bench.py [--windows N] [--warmup W] [--kernel 0|1|4] [--out FILE]
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
PASSES = 16


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True, timeout=60).stdout.strip()
        name, power, clock = [x.strip() for x in out.split(",")]
        return {"gpu": name, "power_limit": power, "sm_max_clock": clock}
    except Exception as e:      # the numbers are still measured; say why the card is not named
        return {"gpu": None, "power_limit": None, "error": repr(e)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--windows", type=int, default=20, help="timed windows per leg")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--kernel", type=int, default=0)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()

    import torch
    from chunkyclplugin_b200 import native, scenes as S
    from chunkyclplugin_b200.javarandom import JavaRandom
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    from conftest import load_scene

    plain = S.terrain_scene(256, 1920, 1080)
    glossy = S.glossy(plain)
    ctx_plain, ctx_glossy = native.Context(0), native.Context(0)
    load_scene(ctx_plain, plain)
    load_scene(ctx_glossy, glossy)
    legs = {"a_flag_off": (ctx_plain, 0), "b_flag_on_zero_words": (ctx_plain, native.CCU_RENDER_SPECULAR),
            "c_flag_on_glossy": (ctx_glossy, native.CCU_RENDER_SPECULAR)}
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")      # > 126 MB L2
    rand = JavaRandom(0)
    ms = {k: [] for k in legs}
    for i in range(args.warmup + args.windows):
        seeds = np.asarray([rand.next_int() for _ in range(PASSES)], np.int32)
        for name, (ctx, flags) in legs.items():
            ctx.render_set_params(kernel=args.kernel, flags=flags)
            flush.fill_(i & 0xFF)
            torch.cuda.synchronize()
            ctx.render_reset_window()
            ctx.render_passes(seeds)
            if i >= args.warmup:
                ms[name].append(ctx.last_kernel_ms())
    samples = plain.width * plain.height * PASSES
    result = dict(gpu_info(), workload="config 1 (256^3 terrain, 1920x1080, 16-pass windows, L2 flushed)",
                  kernel=args.kernel, windows=args.windows, warmup=args.warmup,
                  legs={k: {"ms_mean": float(np.mean(v)), "ms_min": float(np.min(v)), "ms_max": float(np.max(v)),
                            "gsamples_per_s": samples / (float(np.mean(v)) * 1e-3) / 1e9} for k, v in ms.items()})
    for ctx in (ctx_plain, ctx_glossy):
        ctx.render_end()
        ctx.close()
    line = json.dumps(result)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")
    return 0


if __name__ == "__main__":
    sys.exit(main())
