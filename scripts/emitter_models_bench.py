"""Cost and gain of CCU_RENDER_EMITTER_MODELS (DESIGN §12) on the two model-lit variants of scenes.py at 1920 x 1080: config 3
lit by torches and lanterns only (indoor_models_scene(256), sun off), and config 1 with decorations whose CROSS (quad) and SLAB
(AABB) blocks are made emissive (emissive_models, sun on), so that cube and model emitters share the lists.

Per config, three legs on kernel 0 (the wavefront kernel, what bench.py times) alternated window by window in one process
(16-pass windows, L2 flushed before each): `off` with the flags off, `on` with CCU_RENDER_EMITTER_SAMPLING |
CCU_RENDER_EMITTER_MODELS and `near` with CCU_RENDER_EMITTER_NEAR_FIELD added.  Then the gain: RMSE of a K-pass
render of each leg against a --ref-spp flag-off render on a disjoint seed stream, for each K of --spp.  For an unbiased
estimator the RMSE falls as 1 / sqrt(K) (variance, not bias): `rmse_ratio_hi_lo` compares the RMSE at the largest K with the
RMSE at the smallest, against the 1 / sqrt ratio.  At equal device time the flag-off kernel renders t_on / t_off times the
passes, so its RMSE becomes rmse(off) * sqrt(t_off / t_on); `equal_time_ratio` divides the `on` RMSE by that, and
`equal_time_ratio_near` the `near` RMSE by the same with t_near.  The
per-pixel median absolute error is reported beside the RMSE (robust to a few very bright pixels).  Also the commit times of
configs 1, 3, 4 and 5, which have no model emitter, with whether the model table was built (it must not be).  Prints one JSON
line with the GPU's name, power limit and SM clock.

    python scripts/emitter_models_bench.py [--windows N] [--warmup W] [--spp K1 K2 ..] [--ref-spp R] [--out FILE]
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
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.sm,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True, timeout=60).stdout.strip()
        name, power, clock, max_clock = [x.strip() for x in out.split(",")]
        return {"gpu": name, "power_limit": power, "sm_clock": clock, "sm_max_clock": max_clock}
    except Exception as e:      # the numbers are still measured; say why the card is not named
        return {"gpu": None, "power_limit": None, "error": repr(e)}


def render(ctx, p, seeds, kernel, flags):
    ctx.render_set_params(kernel=kernel, flags=flags)
    ctx.render_begin(p.width, p.height)
    for i in range(0, len(seeds), 256):
        ctx.render_passes(np.asarray(seeds[i:i + 256], np.int32))
    img = ctx.render_read()[0].astype(np.float64)
    ctx.render_end()
    return img


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--windows", type=int, default=12, help="timed windows per leg")
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--spp", type=int, nargs="+", default=[64, 256])
    ap.add_argument("--ref-spp", type=int, default=4096)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()

    import torch
    from chunkyclplugin_b200 import native, scenes as S
    from chunkyclplugin_b200.javarandom import JavaRandom
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    from conftest import load_scene

    NEE = native.CCU_RENDER_EMITTER_SAMPLING | native.CCU_RENDER_EMITTER_MODELS
    legs = {"off": (0, 0), "on": (0, NEE), "near": (0, NEE | native.CCU_RENDER_EMITTER_NEAR_FIELD)}
    configs = {"config3_models256": S.indoor_models_scene(256, 1920, 1080),
               "config1_decorated_lit_models": S.emissive_models(S.terrain_scene(256, 1920, 1080, decorate=True))}
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")      # > 126 MB L2
    result = dict(gpu_info(), windows=args.windows, warmup=args.warmup, passes_per_window=PASSES, spp=args.spp,
                  ref_spp=args.ref_spp, configs={})
    for cname, p in configs.items():
        ctx = native.Context(0)
        load_scene(ctx, p)
        rand = JavaRandom(0)
        ms = {k: [] for k in legs}
        for i in range(args.warmup + args.windows):
            seeds = np.asarray([rand.next_int() for _ in range(PASSES)], np.int32)
            for name, (kernel, flags) in legs.items():
                ctx.render_set_params(kernel=kernel, flags=flags)
                flush.fill_(i & 0xFF)
                torch.cuda.synchronize()
                ctx.render_reset_window()
                ctx.render_passes(seeds)
                if i >= args.warmup:
                    ms[name].append(ctx.last_kernel_ms())
        ctx.render_end()
        rr = JavaRandom(12345)
        ref = render(ctx, p, [rr.next_int() for _ in range(args.ref_spp)], 0, 0)
        rs = JavaRandom(777)
        seeds = [rs.next_int() for _ in range(max(args.spp))]
        err = {k: {} for k in legs}
        for k, (kernel, flags) in legs.items():
            for spp in args.spp:
                e = np.abs(render(ctx, p, seeds[:spp], kernel, flags) - ref)
                err[k][spp] = {"rmse": float(np.sqrt((e ** 2).mean())), "median_abs": float(np.median(e))}
        commit_ms = ctx.scene_commit_ms()
        ctx.close()
        per_pass = {k: float(np.mean(v)) / PASSES for k, v in ms.items()}
        lo, hi = min(args.spp), max(args.spp)
        result["configs"][cname] = {
            "commit_ms": commit_ms,
            "legs": {k: {"ms_per_window_mean": float(np.mean(v)), "ms_min": float(np.min(v)), "ms_max": float(np.max(v)),
                         "ms_per_pass": per_pass[k], "error": {str(n): e for n, e in err[k].items()},
                         "rmse_ratio_hi_lo": err[k][hi]["rmse"] / err[k][lo]["rmse"], "rmse_ratio_if_variance": float(np.sqrt(lo / hi))}
                     for k, v in ms.items()},
            "equal_time_ratio": {str(n): err["on"][n]["rmse"] / (err["off"][n]["rmse"] * float(np.sqrt(per_pass["off"] / per_pass["on"])))
                                 for n in args.spp},
            "equal_time_ratio_near": {str(n): err["near"][n]["rmse"] / (err["off"][n]["rmse"] * float(np.sqrt(per_pass["off"] / per_pass["near"])))
                                      for n in args.spp},
        }
    result["commit_without_model_emitters"] = {}
    for cname, make in (("config1", lambda: S.terrain_scene(256, 1920, 1080)), ("config3", lambda: S.indoor_scene(256, 1920, 1080)),
                        ("config4", lambda: S.entity_scene(256, 1920, 1080)), ("config5", S.large_world_scene)):
        p = make()
        ctx = native.Context(0)
        load_scene(ctx, p)
        result["commit_without_model_emitters"][cname] = {"commit_ms": ctx.scene_commit_ms(),
                                                          "model_table": native.debug_emitter_models(p)["has_emitters"]}
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
