#!/usr/bin/env python3
"""Benchmark of the ChunkyCL render path on B200 (contract: see the task statement / DESIGN.md "Measurement").

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload config1|indoor|entities|large]
                  [--dump-outputs DIR]
  python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P bench.py --gpus N ...

A step = one window of SPP_PER_STEP path-tracing passes over the full canvas of the BASELINE config-1 scene (synthetic 256^3
terrain, sun + sky, no entities) on every rank, followed - for N > 1 - by the NCCL reduce-scatter of the per-GPU window
buffers inside libchunkycu.so (weak scaling: per-GPU work is fixed, the N-GPU job renders N x the samples).
`value` is device-timed (CUDA events on the launching stream, max over ranks) with the scene resident in HBM; `e2e` goes
through the host renderer / the library's group API with host buffers (seed upload + read-back + merge into the double
sample buffer inside the timed region).  `--spp-total T --workload large` is the strong-scaling run of BASELINE config 5
(T passes in 1024-pass windows split over the ranks).
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

SPP_PER_STEP = 16
DUMP_LIMIT_BYTES = 64 << 20
METRIC = "path samples/sec"
UNIT = "samples/s"
# The contract line is config1 (the configuration the metric is quoted on that fits one GPU).  --workload selects one of the
# other BASELINE configurations (same JSON shape, named in config.workload); a default N=1 run also times one step of each
# of them (`other_workloads`).
WORKLOADS = {
    "config1": ("config1: synthetic 256^3 terrain octree, 1920x1080, 16 spp per step, sun+sky, no entities (path tracing, max depth 5)", 1920, 1080),
    "indoor": ("config3: 256^3 carved rooms with emissive blocks, sunlight disabled, 1920x1080, 16 spp per step (max depth 5 = 4 bounces)", 1920, 1080),
    "entities": ("config4: config1 terrain + synthetic triangle meshes in world/actor BVHs, 1920x1080, 16 spp per step", 1920, 1080),
    "large": ("config5: 2048x256x2048 world in a depth-11 octree, 3840x2160, 16 spp per step", 3840, 2160),
}
ALG_BYTES_KEYS = {"config1": "terrain256_1080p_bytes_per_sample", "indoor": "indoor256_1080p_bytes_per_sample",
                  "entities": "entities256_1080p_bytes_per_sample", "large": "large2048_4k_bytes_per_sample"}


def config_dict(workload: str, world: int, spp_total: int = 0):
    """The same dict in both arms (ours / reference), so that the driver's same_config check compares like with like."""
    name, _, _ = WORKLOADS[workload]
    d = {"workload": name, "spp_per_step_per_gpu": SPP_PER_STEP, "global_spp_per_step": SPP_PER_STEP * world,
         "parallelism": f"sample-parallel x{world}" + (" + NCCL reduce-scatter per step" if world > 1 else ""),
         "l2": "flushed between timed steps (256 MB write); the scene itself is cache-resident by nature"}
    if spp_total:
        d.update({"spp_per_step_per_gpu": 1024 // world, "global_spp_per_step": 1024, "spp_total": spp_total,
                  "workload": name.replace("16 spp per step", f"{spp_total} spp in 1024-pass windows split over the GPUs")})
    return d


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        return json.load(open(p)), "measured (MEASURED_PEAKS.json)"
    return {"hbm_gbs": 6650.0}, "fallback (B200_PROFILING.md)"


class ClockSampler(threading.Thread):
    """Samples SM clocks / throttle reasons through NVML while the timed region runs."""

    def __init__(self, index: int):
        super().__init__(daemon=True)
        self.index, self.samples, self.reasons, self.stop_flag, self.max_mhz = index, [], set(), False, None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nv = None

    def run(self):
        if self.nv is None:
            return
        nv = self.nv
        names = {
            nv.nvmlClocksThrottleReasonSwPowerCap: "sw_power_cap", nv.nvmlClocksThrottleReasonHwSlowdown: "hw_slowdown",
            nv.nvmlClocksThrottleReasonSwThermalSlowdown: "sw_thermal_slowdown",
            nv.nvmlClocksThrottleReasonHwThermalSlowdown: "hw_thermal_slowdown",
            nv.nvmlClocksThrottleReasonHwPowerBrakeSlowdown: "hw_power_brake", nv.nvmlClocksThrottleReasonSyncBoost: "sync_boost",
        }
        while not self.stop_flag:
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for bit, name in names.items():
                    if r & bit:
                        self.reasons.add(name)
            except Exception:
                pass
            time.sleep(0.05)

    def summary(self):
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": ["nvml unavailable"]}
        return {"sm_mhz": float(np.median(self.samples)), "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons)}


def build_scene(workload: str = "config1"):
    from chunkyclplugin_b200 import scenes as S
    _, w, h = WORKLOADS[workload]
    if workload == "indoor":
        return S.indoor_scene(256, w, h)
    if workload == "entities":
        return S.entity_scene(256, w, h)
    if workload == "large":
        return S.large_world_scene(width=w, height=h)
    return S.terrain_scene(256, w, h)


def cpu_port_rate(scene, seeds, stride: int, threads: int = 0):
    """The oracle (CPU port of the same algorithm, OpenMP over pixels) on a strided pixel subset; returns
    (samples/s, counters, n_samples, cores)."""
    import oracle
    o = oracle.Oracle(scene)
    gids = np.arange(0, scene.width * scene.height, stride, dtype=np.int32)
    t0 = time.perf_counter()
    threads = threads or (os.cpu_count() or 1)          # torchrun exports OMP_NUM_THREADS=1; use every host core anyway
    o.render(seeds, gids=gids, threads=threads)
    dt = time.perf_counter() - t0
    n = gids.size * len(seeds)
    return n / dt, o.last_counters, n, threads


def run_reference(args):
    """--impl reference: the CPU arm.  Chunky's own Java path tracer cannot run here (no JVM, chunky-core not
    vendored), so the reference arm is the oracle port of the same algorithm on all host cores (kind = "port")."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    from chunkyclplugin_b200.javarandom import pass_seeds
    scene = build_scene(args.workload)
    _, width, height = WORKLOADS[args.workload]
    seeds = pass_seeds(SPP_PER_STEP)
    stride = 16 if args.workload != "entities" else 256   # each step = a strided pixel subset of the frame x 16 spp
    rates = []
    for i in range(args.warmup + args.steps):
        rate, counters, n, cores = cpu_port_rate(scene, seeds, stride)
        if i >= args.warmup:
            rates.append((rate, n))
    total = sum(n for _, n in rates)
    secs = sum(n / r for r, n in rates)
    value = total / secs
    sample = f"every {stride}th pixel of the {width}x{height} frame x {SPP_PER_STEP} spp per step ({rates[0][1]} samples/step), OpenMP over pixels"
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * secs / len(rates), "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": config_dict(args.workload, args.gpus),
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
        "note": "Chunky's Java CPU path tracer (the reference's CPU path) needs a JVM + chunky-core, neither available; "
                "this arm times the C port of the reference kernel's algorithm (oracle/) on all host cores",
    }
    # same-box GPU bar: the reference's own OpenCL kernel JIT-compiled by the NVIDIA OpenCL runtime, if present
    try:
        from oracle import clref
        why = clref.available()
        if why is None:
            ref = clref.ClReference(scene, strict=False)
            _, times = ref.render(pass_seeds(SPP_PER_STEP + 4))
            ms = float(np.median(times[4:]))
            fh = ref.first_hit(pass_seeds(1)[0])
            line["opencl_reference_same_gpu"] = {"value": width * height / (ms * 1e-3), "unit": UNIT, "ms_per_pass": ms,
                                                 "first_hit_ms": fh["ms"], "device": ref.device_name(),
                                                 "how": "unmodified reference kernel, one launch per pass, cl_event profiling"}
            ref.close()
        else:
            line["opencl_reference_same_gpu"] = {"unavailable": why}
    except Exception as e:          # never let the extra evidence break the contract line
        line["opencl_reference_same_gpu"] = {"unavailable": repr(e)}
    print(json.dumps(line))
    return 0


class Dist:
    """Host-side plumbing of a one-process-per-GPU job: barriers and max-over-ranks of python floats (gloo).  The data
    plane (reduce-scatter of the window buffers) is NCCL inside libchunkycu.so."""

    def __init__(self):
        self.rank = int(os.environ.get("RANK", "0"))
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.local_rank = int(os.environ.get("LOCAL_RANK", "0"))
        self.dist = None
        if self.world > 1:
            import torch.distributed as dist
            dist.init_process_group("gloo")
            self.dist = dist

    def barrier(self):
        if self.dist:
            self.dist.barrier()

    def max(self, x: float) -> float:
        if not self.dist:
            return x
        import torch
        t = torch.tensor([x], dtype=torch.float64)
        self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return float(t.item())

    def broadcast(self, obj):
        if not self.dist:
            return obj
        box = [obj]
        self.dist.broadcast_object_list(box, src=0)
        return box[0]

    def close(self):
        if self.dist:
            self.dist.destroy_process_group()


def timed_window(ctx, group, seeds, flush, d: Dist):
    """One device-timed step: L2 flush (outside the events), barrier, the window's passes on every GPU [+ reduce-scatter]."""
    import torch
    flush.fill_(d.rank + 1)
    torch.cuda.synchronize()
    d.barrier()
    t0 = time.perf_counter()
    if group is None:
        ctx.render_reset_window()
        ctx.render_passes(np.asarray(seeds, np.int32))
        ms = ctx.last_kernel_ms()
    else:
        group.render_passes(np.asarray(seeds, np.int32))
        group.render_sync()
        group.reduce_only()                      # reduce-scatter of the window, no read-back (device-resident result)
        r_ms, x_ms = group.last_ms()
        ms = r_ms + x_ms
    return ms, (time.perf_counter() - t0) * 1e3


def measure_workload(workload: str, ctx, loader, steps: int, warmup: int, flush, d: Dist, kernel: int):
    """Device-timed steps of one workload on one GPU (used for `other_workloads`)."""
    from chunkyclplugin_b200.javarandom import JavaRandom
    from chunkyclplugin_b200.renderer import Scene
    scene = build_scene(workload)
    _, w, h = WORKLOADS[workload]
    loader.ensureLoad(Scene(scene, target_spp=SPP_PER_STEP))
    commit_ms = ctx.scene_commit_ms()
    ctx.camera_set(scene.projector_type, scene.camera)
    ctx.render_begin(w, h)
    ctx.render_set_params(kernel=kernel)
    rand = JavaRandom(0)
    ms = []
    for i in range(warmup + steps):
        m, _ = timed_window(ctx, None, [rand.next_int() for _ in range(SPP_PER_STEP)], flush, d)
        if i >= warmup:
            ms.append(m)
    ctx.render_end()
    t = float(np.mean(ms))
    return {"workload": WORKLOADS[workload][0], "value": w * h * SPP_PER_STEP / (t * 1e-3), "unit": UNIT, "ms_per_step": t,
            "steps": steps, "warmup": warmup, "scene_commit_ms": commit_ms, "scene_device_bytes": ctx.scene_device_bytes()}


def dump_window(ctx, out_dir: str, width: int, height: int):
    """What a caller of the timed path receives after the last step: the window's mean RGB (ccu_render_read), float32
    [rows, width, 3].  Frames above DUMP_LIMIT_BYTES keep every k-th row (the smallest k that fits)."""
    img, _ = ctx.render_read()
    img = img.reshape(height, width, 3)
    k = -(-img.nbytes // DUMP_LIMIT_BYTES)
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "window_rgb.npy"), np.ascontiguousarray(img[::k]))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--kernel", type=int, default=0, help="0 auto, 1 thread-per-pixel, 4 persistent wavefront")
    ap.add_argument("--workload", default="config1", choices=sorted(WORKLOADS))
    ap.add_argument("--spp-total", type=int, default=0, help="strong scaling: render this many passes in 1024-pass windows split over the GPUs")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-other-workloads", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps, write the last step's output to DIR/window_rgb.npy")
    args = ap.parse_args()
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup
    if args.impl == "reference":
        return run_reference(args)
    workload_name, WIDTH, HEIGHT = WORKLOADS[args.workload]

    import torch
    from chunkyclplugin_b200 import native
    from chunkyclplugin_b200.javarandom import JavaRandom
    from chunkyclplugin_b200.multigpu import SampleParallelRenderer, SharedSampleBuffer, join_process_group
    from chunkyclplugin_b200.renderer import (CudaPathTracingRenderer, CudaSceneLoader, DefaultRenderManager, RendererInstance, Scene)

    d = Dist()
    rank, world, local_rank = d.rank, d.world, d.local_rank
    if world != args.gpus and world == 1 and args.gpus > 1:
        print(f"bench.py: --gpus {args.gpus} needs torchrun with {args.gpus} ranks", file=sys.stderr)
        return 2
    if args.dump_outputs and world > 1:
        print("bench.py: --dump-outputs needs a single-GPU run (each rank holds only its share of the reduced window)", file=sys.stderr)
        return 2
    torch.cuda.set_device(local_rank)

    scene = build_scene(args.workload)
    inst = RendererInstance.get(local_rank)
    ctx = inst.context
    loader = CudaSceneLoader(inst)
    chunky_scene = Scene(scene, target_spp=SPP_PER_STEP)
    loader.ensureLoad(chunky_scene)
    commit_ms = ctx.scene_commit_ms()
    ctx.render_set_params(kernel=args.kernel)
    group = None
    if world > 1:
        group = join_process_group(ctx, rank, world)      # NCCL communicator inside the library
        group.camera_set(scene.projector_type, scene.camera)
        group.render_begin(WIDTH, HEIGHT)
    else:
        ctx.camera_set(scene.projector_type, scene.camera)
        ctx.render_begin(WIDTH, HEIGHT)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")      # > 126 MB L2
    rand = JavaRandom(0)
    strong = args.spp_total > 0
    window = 1024 if strong else SPP_PER_STEP * world       # global passes per step
    if strong:
        args.steps = max(1, args.spp_total // window)

    def step_seeds(n=None):
        return [rand.next_int() for _ in range(n or window)]

    launches0 = ctx.launch_count()
    for _ in range(args.warmup):
        timed_window(ctx, group, step_seeds(SPP_PER_STEP * world), flush, d)
    launches_w = ctx.launch_count()
    sampler = ClockSampler(local_rank)
    sampler.start()
    torch.cuda.synchronize()
    d.barrier()
    dev_ms, wall_ms = [], []
    for _ in range(args.steps):
        ms, wall = timed_window(ctx, group, step_seeds(), flush, d)
        dev_ms.append(ms)
        wall_ms.append(wall)
    torch.cuda.synchronize()
    d.barrier()
    sampler.stop_flag = True
    sampler.join()
    launches = ctx.launch_count() - launches_w
    if args.dump_outputs:
        dump_window(ctx, args.dump_outputs, WIDTH, HEIGHT)
    total_ms = d.max(float(sum(dev_ms)))
    samples_per_step = WIDTH * HEIGHT * window
    value = samples_per_step * args.steps / (total_ms * 1e-3)

    # ---- first-hit pass (BASELINE config 2): primary-ray Mrays/s on the same scene ----------------------------
    fh_ms = None
    if rank == 0:
        ts = []
        lib = native.load()
        for i in range(6):
            flush.fill_(i)
            torch.cuda.synchronize()
            native.check(lib.ccu_first_hit(ctx._h, 12345 + i, None, None, None, None, None, None, None))
            ts.append(ctx.last_kernel_ms())
        fh_ms = float(np.median(ts[2:]))

    # ---- memory-system denominators of this path (SURVEY 8d): random 32-byte-sector gathers, L2- and HBM-resident --------
    memsys = None
    if rank == 0:
        l2_bw, _ = ctx.bench_gather(4 << 20)
        hbm_bw, _ = ctx.bench_gather(1 << 30)
        _, l2_ns = ctx.bench_gather(4 << 20, dependent=True)
        _, hbm_ns = ctx.bench_gather(1 << 30, dependent=True)
        memsys = {"l2_random_sector_gbs": l2_bw, "hbm_random_sector_gbs": hbm_bw, "l2_dependent_gather_ns": l2_ns,
                  "hbm_dependent_gather_ns": hbm_ns,
                  "how": "ccu_bench_gather: random 16-byte ld.global.cg per 32-byte sector over a 4 MiB / 1 GiB array, all SMs"}

    # ---- end to end through the public API: seeds H2D + read-back + merge into the host double buffer, every step -----
    e_steps = args.steps
    n_floats = WIDTH * HEIGHT * 3
    if world == 1:
        # CudaPathTracingRenderer.render() exactly as Chunky drives it: ONE render of e_steps windows; every window = 16
        # passes (one C-ABI call), closed by ccu_render_merge_async, whose read-back + merge overlaps the next window's passes
        ctx.render_end()
        renderer = CudaPathTracingRenderer(loader, merge_window=window, passes_per_call=window)
        warm = Scene(scene, target_spp=3 * SPP_PER_STEP)
        warm.packed = scene
        renderer.render(DefaultRenderManager(warm))
        cs = Scene(scene, target_spp=window * e_steps)
        cs.packed = scene                                  # same scene object: no re-upload
        flush.fill_(7)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        renderer.render(DefaultRenderManager(cs))          # render_begin, e_steps x (passes + merge), render_end
        e_secs = time.perf_counter() - t0
        assert cs.spp == window * e_steps and cs.sample_buffer.max() > 0 and cs.post_process_calls == e_steps
        e_how = "one CudaPathTracingRenderer.render() of %d windows: per window one ccu_render_passes (16 seeds H2D) + ccu_render_merge_async (float window D2H + merge into the host double buffer, overlapped with the next window)" % e_steps
    else:
        # N GPUs: per step every rank queues its passes, then the collective ccu_group_render_merge: reduce-scatter over NVLink,
        # every GPU reads its share back over its own PCIe link and merges it into the shared-memory sample buffer
        name = d.broadcast(f"ccu_bench_{os.getpid()}" if rank == 0 else None)
        sb = SharedSampleBuffer(n_floats, name=name, create=True) if rank == 0 else None
        d.barrier()
        if rank != 0:
            sb = SharedSampleBuffer(n_floats, name=name, create=False)
        spr = SampleParallelRenderer(group)
        spp = 0
        for i in range(2):
            spp += spr.render_and_merge(step_seeds(SPP_PER_STEP * world), sb.array, spp)
        flush.fill_(7)
        torch.cuda.synchronize()
        d.barrier()
        t0 = time.perf_counter()
        for i in range(e_steps):
            spp += spr.render_and_merge(step_seeds(), sb.array, spp, overlap=True)    # the share merge overlaps the next window's passes
        spr.finish()
        d.barrier()
        e_secs = time.perf_counter() - t0
        assert sb.array.max() > 0
        e_how = "per step: ccu_group_render_passes (seeds H2D on every rank) + ccu_group_render_merge_async (NCCL reduce-scatter, per-GPU share D2H + merge into the shared host double buffer, overlapped with the next step)"
    e_secs = d.max(e_secs)
    e2e = {"value": WIDTH * HEIGHT * window * e_steps / e_secs, "unit": UNIT, "h2d_bytes_per_step": 4 * window,
           "d2h_bytes_per_step": 4 * n_floats, "steps": e_steps, "how": e_how}

    if rank != 0:
        if world > 1:
            sb.close()
            group.render_end()
            group.close()
        d.close()
        return 0

    # ---- other BASELINE configurations: one short device-timed measurement each (N = 1 default run only) -----------
    others = None
    if world == 1 and args.workload == "config1" and not args.no_other_workloads and not strong:
        others = {}
        for wl in ("indoor", "entities", "large"):
            try:
                others[wl] = measure_workload(wl, ctx, loader, steps=3, warmup=1, flush=flush, d=d, kernel=args.kernel)
            except Exception as e:      # never let the extra evidence break the contract line
                others[wl] = {"error": repr(e)}

    # ---- CPU baseline + algorithmic bytes (bounded sample of the same workload) ---------------------------------
    peaks, peak_src = measured_peaks()
    cpu = None
    bytes_per_sample = None
    if not args.no_cpu_baseline:
        import oracle
        from chunkyclplugin_b200.javarandom import pass_seeds
        stride = 8 if args.workload != "entities" else 128
        rate, counters, n, cores = cpu_port_rate(scene, pass_seeds(SPP_PER_STEP), stride)
        bytes_per_sample = oracle.algorithmic_bytes(counters) / counters["samples"]
        cpu = {"value": rate, "unit": UNIT, "cores": cores, "kind": "port",
               "sample": f"every {stride}th pixel of the {WIDTH}x{HEIGHT} frame x {SPP_PER_STEP} spp ({n} samples), oracle C port, OpenMP"}
    else:
        alg = os.path.join(ROOT, "profiles", "alg_bytes.json")
        if os.path.exists(alg):
            bytes_per_sample = json.load(open(alg)).get(ALG_BYTES_KEYS[args.workload])
    kernel_ms = float(np.mean(dev_ms))
    roofline = None
    if bytes_per_sample and memsys:
        achieved = bytes_per_sample * samples_per_step / world / (kernel_ms * 1e-3) / 1e9      # per GPU
        # SURVEY 8d: the scene is cache-resident, the bound of this path is the random-sector bandwidth of the L2 (configs 1-4);
        # the fraction of the nominal HBM copy bandwidth is kept beside it
        l2 = memsys["l2_random_sector_gbs"]
        roofline = {"bound": "l2_random_sector", "achieved": achieved, "peak": l2, "unit": "GB/s", "frac": achieved / l2,
                    "peak_source": "ccu_bench_gather in this run (random 32-byte sectors, 4 MiB array, all SMs)",
                    "frac_hbm_nominal": achieved / peaks["hbm_gbs"], "peak_hbm_gbs": peaks["hbm_gbs"], "peak_hbm_source": peak_src,
                    "traffic": None, "algorithmic_bytes_per_sample": bytes_per_sample,
                    "kernel": "k_render_queue, one launch per window", "kernel_ms": kernel_ms,
                    "note": "algorithmic bytes follow the reference's root descent per march step (SURVEY 8d); this kernel reads far fewer "
                            "(commit-time layouts) and is limited by instruction issue and dependent-gather latency - see profiles/"}
        ncu_file = os.path.join(ROOT, "profiles", "r02_queue_ncu_metrics.json")
        if os.path.exists(ncu_file):
            m = json.load(open(ncu_file))
            roofline["traffic"] = m.get("dram_bytes_per_launch")
            roofline["traffic_source"] = m.get("source")
            roofline["lane_efficiency"] = m.get("lane_efficiency")
            roofline["warp_inst_per_sample"] = m.get("warp_inst_per_sample")

    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": total_ms / args.steps, "higher_is_better": True, "scaling": "strong" if strong else "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic",
        "config": config_dict(args.workload, world, args.spp_total),
        "clocks": sampler.summary(),
        "e2e": e2e, "gpu_launches": int(launches),
        "roofline": roofline, "cpu_baseline": cpu,
        "primary_rays": {"value": WIDTH * HEIGHT / (fh_ms * 1e-3) / 1e6, "unit": "Mrays/s", "ms": fh_ms,
                         "workload": "config2: first-hit pass, same scene and canvas"} if fh_ms else None,
        "memory_system": memsys,
        "scene_commit_ms": commit_ms, "scene_device_bytes": ctx.scene_device_bytes(),
        "other_workloads": others,
        "wall_ms_per_step": float(np.mean(wall_ms)),
    }
    print(json.dumps(line))
    if world > 1:
        sb.close()
        group.render_end()
        group.close()
    d.close()
    return 0


if __name__ == "__main__":
    sys.exit(main())
