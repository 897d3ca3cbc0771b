"""bench.py contract: the reference arm runs without a GPU and prints one JSON line with the agreed keys; the GPU arm's
line is checked on the GPU box."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

import oracle
from chunkyclplugin_b200 import scenes
from chunkyclplugin_b200.javarandom import JavaRandom

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BASE_KEYS = {"metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline",
             "dtype", "data", "config", "e2e", "cpu_baseline"}


def _run(args, timeout=600):
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + args, capture_output=True, text=True, timeout=timeout, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1, r.stdout[-2000:]
    return json.loads(lines[0])


def test_reference_arm_line():
    d = _run(["--impl", "reference", "--steps", "1", "--warmup", "0"])
    assert d["impl"] == "reference" and BASE_KEYS <= set(d)
    assert d["metric"] == "path samples/sec" and d["unit"] == "samples/s" and d["higher_is_better"] is True
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["value"] == d["value"]
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert "workload" in d["config"] and d["value"] > 0 and d["vs_baseline"] is None


def test_reference_arm_other_ranks_stay_silent():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2", "--steps", "1", "--warmup", "0"],
                       capture_output=True, text=True, timeout=120, cwd=ROOT, env=env)
    assert r.returncode == 0 and r.stdout.strip() == ""


@pytest.mark.gpu
def test_gpu_arm_line(tmp_path):
    d = _run(["--steps", "2", "--warmup", "3", "--no-other-workloads", "--dump-outputs", str(tmp_path)])
    assert BASE_KEYS | {"roofline", "clocks", "gpu_launches", "primary_rays", "memory_system"} <= set(d)
    assert d["gpu_launches"] >= 2 and d["n_gpus"] == 1 and d["dtype"] == "f32" and d["data"] == "synthetic"
    rf = d["roofline"]
    assert rf["bound"] == "l2_random_sector" and rf["unit"] == "GB/s" and abs(rf["frac"] - rf["achieved"] / rf["peak"]) < 1e-9
    assert 0 < rf["frac_hbm_nominal"] < rf["frac"] * 2 and d["scene_commit_ms"] > 0
    e = d["e2e"]
    assert e["h2d_bytes_per_step"] > 0 and e["d2h_bytes_per_step"] == 4 * 3 * 1920 * 1080 and 0 < e["value"] <= d["value"] * 1.05
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["value"] > 0
    assert d["clocks"]["sm_mhz"] and not set(d["clocks"]["reasons"]) & {"hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown"}
    assert d["steps"] == 2 and e["steps"] == 2
    # the dump is the last timed window: the fifth 16-pass window of JavaRandom(0) (3 warm-up + 2 timed steps)
    img = np.load(tmp_path / "window_rgb.npy")
    assert img.dtype == np.float32 and img.shape == (1080, 1920, 3)
    r = JavaRandom(0)
    seeds = [r.next_int() for _ in range(5 * 16)][4 * 16:]
    gids = np.arange(5, 1920 * 1080, 4099, dtype=np.int32)
    ref = oracle.Oracle(scenes.terrain_scene(256, 1920, 1080)).render(seeds, gids=gids).reshape(-1, 3)
    assert np.array_equal(img.reshape(-1, 3)[gids].view(np.uint32), ref[gids].view(np.uint32))
