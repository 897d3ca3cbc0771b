"""The octree march step of the default wavefront kernel stays within its instruction budget (compiled here, no GPU needed)."""
import json
import os
import shutil
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.mark.skipif(shutil.which("nvcc") is None and not os.path.exists("/usr/local/cuda/bin/nvcc"), reason="needs nvcc")
def test_march_step_instruction_budget():
    r = subprocess.run([sys.executable, os.path.join(ROOT, "scripts", "sass_march_step.py"), "--json"],
                       capture_output=True, text=True, check=True)
    res = json.loads(r.stdout.strip().splitlines()[-1])
    assert res["march_loop_insns"] <= 75, res
    assert res["registers"] <= 72, res          # one 896-thread CTA per SM
    assert res["spill_store_bytes"] <= 32, res
