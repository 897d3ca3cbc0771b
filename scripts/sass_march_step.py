"""Size of the octree march step of the default wavefront kernel, from its SASS (no GPU needed).

Compiles k_render_queue<false, 0, PlainShade> (no BVHs, top table in shared memory, no render flags) from the
headers under chunkyclplugin_b200/csrc with the library's nvcc flags, finds the inner march loop - the smallest loop,
closed by a backward branch, whose body holds the brick load (LDG) and the three F2I.FLOOR of the voxel coordinates - and
prints its instruction count with the kernel's registers and spill bytes.

    python scripts/sass_march_step.py            # human-readable
    python scripts/sass_march_step.py --json     # one JSON line
    python scripts/sass_march_step.py --print    # also the loop's SASS
"""
from __future__ import annotations

import argparse
import json
import os
import re
import shutil
import subprocess
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from chunkyclplugin_b200.build import CSRC, NVCC_FLAGS  # noqa: E402

KERNEL = "k_render_queue<false, 0, PlainShade>"
INSN = re.compile(r"^\s*/\*([0-9a-f]{4,})\*/\s+(.*?)\s*;")


def compile_kernel(tmp: str) -> tuple[str, str]:
    """Build a cubin holding just the default kernel; return (cubin path, ptxas -v output)."""
    src = os.path.join(tmp, "march_step.cu")
    with open(src, "w") as f:
        f.write('#include "ccu_queue.cuh"\n'
                f"namespace ccu {{ void *march_step_kernel() {{ return (void *)&{KERNEL}; }} }}\n")
    flags = [f for f in NVCC_FLAGS if f not in ("-shared", "-cudart", "static", "--threads", "2", "-Xcompiler", "-fPIC")]
    cubin = os.path.join(tmp, "march_step.cubin")
    nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    r = subprocess.run([nvcc] + flags + ["-I", CSRC, "-cubin", "-Xptxas", "-v", "-o", cubin, src], capture_output=True, text=True)
    if r.returncode != 0:
        raise SystemExit("nvcc failed:\n" + r.stdout + r.stderr)
    return cubin, r.stderr


def resources(ptxas: str) -> tuple[int, int]:
    """(registers, spill store bytes) of the k_render_queue entry in ptxas -v output."""
    lines = ptxas.splitlines()
    for i, l in enumerate(lines):
        if "Compiling entry function" in l and "k_render_queue" in l:
            spill = regs = None
            for m in lines[i + 1:i + 6]:
                s = re.search(r"(\d+) bytes spill stores", m)
                if s:
                    spill = int(s.group(1))
                g = re.search(r"Used (\d+) registers", m)
                if g:
                    regs = int(g.group(1))
            if regs is not None and spill is not None:
                return regs, spill
    raise SystemExit("no ptxas resource line for k_render_queue")


def march_loop(sass: str) -> list[tuple[int, str]]:
    insns = [(int(m.group(1), 16), m.group(2)) for m in map(INSN.match, sass.splitlines()) if m]
    at = {a: i for i, (a, _) in enumerate(insns)}
    best = None
    for j, (a, text) in enumerate(insns):
        m = re.search(r"\bBRA\b.*0x([0-9a-f]+)\s*$", text)
        if not m or int(m.group(1), 16) >= a or int(m.group(1), 16) not in at:
            continue
        body = insns[at[int(m.group(1), 16)]:j + 1]
        ops = [t.split()[1] if t.startswith("@") else t.split()[0] for _, t in body]
        if sum(o.startswith("F2I.FLOOR") for o in ops) >= 3 and any(o.startswith("LDG") for o in ops):
            if best is None or len(body) < len(best):
                best = body
    if best is None:
        raise SystemExit("march loop not found")
    return best


def main() -> None:
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--json", action="store_true", help="print one JSON line")
    ap.add_argument("--print", action="store_true", help="print the loop's instructions")
    a = ap.parse_args()
    with tempfile.TemporaryDirectory() as tmp:
        cubin, ptxas = compile_kernel(tmp)
        cuobjdump = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"
        sass = subprocess.run([cuobjdump, "-sass", cubin], capture_output=True, text=True, check=True).stdout
    regs, spill = resources(ptxas)
    loop = march_loop(sass)
    res = {"kernel": KERNEL, "march_loop_insns": len(loop), "first": f"{loop[0][0]:04x}", "last": f"{loop[-1][0]:04x}",
           "registers": regs, "spill_store_bytes": spill}
    if a.print:
        for addr, text in loop:
            print(f"/*{addr:04x}*/  {text}")
    if a.json:
        print(json.dumps(res))
    else:
        print(f"{KERNEL}: march loop {res['first']}..{res['last']} = {len(loop)} instructions, "
              f"{regs} registers, {spill} bytes spilled")


if __name__ == "__main__":
    main()
