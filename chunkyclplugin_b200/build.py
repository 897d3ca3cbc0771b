"""Ahead-of-time build of libchunkycu.so for sm_100a (replaces the reference's runtime JIT, KernelLoader.java:17-60)."""
from __future__ import annotations

import os
import shutil
import subprocess
import sys
import tempfile
from concurrent.futures import ThreadPoolExecutor

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(HERE, "libchunkycu.so")

NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-O3", "-lineinfo", "-std=c++17",
    # arithmetic contract (DESIGN.md): no contraction, IEEE division / sqrt, denormals kept
    "-fmad=false", "-prec-div=true", "-prec-sqrt=true", "-ftz=false",
    "-Xcompiler", "-fPIC",
]
LINK_FLAGS = ["-ldl"]   # NCCL is bound at run time (ccu_group.cu)


def sources():
    return [os.path.join(CSRC, f) for f in sorted(os.listdir(CSRC)) if f.endswith(".cu")]


def needs_build() -> bool:
    if not os.path.exists(LIB):
        return True
    t = os.path.getmtime(LIB)
    deps = [os.path.join(CSRC, f) for f in os.listdir(CSRC)] + [os.path.join(os.path.dirname(HERE), "include", "chunkycu.h")]
    return any(os.path.getmtime(d) > t for d in deps)


def build(force: bool = False, verbose: bool = False) -> str:
    """Compiles every translation unit of csrc/ in parallel (the render-kernel instances are spread over several units,
    ccu_render.cuh), then links them into LIB.  The objects go to a temporary directory."""
    if not force and not needs_build():
        return LIB
    nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    extra = os.environ.get("CCU_NVCC_EXTRA", "").split()
    flags = [nvcc] + NVCC_FLAGS + extra + (["-Xptxas", "-v"] if verbose else [])
    srcs = sources()
    # largest units first, so that the longest compiles start at once
    srcs.sort(key=lambda f: -os.path.getsize(f))
    with tempfile.TemporaryDirectory(prefix="ccu_build_") as tmp:
        def compile_one(src):
            obj = os.path.join(tmp, os.path.basename(src) + ".o")
            cmd = flags + ["-c", "-o", obj, src]
            return cmd, obj, subprocess.run(cmd, capture_output=True, text=True)
        with ThreadPoolExecutor(max_workers=max(1, os.cpu_count() or 1)) as pool:
            results = list(pool.map(compile_one, srcs))
        log = []
        for cmd, _, r in results:
            if r.returncode != 0:
                raise RuntimeError("nvcc failed:\n" + " ".join(cmd) + "\n" + r.stdout + r.stderr)
            log.append(r.stderr)
        objs = [obj for _, obj, _ in results]
        cmd = [nvcc, "-gencode", "arch=compute_100a,code=sm_100a", "-shared", "-cudart", "static", "-o", LIB] + extra + objs + LINK_FLAGS
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError("nvcc link failed:\n" + " ".join(cmd) + "\n" + r.stdout + r.stderr)
    if verbose:
        print("".join(log))
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
