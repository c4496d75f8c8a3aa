"""Builds ``lib/libagym_b200.so`` in-tree with nvcc for sm_100a.

    python -m active_gym_b200.build [--force]

nvcc cross-compiles without a GPU.  The .so is git-ignored but travels with the working tree.
"""
from __future__ import annotations

import os
import shutil
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
OUT = os.path.join(HERE, "lib", "libagym_b200.so")
SOURCES = ["agym_ingest.cu", "agym_ingest_std.cu", "agym_observe.cu", "agym_flexible.cu", "agym_memory.cu", "agym_misc.cu", "agym_abi.cu", "agym_tables.cpp"]
HEADERS = ["agym_kernels.cuh", "agym_device.cuh", "agym_tables.h", os.path.join("..", "..", "include", "agym_b200.h")]
NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
    "-Xcompiler", "-fPIC,-fvisibility=hidden", "-shared",
]


def _nvcc() -> str:
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found")


def needs_build() -> bool:
    if not os.path.exists(OUT):
        return True
    t = os.path.getmtime(OUT)
    return any(os.path.getmtime(os.path.join(CSRC, f)) > t for f in SOURCES + HEADERS)


def build(force: bool = False, verbose: bool = False) -> str:
    if not force and not needs_build():
        return OUT
    os.makedirs(os.path.dirname(OUT), exist_ok=True)
    objdir = os.path.join(HERE, "lib", "obj")
    os.makedirs(objdir, exist_ok=True)
    # AGYM_NVCC_EXTRA: extra compiler flags (-D tuning switches) for timing experiments
    compile_flags = [f for f in NVCC_FLAGS if f != "-shared"] + (["-Xptxas", "-v"] if verbose else []) + os.environ.get("AGYM_NVCC_EXTRA", "").split()

    def compile_one(src: str):
        obj = os.path.join(objdir, os.path.splitext(src)[0] + ".o")
        cmd = [_nvcc()] + compile_flags + ["-c", "-o", obj, os.path.join(CSRC, src)]
        return obj, subprocess.run(cmd, capture_output=True, text=True)

    # one translation unit per kernel family: compiled side by side, then linked into the in-tree .so
    with ThreadPoolExecutor(max_workers=len(SOURCES)) as pool:
        results = list(pool.map(compile_one, SOURCES))
    failed = False
    for _, r in results:
        if verbose or r.returncode != 0:
            sys.stderr.write(r.stdout + r.stderr)
        failed = failed or r.returncode != 0
    if failed:
        raise RuntimeError("nvcc failed building libagym_b200.so")
    link = subprocess.run([_nvcc()] + NVCC_FLAGS + ["-o", OUT] + [o for o, _ in results], capture_output=True, text=True)
    if verbose or link.returncode != 0:
        sys.stderr.write(link.stdout + link.stderr)
    if link.returncode != 0:
        raise RuntimeError("nvcc failed linking libagym_b200.so")
    return OUT


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
