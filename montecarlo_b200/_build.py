"""In-tree build of libarianna_cuda.so with nvcc for sm_100a (no torch, no JIT cache: the .so travels with the
repo snapshot to the GPU box)."""
from __future__ import annotations

import os
import shutil
import subprocess

_HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(_HERE, "csrc")
INCLUDE = os.path.join(os.path.dirname(_HERE), "include")
LIB_PATH = os.path.join(_HERE, "libarianna_cuda.so")

NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-lineinfo", "-O3", "-std=c++17",
    "-Xcompiler", "-fPIC,-fvisibility=hidden",
    "-shared",
]


def _sources():
    return [os.path.join(CSRC, f) for f in sorted(os.listdir(CSRC)) if f.endswith((".cu", ".cuh", ".inc"))] + [
        os.path.join(INCLUDE, "arianna_cuda.h")]


def is_stale() -> bool:
    if not os.path.exists(LIB_PATH):
        return True
    t = os.path.getmtime(LIB_PATH)
    return any(os.path.getmtime(s) > t for s in _sources())


def build_library(force: bool = False, verbose: bool = False) -> str:
    """Compile csrc/arianna_cuda.cu -> montecarlo_b200/libarianna_cuda.so.  Needs nvcc; no GPU required."""
    if not force and not is_stale():
        return LIB_PATH
    nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not os.path.exists(nvcc):
        raise RuntimeError("nvcc not found: cannot build libarianna_cuda.so (there is no CPU fallback)")
    cmd = [nvcc] + NVCC_FLAGS + (["-Xptxas", "-v"] if verbose else []) + [
        "-o", LIB_PATH, os.path.join(CSRC, "arianna_cuda.cu")]
    res = subprocess.run(cmd, capture_output=True, text=True)
    if res.returncode != 0:
        raise RuntimeError("nvcc failed:\n" + res.stdout + res.stderr)
    if verbose:
        print(res.stderr)
    return LIB_PATH


if __name__ == "__main__":
    print(build_library(force=True, verbose=True))
