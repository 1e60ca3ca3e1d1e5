"""Build the CUDA engine in-tree: sparselm_b200/lib/libsparselm_b200.so (sm_100a)."""

from __future__ import annotations

import os
import shutil
import subprocess

_PKG = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(_PKG, "csrc")
LIB_DIR = os.path.join(_PKG, "lib")
LIB_PATH = os.path.join(LIB_DIR, "libsparselm_b200.so")
SOURCES = ["engine.cu"]
HEADERS = ["gemm_f64.cuh", "gemm_f64_tma.cuh", "solver_kernels.cuh", "whiten_kernels.cuh", "cg_kernels.cuh", "coop_kernels.cuh", "newton_kernels.cuh", "select_kernels.cuh", os.path.join("..", "..", "include", "sparselm_b200.h")]

NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-O3", "-lineinfo", "-std=c++17",
    "-Xcompiler", "-fPIC", "-shared",
]


def find_nvcc() -> str:
    nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not os.path.exists(nvcc):
        raise RuntimeError("nvcc not found: the sparselm_b200 CUDA engine cannot be built")
    return nvcc


def is_stale() -> bool:
    if not os.path.exists(LIB_PATH):
        return True
    t = os.path.getmtime(LIB_PATH)
    deps = [os.path.join(CSRC, s) for s in SOURCES] + [os.path.join(CSRC, h) for h in HEADERS]
    return any(os.path.getmtime(d) > t for d in deps)


def build(force: bool = False, verbose: bool = False) -> str:
    """Compile every CUDA source for sm_100a (nvcc cross-compiles without a GPU)."""
    if not force and not is_stale():
        return LIB_PATH
    os.makedirs(LIB_DIR, exist_ok=True)
    cmd = [find_nvcc(), *NVCC_FLAGS, "-o", LIB_PATH] + [os.path.join(CSRC, s) for s in SOURCES]
    if verbose:
        cmd.insert(1, "-Xptxas")
        cmd.insert(2, "-v")
    res = subprocess.run(cmd, capture_output=True, text=True)
    if res.returncode != 0:
        raise RuntimeError("nvcc failed:\n" + res.stdout + res.stderr)
    if verbose:
        print(res.stderr)
    return LIB_PATH


if __name__ == "__main__":
    print(build(force=True, verbose=True))
