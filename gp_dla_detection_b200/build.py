"""In-tree build of libgpdla.so (explicit nvcc, sm_100a only)."""
from __future__ import annotations

import os
import subprocess

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(HERE, "libgpdla.so")
SOURCES = ["gpdla_capi.cu"]
HEADERS = ["gpdla_kernels.cuh", "gpdla_i8_kernels.cuh", "gpdla_preload.cuh", "gpdla_objective.cuh", "gpdla_training.cuh", "gpdla_statistics.cuh", "gpdla_posteriors.cuh", "gpdla_reconstruct.cuh", "gpdla_draw.cuh", "gpdla_math.cuh", "voigt_tables.h", "gpdla_rest_table.h", os.path.join("..", "..", "include", "gpdla.h")]
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17",
              "-shared", "-Xcompiler", "-fPIC"]


def needs_build() -> bool:
    if not os.path.exists(LIB):
        return True
    t = os.path.getmtime(LIB)
    return any(os.path.getmtime(os.path.join(CSRC, f)) > t for f in SOURCES + HEADERS)


def build_extension(force: bool = False, verbose: bool = False) -> str:
    if not force and not needs_build():
        return LIB
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    cmd = [nvcc] + NVCC_FLAGS + (["-Xptxas", "-v"] if verbose else []) + ["-o", LIB] + SOURCES
    res = subprocess.run(cmd, cwd=CSRC, capture_output=True, text=True)
    if res.returncode != 0:
        raise RuntimeError("nvcc failed:\n" + res.stdout + res.stderr)
    if verbose:
        print(res.stderr)
    return LIB


if __name__ == "__main__":
    print(build_extension(force=True, verbose=True))
