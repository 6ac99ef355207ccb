"""Builds libcvs_b200.so (the CUDA kernels + C ABI + CUDACore shim) in-tree for sm_100a.

nvcc cross-compiles without a GPU, so this also runs on the CPU-only build box; the resulting .so is
git-ignored but travels to the GPU box with the working tree.
"""
from __future__ import annotations

import os
import shutil
import subprocess

_HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(_HERE, "csrc")
LIB = os.path.join(_HERE, "libcvs_b200.so")
SOURCES = ["cvs_api.cu", "cvs_shim.cu"]
HEADERS = ["cvs_device.cuh", "cvs_pixel.cuh", "cvs_stream_kernel.cuh", "cvs_stream_ws.cuh", "cvs_filter_kernels.cuh", "cvs_jpeg.cuh", "cvs_jpeg_host.hpp", "cvs_yuv.cuh", "cvs_bayer.cuh",
           os.path.join("..", "..", "include", "cvs_b200.h"), os.path.join("..", "..", "include", "cvs_cuda_core.hpp")]

NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
              "-Xcompiler", "-fPIC,-fvisibility=hidden", "-shared", "-cudart", "shared"]


def _nvcc() -> str:
    for cand in (shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found: libcvs_b200.so cannot be built (there is no CPU fallback)")


def stale() -> bool:
    if not os.path.exists(LIB):
        return True
    t = os.path.getmtime(LIB)
    deps = [os.path.join(CSRC, s) for s in SOURCES + HEADERS] + [os.path.abspath(__file__)]
    return any(os.path.getmtime(d) > t for d in deps if os.path.exists(d))


def build_library(force: bool = False, verbose: bool = False) -> str:
    if not force and not stale():
        return LIB
    cmd = [_nvcc()] + NVCC_FLAGS + (["-Xptxas", "-v"] if verbose else []) + \
          ["-I", os.path.join(_HERE, "..", "include"), "-o", LIB] + [os.path.join(CSRC, s) for s in SOURCES] + ["-ldl"]
    subprocess.check_call(cmd, cwd=CSRC)
    return LIB


if __name__ == "__main__":
    print(build_library(force=True, verbose=False))
