"""Builds libmeao.so (CUDA, sm_100a only) in-tree with nvcc.

nvcc cross-compiles without a GPU, so this also runs in the CPU-only build container.
-fmad=false: fused multiply-adds appear only where the sources call fmaf() (the arithmetic
contract shared with the oracle); -prec-div / -prec-sqrt stay at their IEEE defaults.
"""
from __future__ import annotations

import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(HERE, "libmeao.so")
SOURCES = ["meao_api.cu", "prepare_depth.cu", "prepare_depth_batch.cu", "render_ao.cu", "render_ao_batch.cu", "blur_upsample.cu", "blur_upsample_batch.cu", "selftest.cu", "halo.cu", "band_exchange.cu", "composite.cu", "debug_view.cu"]
HEADERS = ["common.cuh", "kernels.h", "blur_upsample_kernel.inc", "prepare_depth_kernel.inc", "render_ao_kernel.inc", os.path.join("..", "..", "include", "meao.h")]

NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-O3", "-std=c++17", "-lineinfo",
    "-fmad=false",
    "-Xcompiler", "-fPIC,-O2,-fvisibility=hidden",
    "-Xptxas", "-v",
    "-shared", "-cudart", "static", "--threads", "0",
    "-Xlinker", "--exclude-libs,ALL", "-Xlinker", "-Bsymbolic",
]


def _nvcc() -> str:
    for cand in (os.environ.get("NVCC"), "/usr/local/cuda/bin/nvcc", "nvcc"):
        if cand and (os.path.isabs(cand) and os.path.exists(cand) or not os.path.isabs(cand)):
            return cand
    return "nvcc"


def is_stale() -> bool:
    if not os.path.exists(LIB):
        return True
    t = os.path.getmtime(LIB)
    deps = [os.path.join(CSRC, f) for f in SOURCES + HEADERS] + [os.path.abspath(__file__)]
    return any(os.path.getmtime(d) > t for d in deps)


def build(force: bool = False, verbose: bool = False) -> str:
    if not force and not is_stale():
        return LIB
    extra = os.environ.get("MEAO_NVCC_DEFS", "").split()      # tuning experiments, e.g. "-DMEAO_REN_MINB=12"
    cmd = [_nvcc()] + NVCC_FLAGS + extra + ["-o", LIB] + [os.path.join(CSRC, f) for f in SOURCES]
    proc = subprocess.run(cmd, capture_output=True, text=True)
    if verbose or proc.returncode != 0:
        sys.stderr.write(proc.stdout + proc.stderr)
    if proc.returncode != 0:
        raise RuntimeError("nvcc failed building libmeao.so")
    with open(os.path.join(HERE, "build_ptxas.log"), "w") as f:
        f.write(proc.stdout + proc.stderr)
    return LIB


if __name__ == "__main__":
    build(force="--force" in sys.argv, verbose=True)
    print(LIB)
