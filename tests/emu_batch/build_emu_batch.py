"""Builds tests/emu_batch/libmeao_emu_batch.so: the host emulator of tests/emu plus the BATCHED kernel sources
(prepare_depth_batch.cu, render_ao_batch.cu, blur_upsample_batch.cu) and the batch driver.  TEST INFRASTRUCTURE ONLY
(see ../emu/cuda_emu.h); every translation unit but the fiber runtime gets the 3-D TMA emulation (cuda_emu_3d.h)."""
from __future__ import annotations

import importlib.util
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
EMU = os.path.join(os.path.dirname(HERE), "emu")
_spec = importlib.util.spec_from_file_location("_meao_build_emu", os.path.join(EMU, "build_emu.py"))
build_emu = importlib.util.module_from_spec(_spec)
_spec.loader.exec_module(build_emu)

CSRC = build_emu.CSRC
LIB = os.path.join(HERE, "libmeao_emu_batch.so")
KERNELS = build_emu.KERNELS + ["prepare_depth_batch.cu", "render_ao_batch.cu", "blur_upsample_batch.cu"]
FLAGS = build_emu.FLAGS + ["-include", os.path.join(HERE, "cuda_emu_3d.h")]


def is_stale() -> bool:
    if not os.path.exists(LIB):
        return True
    t = os.path.getmtime(LIB)
    deps = [os.path.join(CSRC, f) for f in os.listdir(CSRC)] + \
           [os.path.join(d, f) for d in (HERE, EMU) for f in os.listdir(d) if f.endswith((".h", ".cpp", ".py"))]
    return any(os.path.getmtime(d) > t for d in deps)


def build(force: bool = False) -> str:
    if not force and not is_stale():
        return LIB
    objs = []
    units = [(os.path.join(EMU, "emu_runtime.cpp"), build_emu.FLAGS), (os.path.join(HERE, "emu_batch_driver.cpp"), FLAGS)] + \
            [(os.path.join(CSRC, k), FLAGS + ["-x", "c++"]) for k in KERNELS]
    for src, flags in units:
        obj = os.path.join(HERE, f"libmeao_emu_batch_{os.path.basename(src)}.o")
        p = subprocess.run(["g++"] + flags + ["-c", src, "-o", obj], capture_output=True, text=True)
        if p.returncode != 0:
            sys.stderr.write(p.stdout + p.stderr)
            raise RuntimeError(f"batch emulator build failed: {os.path.basename(src)}")
        objs.append(obj)
    subprocess.check_call(["g++", "-shared", "-o", LIB] + objs)
    for o in objs:
        os.remove(o)
    return LIB


if __name__ == "__main__":
    print(build(force=True))
