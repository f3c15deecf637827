"""ctypes front end of tests/emu_batch/libmeao_emu_batch.so -- the batched kernel sources compiled for the host.
TEST INFRASTRUCTURE ONLY (see ../emu/cuda_emu.h): used by tests/test_batch_emulated.py."""
from __future__ import annotations

import ctypes as C

import numpy as np

from emu.emu import EmulatedFrame, _aligned  # (tests/ is on sys.path via conftest)
from emu_batch import build_emu_batch

_lib: C.CDLL | None = None


def lib() -> C.CDLL:
    global _lib
    if _lib is None:
        l = C.CDLL(build_emu_batch.build())
        l.emu_create.restype = C.c_void_p
        l.emu_create.argtypes = [C.c_int, C.c_int]
        l.emu_destroy.argtypes = [C.c_void_p]
        l.emu_set_constants.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_float, C.c_int, C.c_int, C.c_int, C.c_int]
        l.emu_set_tma.argtypes = [C.c_void_p, C.c_int]
        l.emu_set_render_tile.argtypes = [C.c_void_p, C.c_int]
        l.emu_set_single_scale.argtypes = [C.c_void_p, C.c_int]
        l.emu_tma_box_loads.restype = C.c_longlong
        l.emu_run_batch.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_void_p]
        l.emu_get_batch_buffer.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_void_p]
        _lib = l
    return _lib


class EmulatedBatch(EmulatedFrame):
    """B frames through the host-compiled batched kernels (meao_render_batch), planned like EmulatedFrame."""

    def __init__(self, plan, *, use_tma: bool = True, render_tile: int = -1):
        super().__init__(plan, use_tma=use_tma, render_tile=render_tile)
        # the same context, re-created in the library that also holds the batched kernels
        from miniengineao_b200 import _native as N
        old_lib, old_h = self._lib, self._h
        self._lib = lib()
        nl = N.lib()
        rc, rcw, uc, zb = (C.c_float * 112)(), (C.c_float * 112)(), (C.c_float * 32)(), (C.c_float * 4)()
        for k in range(1, 5):
            N.check(plan._ctx, nl.meao_render_constants(plan._ctx, k, C.cast(C.byref(rc, 112 * (k - 1)), C.POINTER(C.c_float))))
            N.check(plan._ctx, nl.meao_render_constants_wide(plan._ctx, k, C.cast(C.byref(rcw, 112 * (k - 1)), C.POINTER(C.c_float))))
            N.check(plan._ctx, nl.meao_upsample_constants(plan._ctx, k, C.cast(C.byref(uc, 32 * (k - 1)), C.POINTER(C.c_float))))
        N.check(plan._ctx, nl.meao_zbuffer_params(plan._ctx, zb))
        rz = bool(plan.camera.usesReversedZBuffer)
        pad12 = 1e5 if rz else float(np.float32(1) / np.float32(zb[1]))     # Linearize(OOB load = 0): DS1:40-45 (raw ingest)
        self._h = self._lib.emu_create(self.W, self.H)
        old_lib.emu_destroy(old_h)
        self._lib.emu_set_tma(self._h, int(use_tma))
        self._lib.emu_set_render_tile(self._h, int(render_tile))
        self._lib.emu_set_single_scale(self._h, int(getattr(plan, "singleScale", False)))
        self._lib.emu_set_constants(self._h, rc, rcw, uc, zb, pad12, 1, int(rz), int(plan.highQualityMask), int(plan.sampleExhaustively))

    def run_batch(self, depth: np.ndarray) -> np.ndarray:
        """depth [B, H, W] (raw f32 / D16 codes / D24S8 words) -> AO [B, H, W]; frame f's intermediates are then batch_buffer(f, id)."""
        fmt = {"float32": 0, "uint16": 1, "uint32": 2}[depth.dtype.name]
        d = _aligned(np.ascontiguousarray(depth))
        assert d.ndim == 3 and d.shape[1:] == (self.H, self.W)
        out = _aligned(np.zeros(d.shape, np.uint8))
        self._lib.emu_run_batch(self._h, d.ctypes.data, fmt, d.shape[0], out.ctypes.data)
        return out.copy()

    def batch_buffer(self, frame: int, bid: int) -> np.ndarray:
        d = self.plan.buffer_desc(bid)
        dt = {1: np.uint8, 2: np.float16, 4: np.float32}[d.elem_bytes]
        shape = (d.slices, d.height, d.width) if d.slices > 1 else (d.height, d.width)
        out = np.zeros(shape, dt)
        assert self._lib.emu_get_batch_buffer(self._h, frame, bid, out.ctypes.data) == 0
        return out
