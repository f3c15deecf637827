"""ctypes binding of libmeao.so (include/meao.h).  No fallback: if the library is missing or no
B200 is usable, loading / context creation raises."""
from __future__ import annotations

import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "libmeao.so")

MEAO_OK, MEAO_ERR_INVALID, MEAO_ERR_CUDA, MEAO_ERR_UNSUPPORTED, MEAO_ERR_NOMEM, MEAO_ERR_PEER = 0, -1, -2, -3, -4, -5
MEAO_ABI_VERSION = 3
MEAO_PEER_HANDLE_BYTES = 128
MEAO_FLAG_NONE, MEAO_FLAG_NO_GRAPH = 0, 1
MEAO_DEPTH_RAW_F32, MEAO_DEPTH_LINEAR_F32, MEAO_DEPTH_RAW_D16_UNORM, MEAO_DEPTH_RAW_D24S8 = 0, 1, 2, 3
MEAO_FMT_RGBA8_UNORM, MEAO_FMT_RGBA16_FLOAT = 0, 1


class MeaoParams(C.Structure):
    _fields_ = [("noise_filter_tolerance", C.c_float), ("blur_tolerance", C.c_float),
                ("upsample_tolerance", C.c_float), ("thickness_modifier", C.c_float),
                ("intensity", C.c_float), ("debug", C.c_int32), ("ambient_only", C.c_int32)]


class MeaoCamera(C.Structure):
    _fields_ = [("near_clip", C.c_float), ("far_clip", C.c_float),
                ("tan_half_fov_h", C.c_float), ("reversed_z", C.c_int32)]


class MeaoDeviceCfg(C.Structure):
    _fields_ = [("device", C.c_int32), ("flags", C.c_uint32)]


class MeaoVariants(C.Structure):
    _fields_ = [("single_pass_stereo", C.c_int32), ("sample_exhaustively", C.c_int32), ("high_quality_mask", C.c_int32),
                ("single_scale", C.c_int32)]


class MeaoPeerHandle(C.Structure):
    _fields_ = [("bytes", C.c_ubyte * MEAO_PEER_HANDLE_BYTES)]


class MeaoBufferDesc(C.Structure):
    _fields_ = [("width", C.c_int32), ("height", C.c_int32), ("slices", C.c_int32), ("elem_bytes", C.c_int32)]


RENDER_EVENT_FUNC = C.CFUNCTYPE(None, C.c_int)

# name -> (restype, argtypes); every symbol include/meao.h declares
SIGNATURES = {
    "meao_abi_version": (C.c_int, []),
    "meao_create": (C.c_int, [C.POINTER(MeaoDeviceCfg), C.POINTER(C.c_void_p)]),
    "meao_destroy": (None, [C.c_void_p]),
    "meao_last_error": (C.c_char_p, [C.c_void_p]),
    "meao_set_params": (C.c_int, [C.c_void_p, C.POINTER(MeaoParams)]),
    "meao_get_params": (C.c_int, [C.c_void_p, C.POINTER(MeaoParams)]),
    "meao_default_params": (None, [C.POINTER(MeaoParams)]),
    "meao_set_variants": (C.c_int, [C.c_void_p, C.POINTER(MeaoVariants)]),
    "meao_get_variants": (C.c_int, [C.c_void_p, C.POINTER(MeaoVariants)]),
    "meao_set_camera": (C.c_int, [C.c_void_p, C.POINTER(MeaoCamera)]),
    "meao_resize": (C.c_int, [C.c_void_p, C.c_int32, C.c_int32]),
    "meao_render": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p]),
    "meao_render_host": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p]),
    "meao_render_host_async": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p, C.c_int32]),
    "meao_host_wait": (C.c_int, [C.c_void_p, C.c_int32]),
    "meao_reserve_batch": (C.c_int, [C.c_void_p, C.c_int32]),
    "meao_render_batch": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p]),
    "meao_get_batch_buffer": (C.c_int, [C.c_void_p, C.c_int32, C.c_int32, C.c_void_p, C.c_size_t]),
    "meao_synchronize": (C.c_int, [C.c_void_p]),
    "meao_host_alloc": (C.c_void_p, [C.c_size_t]),
    "meao_host_free": (None, [C.c_void_p]),
    "meao_stage_downsample": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p]),
    "meao_stage_render": (C.c_int, [C.c_void_p, C.c_int32, C.c_void_p]),
    "meao_stage_render_wide": (C.c_int, [C.c_void_p, C.c_int32, C.c_void_p]),
    "meao_stage_upsample": (C.c_int, [C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p]),
    "meao_buffer_desc": (C.c_int, [C.c_void_p, C.c_int32, C.POINTER(MeaoBufferDesc)]),
    "meao_get_buffer": (C.c_int, [C.c_void_p, C.c_int32, C.c_void_p, C.c_size_t]),
    "meao_set_buffer": (C.c_int, [C.c_void_p, C.c_int32, C.c_void_p, C.c_size_t]),
    "meao_render_constants": (C.c_int, [C.c_void_p, C.c_int32, C.POINTER(C.c_float)]),
    "meao_render_constants_wide": (C.c_int, [C.c_void_p, C.c_int32, C.POINTER(C.c_float)]),
    "meao_debug_view": (C.c_int, [C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p]),
    "meao_upsample_constants": (C.c_int, [C.c_void_p, C.c_int32, C.POINTER(C.c_float)]),
    "meao_zbuffer_params": (C.c_int, [C.c_void_p, C.POINTER(C.c_float)]),
    "meao_set_row_band": (C.c_int, [C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_int32]),
    "meao_halo_bytes": (C.c_int64, [C.c_void_p, C.c_int32]),
    "meao_halo_recv_bytes": (C.c_int64, [C.c_void_p, C.c_int32]),
    "meao_halo_rows": (C.c_int, [C.c_void_p, C.c_int32, C.c_int32, C.POINTER(C.c_int32)]),
    "meao_band_rows": (C.c_int, [C.c_void_p, C.POINTER(C.c_int32)]),
    "meao_halo_pack": (C.c_int, [C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p]),
    "meao_halo_unpack": (C.c_int, [C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p]),
    "meao_render_band_prepare": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p]),
    "meao_render_band_finish": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p]),
    "meao_band_phase_a": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p]),
    "meao_band_phase_b": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "meao_composite_framebuffer": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p]),
    "meao_composite_gbuffer": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p]),
    "meao_composite_debug": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p]),
    "meao_band_export": (C.c_int, [C.c_void_p, C.POINTER(MeaoPeerHandle)]),
    "meao_band_connect": (C.c_int, [C.c_void_p, C.c_int32, C.POINTER(MeaoPeerHandle)]),
    "meao_band_step": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p]),
    "meao_band_step_host": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p]),
    "meao_band_status": (C.c_int, [C.c_void_p, C.POINTER(C.c_int32)]),
    "meao_bind_event": (C.c_int, [C.c_void_p, C.c_int32, C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p]),
    "meao_render_event": (None, [C.c_int]),
    "meao_get_render_event_func": (RENDER_EVENT_FUNC, []),
    "meao_launch_count": (C.c_int64, [C.c_void_p]),
    "meao_pdl_level": (C.c_int, [C.c_void_p]),
    "meao_kernels_per_frame": (C.c_int, [C.c_void_p]),
    "meao_algorithmic_bytes": (C.c_int64, [C.c_void_p, C.c_int32]),
    "meao_selftest_div": (C.c_int, [C.c_void_p, C.c_uint64, C.c_uint32, C.POINTER(C.c_uint64)]),
    "meao_set_profile_repeats": (C.c_int, [C.c_void_p, C.c_int32]),
    "meao_profile_frame": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p, C.POINTER(C.c_float),
                                     C.POINTER(C.c_char_p), C.c_int32]),
}

_lib = None


class MeaoError(RuntimeError):
    def __init__(self, code: int, message: str):
        super().__init__(f"libmeao error {code}: {message}")
        self.code = code


def lib() -> C.CDLL:
    """Load libmeao.so (built in-tree by miniengineao_b200/build.py).  Raises if it is absent."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise ImportError(
                f"{LIB_PATH} not found: the CUDA extension is not built. Run `python -c 'import __graft_entry__ as g; "
                "g.build()'` (needs nvcc). There is no CPU fallback.")
        l = C.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(l, name)          # AttributeError if the symbol is missing
            fn.restype = res
            fn.argtypes = args
        _lib = l
    return _lib


def check(ctx, rc: int) -> int:
    if rc < 0:
        msg = lib().meao_last_error(ctx)
        raise MeaoError(rc, msg.decode() if msg else "?")
    return rc
