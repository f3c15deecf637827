"""Host-side mirror of MiniEngineAO.AmbientOcclusion (Assets/MiniEngineAO/AmbientOcclusion.cs).

Same property names, ranges and defaults (AO.cs:20-68), same re-plan triggers (LateUpdate /
CheckPropertiesChanged, AO.cs:84-113, 329-350), same constant math -- but the ten compute
dispatches of the "SSAO" command buffer (AO.cs:511-531) are one call into libmeao.so.
PyTorch is used only to hold device memory and streams.  There is no CPU fallback.
"""
from __future__ import annotations

import ctypes as C
import math
from dataclasses import dataclass

import numpy as np

from . import _native as N


@dataclass
class Camera:
    """The few UnityEngine.Camera fields the hot path reads (AO.cs:338-341, 561-573)."""
    pixelWidth: int
    pixelHeight: int
    nearClipPlane: float = 0.3
    farClipPlane: float = 100.0
    fieldOfView: float = 60.0           # vertical, degrees
    usesReversedZBuffer: bool = True    # SystemInfo.usesReversedZBuffer on D3D11/12
    stereoEnabled: bool = False         # Camera.stereoEnabled (AO.cs:397)
    targetTexture: object = None        # Camera.targetTexture (AO.cs:398)
    allowHDR: bool = True               # Camera.allowHDR (AO.cs:407)
    actualRenderingPath: str = "Forward"    # "Forward" | "DeferredShading" (AO.cs:408)

    @property
    def aspect(self) -> float:
        return self.pixelWidth / self.pixelHeight

    @property
    def projection00(self) -> float:
        """projectionMatrix[0,0] of a perspective camera."""
        return 1.0 / (self.aspect * math.tan(math.radians(self.fieldOfView) / 2.0))


def _clamp(v, lo, hi):
    return max(lo, min(hi, v))


class AmbientOcclusion:
    """Drop-in for the compute path of the AmbientOcclusion component."""

    # debug view ids, AO.cs:787-808
    DEBUG_NAMES = {1: "LinearDepth", 2: "LowDepth1", 3: "LowDepth2", 4: "LowDepth3", 5: "LowDepth4",
                   6: "TiledDepth1", 7: "TiledDepth2", 8: "TiledDepth3", 9: "TiledDepth4",
                   10: "Occlusion1", 11: "Occlusion2", 12: "Occlusion3", 13: "Occlusion4",
                   14: "Combined1", 15: "Combined2", 16: "Combined3", 17: "AmbientOcclusion",
                   # extension ids: HighQuality<k>, the output of Render.compute kernel "main" (highQualityMask)
                   18: "HighQuality1", 19: "HighQuality2", 20: "HighQuality3", 21: "HighQuality4"}

    def __init__(self, camera: Camera, device: int = 0, use_graph: bool = True):
        self._lib = N.lib()
        self._camera = camera
        cfg = N.MeaoDeviceCfg(device, N.MEAO_FLAG_NONE if use_graph else N.MEAO_FLAG_NO_GRAPH)
        h = C.c_void_p()
        rc = self._lib.meao_create(C.byref(cfg), C.byref(h))
        if rc < 0:
            msg = self._lib.meao_last_error(None)
            raise N.MeaoError(rc, msg.decode() if msg else "?")
        self._ctx = h
        self.device = device
        p = N.MeaoParams()
        self._lib.meao_default_params(C.byref(p))
        # serialized fields, AO.cs:20-68
        self._noiseFilterTolerance = p.noise_filter_tolerance
        self._blurTolerance = p.blur_tolerance
        self._upsampleTolerance = p.upsample_tolerance
        self._thicknessModifier = p.thickness_modifier
        self._intensity = p.intensity
        self._debug = 0
        self._ambientOnly = True
        # shader variants the reference ships but never selects (SURVEY.md 8f.2); defaults = reference behaviour
        self.sampleExhaustively = False     # Render.compute:144-159
        self.highQualityMask = 0            # bit k-1: Render.compute kernel "main" on level k + Upsample main_premin*
        self.singleScale = False            # BASELINE.json configs[0]: Downsample1 -> Render level 1 -> final-style Upsample only
        self._band = None                   # (row0, row1) after set_row_band; reset by every re-allocation
        self._drawCountPerFrame = 0         # AO.cs:289: used to detect single-pass stereo
        self._stereo = False                # singlePassStereoEnabled as latched by the last LateUpdate
        self.rebuild_count = 0
        self._width = self._height = 0

    # ---- exposed properties (AO.cs:22-66); Unity clamps to the Range attribute in the inspector only
    noiseFilterTolerance = property(lambda s: s._noiseFilterTolerance, lambda s, v: setattr(s, "_noiseFilterTolerance", float(v)))
    blurTolerance = property(lambda s: s._blurTolerance, lambda s, v: setattr(s, "_blurTolerance", float(v)))
    upsampleTolerance = property(lambda s: s._upsampleTolerance, lambda s, v: setattr(s, "_upsampleTolerance", float(v)))
    thicknessModifier = property(lambda s: s._thicknessModifier, lambda s, v: setattr(s, "_thicknessModifier", float(v)))
    intensity = property(lambda s: s._intensity, lambda s, v: setattr(s, "_intensity", float(v)))
    ambientOnly = property(lambda s: s._ambientOnly, lambda s, v: setattr(s, "_ambientOnly", bool(v)))
    RANGES = {"noiseFilterTolerance": (-8, 0), "blurTolerance": (-8, -1), "upsampleTolerance": (-12, -1),
              "thicknessModifier": (1, 10), "intensity": (0, 2), "debug": (0, 17)}

    @property
    def camera(self) -> Camera:
        return self._camera

    def close(self) -> None:
        if getattr(self, "_ctx", None):
            self._lib.meao_destroy(self._ctx)      # OnDestroy, AO.cs:357-381
            self._ctx = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _check(self, rc: int) -> int:
        return N.check(self._ctx, rc)

    # ---- single-pass stereo detection (AO.cs:352-355, 387-401) ------------------------------------------
    def OnPreRender(self) -> None:
        """Unity calls this once per camera draw; with single-pass stereo both eyes are ONE draw (AO.cs:352-355)."""
        self._drawCountPerFrame += 1

    @property
    def singlePassStereoEnabled(self) -> bool:
        cam = self._camera
        return bool(cam is not None and cam.stereoEnabled and cam.targetTexture is None and self._drawCountPerFrame == 1)

    # ---- LateUpdate: re-plan only when something changed (AO.cs:329-350) ---------------------------
    def LateUpdate(self) -> bool:
        """Once per frame (AO.cs:329-350); render() / render_host() call it themselves.  Returns True when it re-planned."""
        return self._update(True)

    def _update(self, frame: bool) -> bool:
        """The body of LateUpdate.  frame=False (debug / stage / constant queries between two frames) skips the
        per-frame reset of the draw counter (AO.cs:349), so such calls do not toggle the stereo detection."""
        cam = self._camera
        p = N.MeaoParams(self._noiseFilterTolerance, self._blurTolerance, self._upsampleTolerance,
                         self._thicknessModifier, self._intensity, self._debug, int(self._ambientOnly))
        rebuild = self._check(self._lib.meao_set_params(self._ctx, C.byref(p))) == 1      # CheckPropertiesChanged
        c = N.MeaoCamera(cam.nearClipPlane, cam.farClipPlane, 1.0 / cam.projection00, int(cam.usesReversedZBuffer))
        self._check(self._lib.meao_set_camera(self._ctx, C.byref(c)))
        if frame:
            self._stereo = self.singlePassStereoEnabled       # evaluated once per frame, before the counter reset (AO.cs:338-349)
        stereo = self._stereo
        v = N.MeaoVariants(int(stereo), int(self.sampleExhaustively), int(self.highQualityMask), int(self.singleScale))
        rebuild |= self._check(self._lib.meao_set_variants(self._ctx, C.byref(v))) == 1
        width = cam.pixelWidth * (2 if stereo else 1)                                                # AO.cs:338-341, 501-504
        resized = self._check(self._lib.meao_resize(self._ctx, width, cam.pixelHeight)) == 1          # CheckBaseDimensions
        self._width, self._height = width, cam.pixelHeight
        if resized:
            self._band = None       # meao_resize re-allocates: the C context is back to the whole frame and has dropped its neighbours
        if rebuild or resized:
            self.rebuild_count += 1
        if frame:
            self._drawCountPerFrame = 0                                                              # AO.cs:349
        return rebuild or resized

    # ---- frame ----------------------------------------------------------------------------------
    @staticmethod
    def _kind(dtype_name: str, linear: bool) -> int:
        """float32 -> RAW_F32 (or LINEAR_F32); uint16 -> D16_UNORM codes; int32 / uint32 -> D24_UNORM_S8_UINT words."""
        if dtype_name == "float32":
            return N.MEAO_DEPTH_LINEAR_F32 if linear else N.MEAO_DEPTH_RAW_F32
        if linear:
            raise ValueError("linear depth must be float32")
        if dtype_name == "uint16":
            return N.MEAO_DEPTH_RAW_D16_UNORM
        if dtype_name in ("int32", "uint32"):
            return N.MEAO_DEPTH_RAW_D24S8
        raise ValueError(f"unsupported depth dtype {dtype_name}")

    def render(self, depth, out=None, *, linear: bool = False, stream=None):
        """depth: CUDA tensor [H, W]: float32 raw camera depth (or linear if linear=True), uint16 D16_UNORM codes,
        or int32 D24_UNORM_S8_UINT words.  Returns a CUDA uint8 tensor [H, W] -- the AmbientOcclusion R8 texture (AO.cs:475)."""
        import torch
        self.LateUpdate()
        if not (depth.is_cuda and depth.is_contiguous()):
            raise ValueError("depth must be a contiguous CUDA tensor")
        rows = self._band_rows()
        if tuple(depth.shape) != (rows, self._width):
            raise ValueError(f"depth shape {tuple(depth.shape)} != {(rows, self._width)}")
        if out is None:
            out = torch.empty((rows, self._width), dtype=torch.uint8, device=depth.device)
        kind = self._kind(str(depth.dtype).replace("torch.", ""), linear)
        self._check(self._lib.meao_render(self._ctx, depth.data_ptr(), kind, out.data_ptr(), self._stream(stream)))
        return out

    def render_batch(self, depth, out=None, *, linear: bool = False, stream=None):
        """depth: contiguous CUDA tensor [B, H, W] of B independent frames, dtypes as in render().  Returns a CUDA uint8 tensor
        [B, H, W]; frame b equals render(depth[b]).  One graph replay for the whole batch (meao_render_batch).  The first batch
        larger than any before allocates the batch intermediates (synchronous): call reserve_batch(B) first to keep that out of
        a timed loop."""
        import torch
        self.LateUpdate()
        if not (depth.is_cuda and depth.is_contiguous()):
            raise ValueError("depth must be a contiguous CUDA tensor")
        if depth.dim() != 3 or tuple(depth.shape[1:]) != (self._height, self._width):
            raise ValueError(f"depth shape {tuple(depth.shape)} != (B, {self._height}, {self._width})")
        frames = int(depth.shape[0])
        if out is None:
            out = torch.empty((frames, self._height, self._width), dtype=torch.uint8, device=depth.device)
        elif not (out.is_cuda and out.is_contiguous() and out.dtype == torch.uint8 and tuple(out.shape) == tuple(depth.shape)):
            raise ValueError("out must be a contiguous CUDA uint8 tensor of the depth's shape")
        kind = self._kind(str(depth.dtype).replace("torch.", ""), linear)
        self._check(self._lib.meao_render_batch(self._ctx, depth.data_ptr(), kind, frames, out.data_ptr(), self._stream(stream)))
        return out

    def reserve_batch(self, frames: int) -> None:
        """Allocates the batch intermediates for >= frames frames now (render_batch would on first use)."""
        self._update(False)
        self._check(self._lib.meao_reserve_batch(self._ctx, int(frames)))

    def batch_buffer(self, frame: int, debug_id: int) -> np.ndarray:
        """Buffer <id> (1-16, 18-21) of frame <frame> of the last render_batch, like debug_buffer."""
        d = self.buffer_desc(debug_id)
        dt = {1: np.uint8, 2: np.float16, 4: np.float32}[d.elem_bytes]
        shape = (d.slices, d.height, d.width) if d.slices > 1 else (d.height, d.width)
        a = np.empty(shape, dt)
        self._check(self._lib.meao_get_batch_buffer(self._ctx, int(frame), debug_id, a.ctypes.data, a.nbytes))
        return a

    def render_host(self, depth: np.ndarray, out: np.ndarray | None = None, *, linear: bool = False) -> np.ndarray:
        """Host [H, W] depth (float32 / uint16 D16 codes / uint32 D24S8 words) in, host uint8 [H, W] out
        (H2D + the kernels + D2H + sync)."""
        self.LateUpdate()
        rows = self._band_rows()
        d = np.ascontiguousarray(depth)
        if d.shape != (rows, self._width):
            raise ValueError(f"depth shape {d.shape} != {(rows, self._width)}")
        if out is None:
            out = np.empty((rows, self._width), np.uint8)
        kind = self._kind(d.dtype.name, linear)
        self._check(self._lib.meao_render_host(self._ctx, d.ctypes.data, kind, out.ctypes.data))
        return out

    def render_host_batch(self, depths, outs, *, linear: bool = False) -> None:
        """Frame stream with HOST buffers: depths[i] (float32, or uint16 D16_UNORM codes, [H, W]) -> outs[i] (uint8 [H, W]).  Frames alternate
        over the two staging slots of the context, so the H2D copy of frame i+1 overlaps the kernels and the D2H
        copy of frame i.  Pass pinned arrays (meao_host_alloc) for real overlap; the arrays must stay alive and
        untouched until this call returns."""
        self.LateUpdate()
        rows = self._band_rows()
        n = len(depths)
        assert len(outs) == n
        for i in range(n):
            d, o = depths[i], outs[i]
            if d.dtype not in (np.float32, np.uint16) or not d.flags.c_contiguous or d.shape != (rows, self._width):
                raise ValueError("depths[i] must be C-contiguous float32 (or uint16 D16 codes) [rows, W]")
            kind = self._kind(d.dtype.name, linear)
            if o.dtype != np.uint8 or not o.flags.c_contiguous or o.shape != (rows, self._width):
                raise ValueError("outs[i] must be C-contiguous uint8 [rows, W]")
            slot = i & 1
            if i >= 2:
                self._check(self._lib.meao_host_wait(self._ctx, slot))
            self._check(self._lib.meao_render_host_async(self._ctx, d.ctypes.data, kind, o.ctypes.data, slot))
        self._check(self._lib.meao_host_wait(self._ctx, 0))
        self._check(self._lib.meao_host_wait(self._ctx, 1))

    # ---- event / pass selection (AO.cs:403-429, 822-839) ---------------------------------------------------
    @property
    def ambientOnlyEnabled(self) -> bool:
        cam = self._camera
        return bool(self._ambientOnly and cam.allowHDR and cam.actualRenderingPath == "DeferredShading")     # AO.cs:403-410

    @property
    def camera_events(self) -> tuple[str, str]:
        """(event of the render command buffer, event of the composite command buffer), RegisterCommandBuffers AO.cs:412-429."""
        render = "BeforeReflections" if self.ambientOnlyEnabled else "BeforeImageEffects"
        if self._debug > 0:
            comp = "AfterImageEffects"
        else:
            comp = "BeforeLighting" if self.ambientOnlyEnabled else "BeforeImageEffects"
        return render, comp

    def composite(self, ao, *, color=None, gbuffer0=None, gbuffer3=None, stream=None) -> str:
        """PushCompositeCommands (AO.cs:822-839): with `debug` > 0 the selected debug view replaces the camera target
        (Blit.shader pass 3); otherwise the ambient-only deferred branch multiplies the G-buffer occlusion and ambient
        targets (pass 1), otherwise the frame buffer is multiplied (pass 2).  Returns the branch taken."""
        if self._debug > 0:
            if color is None:
                raise ValueError("the debug composite needs the camera target")
            view = ao if self._debug == 17 else self.debug_view(self._debug, stream=stream)       # AO.cs:815-819
            self.composite_debug(view, color, stream=stream)
            return "debug"
        if self.ambientOnlyEnabled:
            if gbuffer0 is None or gbuffer3 is None:
                raise ValueError("ambient-only deferred composite needs gbuffer0 and gbuffer3 (AO.cs:595-598)")
            self.composite_gbuffer(ao, gbuffer0, gbuffer3, stream=stream)
            return "gbuffer"
        if color is None:
            raise ValueError("frame-buffer composite needs the camera target")
        self.composite_framebuffer(ao, color, stream=stream)
        return "framebuffer"

    # ---- composite (Blit.shader passes 1 / 2, AO.cs:822-839) -------------------------------------------
    def composite_framebuffer(self, ao, color, *, stream=None) -> None:
        """color (CUDA uint8 [H, W, 4] = RGBA8, or float16 [H, W, 4] = RGBA16F) *= ao, in place (pass 2)."""
        import torch
        fmt = N.MEAO_FMT_RGBA16_FLOAT if color.dtype == torch.float16 else N.MEAO_FMT_RGBA8_UNORM
        self._check(self._lib.meao_composite_framebuffer(self._ctx, ao.data_ptr(), color.data_ptr(), fmt, self._stream(stream)))

    def composite_gbuffer(self, ao, gbuffer0, gbuffer3, *, stream=None) -> None:
        """gbuffer0 (RGBA8).a *= 1-(1-ao); gbuffer3 (RGBA8 or RGBA16F).rgb *= 1-(1-ao), in place (pass 1)."""
        import torch
        fmt = N.MEAO_FMT_RGBA16_FLOAT if gbuffer3.dtype == torch.float16 else N.MEAO_FMT_RGBA8_UNORM
        self._check(self._lib.meao_composite_gbuffer(self._ctx, ao.data_ptr(), gbuffer0.data_ptr(), gbuffer3.data_ptr(), fmt,
                                                     self._stream(stream)))

    def composite_debug(self, view, color, *, stream=None) -> None:
        """color (RGBA8 / RGBA16F, CUDA) = view.rrrr (Blit.shader pass 3, no blending)."""
        import torch
        fmt = N.MEAO_FMT_RGBA16_FLOAT if color.dtype == torch.float16 else N.MEAO_FMT_RGBA8_UNORM
        self._check(self._lib.meao_composite_debug(self._ctx, view.data_ptr(), color.data_ptr(), fmt, self._stream(stream)))

    # `debug` (AO.cs:60): 0 = normal composite, 1..17 = show that buffer instead
    debug = property(lambda s: s._debug, lambda s, v: setattr(s, "_debug", int(v)))

    def synchronize(self) -> None:
        """Wait for the context's own stream (host-buffer path, debug copies) AND the current torch stream."""
        self._check(self._lib.meao_synchronize(self._ctx))
        import torch
        torch.cuda.current_stream(self.device).synchronize()

    def _stream(self, stream=None):
        """cudaStream_t handle to launch on: the given torch stream or torch's current stream."""
        import torch
        s = stream if stream is not None else torch.cuda.current_stream(self.device)
        return C.c_void_p(s.cuda_stream)

    # ---- stage entry points (mirror Push*Commands) -----------------------------------------------
    def stage_downsample(self, depth, *, linear: bool = False) -> None:
        self._update(False)
        kind = N.MEAO_DEPTH_LINEAR_F32 if linear else N.MEAO_DEPTH_RAW_F32
        self._check(self._lib.meao_stage_downsample(self._ctx, depth.data_ptr(), kind, self._stream()))

    def stage_render(self, level: int) -> None:
        self._update(False)
        self._check(self._lib.meao_stage_render(self._ctx, level, self._stream()))

    def stage_render_wide(self, level: int) -> None:
        """PushRenderCommands for the non-tiled source LowDepth<level> (kernel "main") -> HighQuality<level>."""
        self._update(False)
        self._check(self._lib.meao_stage_render_wide(self._ctx, level, self._stream()))

    def stage_upsample(self, lo_level: int) -> None:
        self._update(False)
        self._check(self._lib.meao_stage_upsample(self._ctx, lo_level, None, self._stream()))

    # ---- debug views (AO.cs:787-820) ---------------------------------------------------------------
    def buffer_desc(self, debug_id: int) -> N.MeaoBufferDesc:
        self._update(False)
        d = N.MeaoBufferDesc()
        self._check(self._lib.meao_buffer_desc(self._ctx, debug_id, C.byref(d)))
        return d

    def debug_buffer(self, debug_id: int) -> np.ndarray:
        """Buffer <id> in the reference layout and native type: float16 / float32 / uint8 codes."""
        d = self.buffer_desc(debug_id)
        dt = {1: np.uint8, 2: np.float16, 4: np.float32}[d.elem_bytes]
        shape = (d.slices, d.height, d.width) if d.slices > 1 else (d.height, d.width)
        a = np.empty(shape, dt)
        self._check(self._lib.meao_get_buffer(self._ctx, debug_id, a.ctypes.data, a.nbytes))
        return a

    def debug_view(self, debug_id: int, out=None, *, stream=None):
        """PushDebugBlitCommands (AO.cs:787-820): the W x H R8 image the `debug` property would put on screen for
        buffer <debug_id>; returns a CUDA uint8 tensor [H, W]."""
        import torch
        self._update(False)
        if out is None:
            out = torch.empty((self._height, self._width), dtype=torch.uint8, device=f"cuda:{self.device}")
        self._check(self._lib.meao_debug_view(self._ctx, debug_id, out.data_ptr(), self._stream(stream)))
        return out

    def dump_debug_view(self, debug_id: int, path: str) -> None:
        """Writes the debug view as a binary PGM (P5) image -- the observable twin of the inspector's debug slider."""
        img = self.debug_view(debug_id)
        self.synchronize()
        a = img.cpu().numpy()
        with open(path, "wb") as f:
            f.write(b"P5\n%d %d\n255\n" % (a.shape[1], a.shape[0]))
            f.write(a.tobytes())

    def set_debug_buffer(self, debug_id: int, values: np.ndarray) -> None:
        d = self.buffer_desc(debug_id)
        dt = {1: np.uint8, 2: np.float16, 4: np.float32}[d.elem_bytes]
        a = np.ascontiguousarray(values, dtype=dt)
        assert a.shape == (d.height, d.width), (a.shape, d.height, d.width)
        self._check(self._lib.meao_set_buffer(self._ctx, debug_id, a.ctypes.data, a.nbytes))

    # ---- constants ----------------------------------------------------------------------------------
    def render_constants(self, level: int, wide: bool = False) -> dict:
        self._update(False)
        out = (C.c_float * 28)()
        fn = self._lib.meao_render_constants_wide if wide else self._lib.meao_render_constants
        self._check(fn(self._ctx, level, out))
        a = np.array(out, np.float32)
        return {"inv_thickness": a[0:12], "sample_weight": a[12:24], "inv_slice_dim": a[24:26],
                "reject_fadeoff": a[26], "intensity": a[27]}

    def upsample_constants(self, lo_level: int) -> dict:
        self._update(False)
        out = (C.c_float * 8)()
        self._check(self._lib.meao_upsample_constants(self._ctx, lo_level, out))
        a = np.array(out, np.float32)
        return {"inv_low": a[0:2], "inv_high": a[2:4], "noise_filter_strength": a[4], "step_size": a[5],
                "blur_tolerance": a[6], "upsample_tolerance": a[7]}

    def zbuffer_params(self) -> np.ndarray:
        self._update(False)
        out = (C.c_float * 4)()
        self._check(self._lib.meao_zbuffer_params(self._ctx, out))
        return np.array(out, np.float32)

    # ---- row bands (multi-GPU frame partition) ---------------------------------------------------
    def set_row_band(self, row0: int, row1: int, prev_row0: int = -1, next_row1: int = -1) -> None:
        self._update(False)
        self._check(self._lib.meao_set_row_band(self._ctx, row0, row1, prev_row0, next_row1))
        self._band = (row0, row1)

    def _band_rows(self) -> int:
        return self._height if self._band is None else self._band[1] - self._band[0]

    def band_rows(self) -> dict:
        """Row ranges of this band per level: rows to produce, LowDepth rows read, LowDepth rows owned."""
        self._update(False)
        out = (C.c_int32 * 30)()
        self._check(self._lib.meao_band_rows(self._ctx, out))
        a = list(out)
        return {"produce": [(a[2 * k], a[2 * k + 1]) for k in range(5)],
                "need_low": [(a[10 + 2 * k], a[11 + 2 * k]) for k in range(5)],
                "own_low": [(a[20 + 2 * k], a[21 + 2 * k]) for k in range(5)]}

    def halo_rows(self, side: int, send: bool) -> list[tuple[int, int]]:
        """[(lo, hi)] rows of LowDepth1..4 sent to / received from `side` (0 = up, 1 = down)."""
        out = (C.c_int32 * 8)()
        self._check(self._lib.meao_halo_rows(self._ctx, side, int(send), out))
        return [(out[2 * i], out[2 * i + 1]) for i in range(4)]

    def halo_bytes(self, side: int) -> int:
        return self._check(self._lib.meao_halo_bytes(self._ctx, side))

    def halo_recv_bytes(self, side: int) -> int:
        return self._check(self._lib.meao_halo_recv_bytes(self._ctx, side))

    def halo_pack(self, side: int, buf, stream=None) -> None:
        self._check(self._lib.meao_halo_pack(self._ctx, side, buf.data_ptr(), self._stream(stream)))

    def halo_unpack(self, side: int, buf, stream=None) -> None:
        self._check(self._lib.meao_halo_unpack(self._ctx, side, buf.data_ptr(), self._stream(stream)))

    def band_prepare(self, depth_band, *, linear: bool = False, stream=None) -> None:
        kind = N.MEAO_DEPTH_LINEAR_F32 if linear else N.MEAO_DEPTH_RAW_F32
        self._check(self._lib.meao_render_band_prepare(self._ctx, depth_band.data_ptr(), kind, self._stream(stream)))

    def band_finish(self, out_band, stream=None) -> None:
        self._check(self._lib.meao_render_band_finish(self._ctx, out_band.data_ptr(), self._stream(stream)))

    # native neighbour exchange (ABI 3): peer stores over NVLink inside the frame's graph, no host code between the phases
    def band_export(self) -> bytes:
        """Opaque handle of this band's arena (contains a cudaIpcMemHandle_t); hand it to the neighbours."""
        h = N.MeaoPeerHandle()
        self._check(self._lib.meao_band_export(self._ctx, C.byref(h)))
        return bytes(h.bytes)

    def band_connect(self, side: int, handle: bytes | None) -> None:
        """side 0 = the band above, 1 = below; None disconnects."""
        if handle is None:
            self._check(self._lib.meao_band_connect(self._ctx, side, None))
            return
        h = N.MeaoPeerHandle()
        C.memmove(h.bytes, handle, N.MEAO_PEER_HANDLE_BYTES)
        self._check(self._lib.meao_band_connect(self._ctx, side, C.byref(h)))

    def band_step(self, depth_band, out_band, *, linear: bool = False, stream=None) -> None:
        """One frame of a connected band as ONE CUDA graph: prepare_depth -> peer exchange -> render x4 + upsample x4."""
        kind = self._kind(str(depth_band.dtype).replace("torch.", ""), linear)
        self._check(self._lib.meao_band_step(self._ctx, depth_band.data_ptr(), kind, out_band.data_ptr(), self._stream(stream)))

    def band_status(self) -> dict:
        out = (C.c_int32 * 4)()
        self._check(self._lib.meao_band_status(self._ctx, out))
        return {"epoch": out[0], "error": out[1], "connected": (bool(out[2]), bool(out[3]))}

    def band_phase_a(self, depth_band, send_up, send_down, *, linear: bool = False, stream=None) -> None:
        """prepare_depth on the band + pack of both halos, replayed as one CUDA graph."""
        kind = N.MEAO_DEPTH_LINEAR_F32 if linear else N.MEAO_DEPTH_RAW_F32
        ptr = lambda t: (t.data_ptr() if t is not None and t.numel() else None)  # noqa: E731
        self._check(self._lib.meao_band_phase_a(self._ctx, depth_band.data_ptr(), kind, ptr(send_up), ptr(send_down), self._stream(stream)))

    def band_phase_b(self, recv_up, recv_down, out_band, stream=None) -> None:
        """unpack of both halos + render x4 + upsample x4, replayed as one CUDA graph."""
        ptr = lambda t: (t.data_ptr() if t is not None and t.numel() else None)  # noqa: E731
        self._check(self._lib.meao_band_phase_b(self._ctx, ptr(recv_up), ptr(recv_down), out_band.data_ptr(), self._stream(stream)))

    # ---- introspection ----------------------------------------------------------------------------
    @property
    def launch_count(self) -> int:
        return self._lib.meao_launch_count(self._ctx)

    @property
    def pdl_level(self) -> int:
        """Programmatic-dependent-launch level the captured graphs use (-1 before the first capture)."""
        return self._lib.meao_pdl_level(self._ctx)

    @property
    def kernels_per_frame(self) -> int:
        return self._lib.meao_kernels_per_frame(self._ctx)

    def algorithmic_bytes(self, stage: int = 0) -> int:
        self._update(False)
        return self._check(self._lib.meao_algorithmic_bytes(self._ctx, stage))

    def selftest_div(self, n: int = 1 << 28, seed: int = 1) -> int:
        """Mismatches between the kernels' guarded fast division / reciprocal and the IEEE operators (must be 0)."""
        self._update(False)
        m = C.c_uint64(0)
        self._check(self._lib.meao_selftest_div(self._ctx, n, seed, C.byref(m)))
        return int(m.value)

    def profile_frame(self, depth, out, *, linear: bool = False, repeats: int = 1) -> list[tuple[str, float]]:
        """(name, ms) per kernel of one serial frame; repeats > 1: every kernel launched that many times back to back, mean reported."""
        self._update(False)
        self._check(self._lib.meao_set_profile_repeats(self._ctx, int(repeats)))
        n = self.kernels_per_frame
        ms = (C.c_float * n)()
        names = (C.c_char_p * n)()
        kind = N.MEAO_DEPTH_LINEAR_F32 if linear else N.MEAO_DEPTH_RAW_F32
        k = self._check(self._lib.meao_profile_frame(self._ctx, depth.data_ptr(), kind, out.data_ptr(), ms, names, n))
        return [(names[i].decode(), float(ms[i])) for i in range(k)]
