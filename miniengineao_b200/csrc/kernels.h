// kernels.h -- argument blocks and host-side launchers of the three libmeao pipeline stages.
//
// All intermediate buffers live in HBM in NATURAL (row-major, non-deinterleaved) layout with
// global frame coordinates; rows are pitched to 128 bytes.  The four 16-slice TiledDepth atlases
// of the reference (Downsample1.compute:71,78, Downsample2.compute:41,49) are never materialised:
// the render kernel reads LowDepth<k> and applies the f16 rounding, the slice-space clamp and the
// atlas padding values itself (see render_ao.cu).
#pragma once

// Build switch: drop the per-pixel range test of the final division in the packed upsample path when the host has proved
// it redundant from the two tolerances (blur_upsample.cu, bilateral2).  Shared by the kernel and the planner.
// Measured on B200 and NOT adopted: the 48 guard instructions per 8 pixels disappear, but under the 48-register cap ptxas
// then spills more (stack 48 -> 80 B, +20 MOV, +19 LDL/STL) and the frame got slower (117.2 vs 119.3 Gpx/s).
#ifndef MEAO_UPS_STATIC_GUARD
#define MEAO_UPS_STATIC_GUARD 0
#endif
// Build switch: the restructured bilateral-upsample phase (blur_upsample.cu, "phase-4 restructure"); it relies on the same
// host-side proof as MEAO_UPS_STATIC_GUARD, so the planner applies the tighter tolerance bounds whenever either is on.
#ifndef MEAO_UPS_V2
#define MEAO_UPS_V2 1
#endif

#ifdef MEAO_EMULATE              // tests/emu only (see common.cuh)
#include "cuda_emu.h"
#else
#include <cuda.h>
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#endif
#include <stdint.h>

// Kernel launch.  `k` is the kernel name IN PARENTHESES (they protect the commas of template arguments from the
// preprocessor).  CUDA build: cudaLaunchKernelEx, with the programmatic-dependent-launch attribute when the recorder asked
// for it (meao::g_launch_pdl, set by meao_api.cu around the launches whose predecessor IN THE SAME STREAM is one of our
// kernels): the dependent grid may then be scheduled while its predecessor drains, runs its prologue and blocks in
// pdl_wait() (griddepcontrol.wait) until the predecessor has completed and flushed -- see common.cuh.
#define MEAO_UNPAREN(...) __VA_ARGS__
#ifdef MEAO_EMULATE
#define MEAO_LAUNCH(k, grid, block, smem, stream, ...) meao_emu::launch((grid), (block), (smem), [&]() { MEAO_UNPAREN k(__VA_ARGS__); })
#else
namespace meao {
inline thread_local bool g_launch_pdl = false;
template <class... KArgs, class... Args>
inline cudaError_t launch_ex(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t s, Args &&...args)
{
    cudaLaunchConfig_t cfg{};
    cfg.gridDim = grid; cfg.blockDim = block; cfg.dynamicSmemBytes = smem; cfg.stream = s;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    at[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = at; cfg.numAttrs = g_launch_pdl ? 1 : 0;
    return cudaLaunchKernelEx(&cfg, kernel, KArgs(args)...);
}
}  // namespace meao
#define MEAO_LAUNCH(k, grid, block, smem, stream, ...) (void)meao::launch_ex(MEAO_UNPAREN k, (grid), (block), (smem), (stream), __VA_ARGS__)
#endif

namespace meao {

// ---- stage 1: prepare_depth = Downsample1.compute + Downsample2.compute fused ----------------
struct PrepareArgs {
    const void *depth;      // input rows [depth_row0, ...) of the frame, row pitch = W elements (f32 / u16 / u32)
    int in_format;          // 0 = f32, 1 = D16_UNORM codes (u16), 2 = D24_UNORM_S8_UINT words (u32, depth in the low 24 bits)
    int W, H;               // full-frame size
    int depth_row0;         // global row of depth[0]
    int row0, row1;         // global L0 rows to process; row0 % 16 == 0
    __half *lin;            // LinearDepth, L0, f16
    int lin_pitch;          // elements
    float *low[4];          // LowDepth1..4, f32
    int low_pitch[4];       // elements
    float zbx, zby;         // ZBufferParams.xy (AmbientOcclusion.cs:561-568)
    int raw;                // 1: Linearize (DS1:37-48); 0: depth is already linear
    int reversed_z;         // UNITY_REVERSED_Z (DS1:41-45)
    int vec_ok;             // depth pointer 16B aligned and rows stay 16B aligned (W % 4 == 0 for f32/u32, W % 8 == 0 for u16)
};
cudaError_t launch_prepare_depth(const PrepareArgs &a, cudaStream_t s);

// ---- stage 2: render_ao = Render.compute main_interleaved, one mip level -----------------------
struct RenderArgs {
    const float *low;       // LowDepth<k>
    int lw, lh, lpitch;     // size of level k, pitch in elements
    uint8_t *occ;           // Occlusion<k>, unorm8
    int opitch;
    int sw, sh;             // size of the (virtual) TiledDepth<k> slice = level k+2
    float pad;              // value of atlas padding texels (already f16-rounded): Linearize(0) for k=1,2; 0 for k=3,4
    float inv_thickness[12];// gInvThicknessTable entries in CALL order: 7 used by Render.compute:162-168 (checker), 12 by :148-159 (exhaustive)
    float neg_front[12];    // -(invThickness - 0.5)  (Render.compute:85)
    float weight[12];       // gSampleWeightTable entries, same order
    float reject_fadeoff;   // gRejectFadeoff
    float intensity;        // gIntensity
    int row0, row1;         // output rows (level k) to produce
    int wide;               // 0: kernel main_interleaved (virtual f16 atlas of level k+2); 1: kernel main (WIDE_SAMPLING on f32 LowDepth<k>;
                            //    sw/sh/pad unused, low_map must carry the kRenderWideBox box)
    int exhaustive;         // SAMPLE_EXHAUSTIVELY (Render.compute:144-159)
    int tile_h;             // output rows per CTA, one of kRenderTileHs (32: big levels; 16 / 8: coarse levels -- 2x / 4x the CTAs and a half / a
                            //    quarter of the per-CTA latency: the coarse renders are latency-bound); low_map must carry the matching box
};
cudaError_t launch_render_ao(const CUtensorMap &low_map, bool use_tma, const RenderArgs &a, cudaStream_t s);
constexpr int kRenderTileVariants = 3;
constexpr int kRenderTileHs[kRenderTileVariants] = {32, 16, 8};
constexpr int kRenderBoxW = 96, kRenderWideBoxW = 80;               // TMA box widths of the render kernel (f32 elements): 64 + 2 x apron (16 / wide: 8)
constexpr int render_box_h(int tile_h, bool wide) { return tile_h + (wide ? 16 : 32); }

// ---- stage 3: blur_upsample = Upsample.compute main / main_blendout, one level ----------------
struct UpsampleArgs {
    const float *lo_depth;  // LoResDB  (LowDepth<lo>)
    int low, loh, lo_dpitch;
    const uint8_t *lo_ao;   // LoResAO1 (Occlusion4 or Combined<lo>)
    int lo_apitch;
    const void *hi_depth;   // HiResDB  (LowDepth<hi> f32, or LinearDepth f16 when hi == 0)
    int hi_is_half;
    int hi_dpitch;
    const uint8_t *hi_ao;   // HiResAO (Occlusion<hi>) or nullptr => kernel "main" (Upsample.compute:223)
    int hi_apitch;
    uint8_t *out;           // AoResult
    int out_pitch;
    int out_row_origin;     // global row stored at out[0]
    int out_vec_ok;         // out is 8B aligned and out_pitch % 8 == 0
    int hiw, hih;
    float noise_filter_strength, step_size, blur_tolerance, upsample_tolerance;
    int fast_div_ok;        // upsample_tolerance and noise_filter_strength are positive normals in [2^-60, 2^60)
                            // (built with MEAO_UPS_STATIC_GUARD: additionally tol >= 2^-55 and 2^-52 <= nfs < 2^59, see blur_upsample.cu)
    int row0, row1;         // output rows (hi level) to produce
    uint32_t *tile_ctr;     // [0] next tile, [1] CTAs that have run out of tiles: device words owned by (context, level), zero between launches
    int tiles_x, tiles_y;   // tile grid (filled by launch_blur_upsample)
};
// main_premin / main_premin_blendout (COMBINE_LOWER_RESOLUTIONS): the same arguments plus LoResAO2 = HighQuality<lo>
struct UpsamplePreminArgs { UpsampleArgs base; const uint8_t *lo_ao2; int lo_a2pitch; };
// lo_ao2 == nullptr: kernels main / main_blendout; otherwise the premin kernels (lo_ao2_map = its TMA descriptor)
cudaError_t launch_blur_upsample(const CUtensorMap &lo_depth_map, const CUtensorMap &lo_ao_map, const CUtensorMap *lo_ao2_map, bool use_tma,
                                 const UpsampleArgs &a, const uint8_t *lo_ao2, int lo_a2pitch, cudaStream_t s);
constexpr int kUpsDepthBoxW = 40, kUpsDepthBoxH = 22; // TMA boxes of the upsample kernel
constexpr int kUpsAoBoxW = 64, kUpsAoBoxH = 22;

// ---- batched frames (meao_render_batch): the three stages over `frames` frames in one launch each -------------------
// Every intermediate of frame f lives at base + f * slot_bytes (one frame slot of the batch arena holds all of them, with the
// single-frame pitches).  The TMA'd buffers get 3-D maps (w, h, capacity) with strides (pitch, slot_bytes).  The argument
// blocks wrap the single-frame ones, whose pointers then address frame 0.
struct PrepareBatchArgs { PrepareArgs base; long long in_frame_bytes; long long slot_bytes; };   // base.vec_ok: holds for EVERY frame
cudaError_t launch_prepare_depth_batch(const PrepareBatchArgs &a, int frames, cudaStream_t s);
struct RenderBatchArgs { RenderArgs base; long long slot_bytes; };                               // low and occ advance by slot_bytes
cudaError_t launch_render_ao_batch(const CUtensorMap &low_map3, bool use_tma, const RenderBatchArgs &a, int frames, cudaStream_t s);
// lo_depth / lo_ao / lo_ao2 / hi_depth / hi_ao advance by slot_bytes, out by out_frame_bytes (base.out_vec_ok: for every frame)
struct UpsampleBatchArgs { UpsamplePreminArgs pa; long long slot_bytes; long long out_frame_bytes; int frames; int tiles_per_frame; };
cudaError_t launch_blur_upsample_batch(const CUtensorMap &lo_depth_map3, const CUtensorMap &lo_ao_map3, const CUtensorMap *lo_ao2_map3,
                                       bool use_tma, const UpsampleBatchArgs &a, cudaStream_t s);

// ---- debug: synthesise a TiledDepth<k> view (reference layout [16][sh][sw], f16 bits) ----------
cudaError_t launch_synth_tiled(const float *low, int lw, int lh, int lpitch, int sw, int sh, float pad,
                               __half *out, cudaStream_t s);

// ---- debug views (PushDebugBlitCommands AO.cs:787-820, Blit.shader pass 4): buffer -> W x H R8 image ----------
struct DebugViewArgs {
    const void *src;        // non-tiled: the buffer itself; tiled: LowDepth<k> (the atlas is virtual)
    int elem;               // bytes per source element: 1 unorm8, 2 f16, 4 f32
    int sw, sh;             // source texture size (tiled: size of one slice)
    int spitch;             // source pitch in elements
    int tiled;              // 1: TiledDepth<k> view synthesised from LowDepth<k>
    int lw, lh;             // tiled: size of level k
    float pad;              // tiled: value of the atlas padding texels (f16-rounded)
    uint8_t *out;           // W x H R8 codes
    int out_pitch;
    int W, H;
};
cudaError_t launch_debug_view(const DebugViewArgs &a, cudaStream_t s);
// Blit.shader pass 3 (AO.cs:826-829): colour target (RGBA8 / RGBA16F, tight) = (r, r, r, r) of the R8 view
cudaError_t launch_debug_composite(const uint8_t *view, void *color, long long npix, int half, cudaStream_t s);

// ---- composite (Blit.shader passes 1 and 2): colour *= ao, 4 pixels per thread ------------------------
cudaError_t launch_composite(const uint8_t *ao, void *color, long long npix, int half, int rgb, int alpha, int one_minus, cudaStream_t s);

// ---- self test: div_fast / rcp_fast vs the IEEE operators on n random in-range operand pairs ------
cudaError_t launch_selftest_div(uint64_t n, uint32_t seed, unsigned long long *mismatch_dev, cudaStream_t s);

// ---- native neighbour exchange (include/meao.h "native neighbour exchange"): peer stores + epoch flags, one launch ------
// Flags live in every band context's arena (zeroed at allocation).  ready / ack are written by the NEIGHBOURS through
// their peer mapping; epoch / done / error are local.
struct BandFlags {
    uint32_t ready[2];      // [side]: epoch of the halo rows the neighbour on `side` has delivered into this arena
    uint32_t ack[2];        // [side]: epoch the neighbour on `side` is about to RECEIVE, i.e. everything it read before is consumed
    uint32_t epoch;         // epoch of this context's next exchange (first = 1)
    uint32_t done;          // CTA completion counter of the running exchange kernel
    uint32_t error;         // sticky: 0 ok, 1 timed out waiting for an ack, 2 timed out waiting for rows
    uint32_t pad_;
};
struct XchgSeg { const uint4 *src; uint4 *dst; uint32_t n16; int32_t side; };     // one flat 16-byte-granular copy into the neighbour on `side`
struct XchgArgs {
    XchgSeg seg[8];         // LowDepth1..4 border rows x 2 sides (whole pitched rows: contiguous, 128-byte aligned)
    int nseg;
    BandFlags *local;
    BandFlags *peer[2];     // neighbour's flags through the peer mapping; nullptr = no neighbour on that side
    uint32_t *host_error;   // mapped host word mirroring local->error (may be nullptr)
    unsigned long long timeout_ns;
};
cudaError_t launch_band_exchange(const XchgArgs &a, cudaStream_t s);

// ---- eager loading ------------------------------------------------------------------------------------------------------
// CUDA loads kernels lazily, on first launch, and that load can wait for kernels already RUNNING on the device.  A band's exchange
// kernel spins until its neighbour has run -- if the neighbour's first launch then has to load a kernel on the same device, the two
// wait for each other until the exchange times out (seen when the band tests ran first in a fresh process).  meao_create therefore
// touches every kernel of the library once per device (cudaFuncGetAttributes forces the load).
#ifndef MEAO_EMULATE
template <class K> inline cudaError_t preload_kernel(K kernel) { cudaFuncAttributes at; return cudaFuncGetAttributes(&at, (const void *)kernel); }
cudaError_t preload_prepare_depth();
cudaError_t preload_prepare_depth_batch();
cudaError_t preload_render_ao();
cudaError_t preload_render_ao_batch();
cudaError_t preload_blur_upsample();
cudaError_t preload_blur_upsample_batch();
cudaError_t preload_band_kernels();
cudaError_t preload_aux_kernels();      // composite, debug views, self test
#endif

// ---- halo pack / unpack: row blocks of pitched buffers <-> contiguous staging, one launch ------
struct HaloSeg { const float *src; float *dst; int src_pitch, dst_pitch, width, rows; };
struct HaloArgs { HaloSeg seg[8]; int nseg; };
cudaError_t launch_halo_copy(const HaloArgs &a, cudaStream_t s);

}  // namespace meao
