// prepare_depth.cu -- stage 1 of the SSAO pipe: depth linearise + point-sampled mip hierarchy.
//
// Replaces Downsample1.compute (Linearize :37-48, main :52-81) and Downsample2.compute (main
// :32-51) with ONE streaming pass:   raw depth (f32, L0)  ->  LinearDepth (f16, L0),
// LowDepth1..4 (f32; LowDepth<k>(i,j) = lin(2^k i, 2^k j), a pure point sample -- DS1:64-66,
// DS2:35).  The deinterleaved f16 atlases are not written (see kernels.h).
//
// Bound: HBM.  Algorithmic bytes per L0 pixel: 4 (read) + 2 + 4/4 + 4/16 + 4/64 + 4/256 = 7.33
// (the reference's Downsample1+2 move 8.24 B/px because they also write and re-read the atlases).
// There is no data reuse between threads, so no shared-memory staging: each thread streams
// 2 x 8 pixels with 128-bit loads (L1::no_allocate) and 128-bit stores.
#include "common.cuh"
#include "kernels.h"

namespace meao {

namespace {

constexpr int kPrepThreads = 256;
constexpr int kPrepTileW = 256;   // 32 lanes x 8 pixels
constexpr int kPrepTileH = 16;    // 8 warps x 2 rows (w, w+8): one LowDepth4 row per tile

template <bool RAW, bool REVERSED>
__device__ __forceinline__ float linearize(float depth, float zbx, float zby)
{
    if (!RAW) return depth;
    float dist = rcp_ieee(fmaf(zbx, depth, zby));       // DS1:40 (mad + IEEE reciprocal)
    if (REVERSED) { if (depth == 0.0f) dist = 1e5f; }   // DS1:41-42
    else          { if (depth == 1.0f) dist = 1e5f; }   // DS1:43-44
    return dist;
}

// Eight pixels at once (MEAO_PACKED_RCP): the mad of DS1:40 is formed directly in negated form, nt = fma(-zbx, d, -zby) = -t
// exactly (round-to-nearest is sign-symmetric), all eight range tests feed ONE branch, and the reciprocals run as packed
// f32x2 (rcp2_fast_neg).  If any element is out of range (inf / NaN / zero / denormal / negative) the group takes the plain
// per-element path of linearize() -- which recomputes t itself, so signed zeros behave exactly as before.
template <bool RAW, bool REVERSED>
__device__ __forceinline__ void linearize8(const float (&v)[8], float zbx, float zby, float (&d)[8])
{
    if (!RAW) {
#pragma unroll
        for (int e = 0; e < 8; e++) d[e] = v[e];
        return;
    }
    const float2 nzx = make_float2(-zbx, -zbx), nzy = make_float2(-zby, -zby);
    float2 nt[4];
    bool ok = true;
#pragma unroll
    for (int q = 0; q < 4; q++) {
        nt[q] = __ffma2_rn(make_float2(v[2 * q], v[2 * q + 1]), nzx, nzy);
        ok = ok & in_safe_range_neg(nt[q].x) & in_safe_range_neg(nt[q].y);
    }
    if (ok) {
#pragma unroll
        for (int q = 0; q < 4; q++) {
            const float2 r = rcp2_fast_neg(nt[q]);
            d[2 * q] = r.x; d[2 * q + 1] = r.y;
        }
#pragma unroll
        for (int e = 0; e < 8; e++) {
            if (REVERSED) { if (v[e] == 0.0f) d[e] = 1e5f; }   // DS1:41-42
            else          { if (v[e] == 1.0f) d[e] = 1e5f; }   // DS1:43-44
        }
    } else {
#pragma unroll
        for (int e = 0; e < 8; e++) d[e] = linearize<RAW, REVERSED>(v[e], zbx, zby);
    }
}

// native depth formats (SURVEY.md 8f.1): the camera depth texture read by Blit.shader pass 0 (:48-64) is a D32_FLOAT,
// D24_UNORM_S8_UINT or D16_UNORM resource; SAMPLE_DEPTH_TEXTURE returns code / (2^n - 1) for the UNORM ones
// (D3D UNORM -> FLOAT rule: (float)code * (1.0f / (2^n - 1))).
enum { IN_F32 = 0, IN_D16 = 1, IN_D24S8 = 2 };

template <int IN>
__device__ __forceinline__ void load8(const void *base, size_t elem_index, bool full, int valid, float (&v)[8])
{
    if (IN == IN_F32) {
        const float *src = reinterpret_cast<const float *>(base) + elem_index;
        if (full) {
            const float4 q0 = ldg_stream_f4(src), q1 = ldg_stream_f4(src + 4);
            v[0] = q0.x; v[1] = q0.y; v[2] = q0.z; v[3] = q0.w; v[4] = q1.x; v[5] = q1.y; v[6] = q1.z; v[7] = q1.w;
        } else {
#pragma unroll
            for (int e = 0; e < 8; e++) v[e] = (e < valid) ? __ldg(src + e) : 0.0f;
        }
    } else if (IN == IN_D16) {
        const uint16_t *src = reinterpret_cast<const uint16_t *>(base) + elem_index;
        uint32_t c[8];
        if (full) {
            const uint4 q = ldg_stream_u4(src);
            c[0] = q.x & 0xffffu; c[1] = q.x >> 16; c[2] = q.y & 0xffffu; c[3] = q.y >> 16;
            c[4] = q.z & 0xffffu; c[5] = q.z >> 16; c[6] = q.w & 0xffffu; c[7] = q.w >> 16;
        } else {
#pragma unroll
            for (int e = 0; e < 8; e++) c[e] = (e < valid) ? __ldg(src + e) : 0u;
        }
#pragma unroll
        for (int e = 0; e < 8; e++) v[e] = __fmul_rn((float)c[e], 1.0f / 65535.0f);
    } else {
        const uint32_t *src = reinterpret_cast<const uint32_t *>(base) + elem_index;
        uint32_t c[8];
        if (full) {
            const uint4 q0 = ldg_stream_u4(src), q1 = ldg_stream_u4(src + 4);
            c[0] = q0.x; c[1] = q0.y; c[2] = q0.z; c[3] = q0.w; c[4] = q1.x; c[5] = q1.y; c[6] = q1.z; c[7] = q1.w;
        } else {
#pragma unroll
            for (int e = 0; e < 8; e++) c[e] = (e < valid) ? __ldg(src + e) : 0u;
        }
#pragma unroll
        for (int e = 0; e < 8; e++) v[e] = __fmul_rn((float)(c[e] & 0xffffffu), 1.0f / 16777215.0f);   // depth = low 24 bits, stencil = high 8
    }
}

// (built a second time with MEAO_PREP_BATCH = 1 by prepare_depth_batch.cu: the batched kernels and their launcher)
#ifndef MEAO_PREP_BATCH
#define MEAO_PREP_BATCH 0
#endif
#include "prepare_depth_kernel.inc"

}  // namespace

#if !MEAO_PREP_BATCH
cudaError_t launch_prepare_depth(const PrepareArgs &a, cudaStream_t s)
{
    if (a.row1 <= a.row0) return cudaSuccess;
    dim3 grid(ceil_div(a.W, kPrepTileW), ceil_div(a.row1 - a.row0, kPrepTileH));
    if (!a.raw) {
        MEAO_LAUNCH((prepare_depth_kernel<false, true, IN_F32>), grid, kPrepThreads, 0, s, a);
    } else if (a.in_format == IN_D16) {
        if (a.reversed_z) MEAO_LAUNCH((prepare_depth_kernel<true, true, IN_D16>), grid, kPrepThreads, 0, s, a);
        else              MEAO_LAUNCH((prepare_depth_kernel<true, false, IN_D16>), grid, kPrepThreads, 0, s, a);
    } else if (a.in_format == IN_D24S8) {
        if (a.reversed_z) MEAO_LAUNCH((prepare_depth_kernel<true, true, IN_D24S8>), grid, kPrepThreads, 0, s, a);
        else              MEAO_LAUNCH((prepare_depth_kernel<true, false, IN_D24S8>), grid, kPrepThreads, 0, s, a);
    } else {
        if (a.reversed_z) MEAO_LAUNCH((prepare_depth_kernel<true, true, IN_F32>), grid, kPrepThreads, 0, s, a);
        else              MEAO_LAUNCH((prepare_depth_kernel<true, false, IN_F32>), grid, kPrepThreads, 0, s, a);
    }
    return cudaGetLastError();
}

#ifndef MEAO_EMULATE
cudaError_t preload_prepare_depth()
{
    cudaError_t e = cudaSuccess;
    auto t = [&](auto k) { if (e == cudaSuccess) e = preload_kernel(k); };
    t(prepare_depth_kernel<false, true, IN_F32>);
    t(prepare_depth_kernel<true, true, IN_F32>); t(prepare_depth_kernel<true, false, IN_F32>);
    t(prepare_depth_kernel<true, true, IN_D16>); t(prepare_depth_kernel<true, false, IN_D16>);
    t(prepare_depth_kernel<true, true, IN_D24S8>); t(prepare_depth_kernel<true, false, IN_D24S8>);
    return e;
}
#endif
#else   // prepare_depth_batch.cu
cudaError_t launch_prepare_depth_batch(const PrepareBatchArgs &b, int frames, cudaStream_t s)
{
    const PrepareArgs &a = b.base;
    if (a.row1 <= a.row0 || frames < 1) return cudaSuccess;
    dim3 grid(ceil_div(a.W, kPrepTileW), ceil_div(a.row1 - a.row0, kPrepTileH), frames);
    if (!a.raw) {
        MEAO_LAUNCH((prepare_depth_batch_kernel<false, true, IN_F32>), grid, kPrepThreads, 0, s, b);
    } else if (a.in_format == IN_D16) {
        if (a.reversed_z) MEAO_LAUNCH((prepare_depth_batch_kernel<true, true, IN_D16>), grid, kPrepThreads, 0, s, b);
        else              MEAO_LAUNCH((prepare_depth_batch_kernel<true, false, IN_D16>), grid, kPrepThreads, 0, s, b);
    } else if (a.in_format == IN_D24S8) {
        if (a.reversed_z) MEAO_LAUNCH((prepare_depth_batch_kernel<true, true, IN_D24S8>), grid, kPrepThreads, 0, s, b);
        else              MEAO_LAUNCH((prepare_depth_batch_kernel<true, false, IN_D24S8>), grid, kPrepThreads, 0, s, b);
    } else {
        if (a.reversed_z) MEAO_LAUNCH((prepare_depth_batch_kernel<true, true, IN_F32>), grid, kPrepThreads, 0, s, b);
        else              MEAO_LAUNCH((prepare_depth_batch_kernel<true, false, IN_F32>), grid, kPrepThreads, 0, s, b);
    }
    return cudaGetLastError();
}

#ifndef MEAO_EMULATE
cudaError_t preload_prepare_depth_batch()
{
    cudaError_t e = cudaSuccess;
    auto t = [&](auto k) { if (e == cudaSuccess) e = preload_kernel(k); };
    t(prepare_depth_batch_kernel<false, true, IN_F32>);
    t(prepare_depth_batch_kernel<true, true, IN_F32>); t(prepare_depth_batch_kernel<true, false, IN_F32>);
    t(prepare_depth_batch_kernel<true, true, IN_D16>); t(prepare_depth_batch_kernel<true, false, IN_D16>);
    t(prepare_depth_batch_kernel<true, true, IN_D24S8>); t(prepare_depth_batch_kernel<true, false, IN_D24S8>);
    return e;
}
#endif
#endif

}  // namespace meao
