// render_ao.cu -- stage 2 of the SSAO pipe: volumetric-obscurance sampling at one mip level.
//
// Replaces Render.compute kernel main_interleaved (TestSamplePair :60-75, TestSamples :77-110,
// MAIN :112-177) for TiledDepth<k> -> Occlusion<k>.
//
// Design (not a port): the reference deinterleaves depth into 16 slices so that its sparse taps
// become unit-stride texture fetches.  Here the level-k depth stays in NATURAL layout: one CTA
// stages a (64+32) x (32+32) f32 tile of LowDepth<k> in shared memory with a single TMA box load,
// rounds it to f16 in place (the reference samples an RHalf atlas), and every thread then reads
// its 36 taps at stride 4 texels -- which, across a warp of consecutive pixels, is unit-stride and
// bank-conflict free.  A thread owns two horizontally adjacent pixels so each tap is one LDS.64.
//
// Virtual atlas semantics that must be preserved (SURVEY.md P3): pixel (X,Y) of level k lives in
// slice (X&3, Y&3) at slice texel (X>>2, Y>>2); a tap (di,dj) reads slice texel
// (clamp(i+di, 0, sw-1), clamp(j+dj, 0, sh-1)), i.e. natural pixel (4*ci + (X&3), 4*cj + (Y&3)),
// which is a padding texel (value `pad`) when it lies outside level k.  Tiles whose footprint is
// entirely inside the level need none of this and take the TMA path; border tiles resolve the
// clamp/padding per texel with a gather from global memory.
//
// Bound: instruction issue (about 250 thread-instructions per output, 2 B + 1 B of HBM traffic).
//
// Variants (SURVEY.md 8f.2; shipped in Render.compute but never dispatched by AmbientOcclusion.cs):
//   MODE 1 = kernel `main` (WIDE_SAMPLING, REN:27-29,46-50,79-82,115-116,125,136,174): plain f32 Texture2D
//            source (LowDepth<k> itself, no f16 rounding, no atlas), taps at 2x the offsets, per-texel
//            clamp-to-edge in level space, output at the same resolution -> HighQuality<k>.  Same CTA
//            shape; the apron shrinks to 8 texels (TMA box 80 x 48) and the tap stride to 2.
//   EXH      = #define SAMPLE_EXHAUSTIVELY (REN:144-159): twelve TestSamples calls (68 taps) instead of seven (36).
#include "common.cuh"
#include "kernels.h"

namespace meao {

namespace {

#ifndef MEAO_REN_THREADS
#define MEAO_REN_THREADS 256
#endif
constexpr int kTW = 64;                     // outputs per CTA: 64 x TH, TH = 32 (64x32 / 256 threads measured 2 % faster than 64x16 / 128 in the
                                            // 3-stream frame pipeline), 16 or 8 for the latency-bound coarse levels (kernels.h kRenderTileHs)
// MODE 0 (main_interleaved): apron 4 slice texels x stride 4 = 16; MODE 1 (main, wide): apron 4 taps x stride 2 = 8
template <int MODE> constexpr int kTapStride = MODE == 0 ? 4 : 2;
template <int MODE, int TH> struct Geo {
    static constexpr int kAp = MODE == 0 ? 16 : 8;
    static constexpr int kSW = kTW + 2 * kAp;       // 96 == kRenderBoxW      | 80 == kRenderWideBoxW
    static constexpr int kSH = TH + 2 * kAp;        // == render_box_h(TH, MODE == 1)
};
#ifndef MEAO_REN_MINB
#define MEAO_REN_MINB 6
#endif
constexpr int kThreads = MEAO_REN_THREADS;
constexpr int kWarps = kThreads / 32;
static_assert(Geo<0, 32>::kSW == kRenderBoxW && Geo<1, 32>::kSW == kRenderWideBoxW, "TMA box mismatch");
static_assert(Geo<0, 32>::kSH == render_box_h(32, false) && Geo<1, 8>::kSH == render_box_h(8, true), "TMA box mismatch");

// Render.compute:60-75 for one sample pair, TWO horizontally adjacent pixels at once (.x / .y lanes).
//   * clamp(d, p, 1) == max(saturate(d), p) for p in [0,1], including d = NaN/+-inf (HLSL min/max return
//     the non-NaN operand, saturate(NaN) = 0), so the result is bit-identical to the reference expression;
//   * the kernel is issue-bound, so everything that has no .SAT / min-max flavour runs as packed f32x2
//     (FFMA2 / FADD2 / FMUL2: two IEEE fp32 operations per lane per issue slot, lane-wise identical to the
//     scalar instruction).
__device__ __forceinline__ float2 pair_eval2(float2 S1, float2 S2, float2 inv_range, float2 neg_front, float rf)
{
    const float2 d1 = __ffma2_rn(S1, inv_range, neg_front);             // REN:65
    const float2 d2 = __ffma2_rn(S2, inv_range, neg_front);             // REN:66
    const float p1x = __saturatef(__fmul_rn(rf, d1.x)), p1y = __saturatef(__fmul_rn(rf, d1.y));   // REN:68
    const float p2x = __saturatef(__fmul_rn(rf, d2.x)), p2y = __saturatef(__fmul_rn(rf, d2.y));   // REN:69
    // clamp(d, p, 1): either max(saturate(d), p) (FADD.SAT on the FMA pipe + FMNMX) or the literal
    // min(max(d, p), 1) (two FMNMX on the ALU pipe); both are exact, the mix balances the two pipes
#ifndef MEAO_REN_CLAMP_MODE
#define MEAO_REN_CLAMP_MODE 1
#endif
#if MEAO_REN_CLAMP_MODE == 0
    const float2 c1 = make_float2(fmaxf(__saturatef(d1.x), p2x), fmaxf(__saturatef(d1.y), p2y));
    const float2 c2 = make_float2(fmaxf(__saturatef(d2.x), p1x), fmaxf(__saturatef(d2.y), p1y));
#elif MEAO_REN_CLAMP_MODE == 1
    const float2 c1 = make_float2(fmaxf(__saturatef(d1.x), p2x), fmaxf(__saturatef(d1.y), p2y));
    const float2 c2 = make_float2(fminf(fmaxf(d2.x, p1x), 1.0f), fminf(fmaxf(d2.y, p1y), 1.0f));
#else
    const float2 c1 = make_float2(fminf(fmaxf(d1.x, p2x), 1.0f), fminf(fmaxf(d1.y, p2y), 1.0f));
    const float2 c2 = make_float2(fminf(fmaxf(d2.x, p1x), 1.0f), fminf(fmaxf(d2.y, p1y), 1.0f));
#endif
    const float2 sum = __fadd2_rn(c1, c2);
    return make_float2(__saturatef(fmaf(-p1x, p2x, sum.x)), __saturatef(fmaf(-p1y, p2y, sum.y)));   // REN:71-74
}

// c points at the (left) centre texel in the smem tile
template <int MODE, int DX, int DY>
__device__ __forceinline__ float2 pair2(const float *c, float2 ir, float2 nf, float rf)
{
    constexpr int OFF = (kTapStride<MODE> * DY) * Geo<MODE, 32>::kSW + kTapStride<MODE> * DX;    // the tile width does not depend on TH
    const float2 s1 = *reinterpret_cast<const float2 *>(c + OFF);
    const float2 s2 = *reinterpret_cast<const float2 *>(c - OFF);
    return pair_eval2(s1, s2, ir, nf, rf);
}

// Render.compute:87-93 (axial), x = N
template <int MODE, int N>
__device__ __forceinline__ void axial2(const float *c, float2 inv, float it, float nfs, float w, float rf, float2 &ao)
{
    const float2 ir = __fmul2_rn(make_float2(it, it), inv), nf = make_float2(nfs, nfs);      // REN:84
    const float2 a = pair2<MODE, N, 0>(c, ir, nf, rf);
    const float2 b = pair2<MODE, 0, N>(c, ir, nf, rf);
    ao = __ffma2_rn(make_float2(w, w), __fmul2_rn(make_float2(0.5f, 0.5f), __fadd2_rn(a, b)), ao);
}
// Render.compute:94-100 (diagonal), x == y == N: offsets x*TILE - x, x*TILE + x
template <int MODE, int N>
__device__ __forceinline__ void diag2(const float *c, float2 inv, float it, float nfs, float w, float rf, float2 &ao)
{
    const float2 ir = __fmul2_rn(make_float2(it, it), inv), nf = make_float2(nfs, nfs);
    const float2 a = pair2<MODE, -N, N>(c, ir, nf, rf);
    const float2 b = pair2<MODE, N, N>(c, ir, nf, rf);
    ao = __ffma2_rn(make_float2(w, w), __fmul2_rn(make_float2(0.5f, 0.5f), __fadd2_rn(a, b)), ao);
}
// Render.compute:101-109 (L-shaped): y*T + x, y*T - x, x*T + y, x*T - y
template <int MODE, int X, int Y>
__device__ __forceinline__ void lshape2(const float *c, float2 inv, float it, float nfs, float w, float rf, float2 &ao)
{
    const float2 ir = __fmul2_rn(make_float2(it, it), inv), nf = make_float2(nfs, nfs);
    const float2 a = pair2<MODE, X, Y>(c, ir, nf, rf);
    const float2 b = pair2<MODE, -X, Y>(c, ir, nf, rf);
    const float2 cc = pair2<MODE, Y, X>(c, ir, nf, rf);
    const float2 d = pair2<MODE, -Y, X>(c, ir, nf, rf);
    const float2 t = __fadd2_rn(__fadd2_rn(__fadd2_rn(a, b), cc), d);
    ao = __ffma2_rn(make_float2(w, w), __fmul2_rn(make_float2(0.25f, 0.25f), t), ao);
}

// (built a second time with MEAO_REN_BATCH = 1 by render_ao_batch.cu: the batched kernels and their launcher)
#ifndef MEAO_REN_BATCH
#define MEAO_REN_BATCH 0
#endif
#include "render_ao_kernel.inc"

#if !MEAO_REN_BATCH
// debug view: TiledDepth<k>[slice][j][i] exactly as Downsample1/2 would have written it
__global__ void synth_tiled_kernel(const float *low, int lw, int lh, int lpitch, int sw, int sh, float pad, __half *out)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x, j = blockIdx.y, s = blockIdx.z;
    if (i >= sw) return;
    const int x = 4 * i + (s & 3), y = 4 * j + (s >> 2);                     // inverse of DS1:69,71
    float v = pad;
    if (x < lw && y < lh) v = low[(size_t)y * lpitch + x];
    out[((size_t)s * sh + j) * sw + i] = __float2half_rn(v);
}
#endif

}  // namespace

#if !MEAO_REN_BATCH
template <int MODE, bool EXH, int TH>
static void launch_render_variant(const CUtensorMap &low_map, int t, const RenderArgs &a, dim3 grid, cudaStream_t s)
{
    const size_t smem = (size_t)Geo<MODE, TH>::kSW * Geo<MODE, TH>::kSH * sizeof(float);
    MEAO_LAUNCH((render_ao_kernel<MODE, EXH, TH>), grid, kThreads, smem, s, low_map, a, t);
}
template <int MODE, bool EXH>
static cudaError_t launch_render_th(const CUtensorMap &low_map, int t, const RenderArgs &a, int gx, int rows, cudaStream_t s)
{
    switch (a.tile_h) {
        case kRenderTileHs[0]: launch_render_variant<MODE, EXH, kRenderTileHs[0]>(low_map, t, a, dim3(gx, ceil_div(rows, kRenderTileHs[0])), s); break;
        case kRenderTileHs[1]: launch_render_variant<MODE, EXH, kRenderTileHs[1]>(low_map, t, a, dim3(gx, ceil_div(rows, kRenderTileHs[1])), s); break;
        case kRenderTileHs[2]: launch_render_variant<MODE, EXH, kRenderTileHs[2]>(low_map, t, a, dim3(gx, ceil_div(rows, kRenderTileHs[2])), s); break;
        default: return cudaErrorInvalidValue;
    }
    return cudaGetLastError();
}

cudaError_t launch_render_ao(const CUtensorMap &low_map, bool use_tma, const RenderArgs &a, cudaStream_t s)
{
    if (a.row1 <= a.row0) return cudaSuccess;
    const int ybase = a.row0 & ~3;
    const int gx = ceil_div(a.lw, kTW), rows = a.row1 - ybase;
    const int t = use_tma ? 1 : 0;
    if (!a.wide) return a.exhaustive ? launch_render_th<0, true>(low_map, t, a, gx, rows, s) : launch_render_th<0, false>(low_map, t, a, gx, rows, s);
    return a.exhaustive ? launch_render_th<1, true>(low_map, t, a, gx, rows, s) : launch_render_th<1, false>(low_map, t, a, gx, rows, s);
}

cudaError_t launch_synth_tiled(const float *low, int lw, int lh, int lpitch, int sw, int sh, float pad,
                               __half *out, cudaStream_t s)
{
    dim3 grid(ceil_div(sw, 128), sh, 16);
    MEAO_LAUNCH((synth_tiled_kernel), grid, 128, 0, s, low, lw, lh, lpitch, sw, sh, pad, out);
    return cudaGetLastError();
}

#ifndef MEAO_EMULATE
cudaError_t preload_render_ao()
{
    cudaError_t e = cudaSuccess;
    auto t = [&](auto k) { if (e == cudaSuccess) e = preload_kernel(k); };
    t(render_ao_kernel<0, false, 32>); t(render_ao_kernel<0, false, 16>); t(render_ao_kernel<0, false, 8>);
    t(render_ao_kernel<0, true, 32>); t(render_ao_kernel<0, true, 16>); t(render_ao_kernel<0, true, 8>);
    t(render_ao_kernel<1, false, 32>); t(render_ao_kernel<1, false, 16>); t(render_ao_kernel<1, false, 8>);
    t(render_ao_kernel<1, true, 32>); t(render_ao_kernel<1, true, 16>); t(render_ao_kernel<1, true, 8>);
    t(synth_tiled_kernel);
    return e;
}
#endif
#else   // render_ao_batch.cu
template <int MODE, bool EXH, int TH>
static void launch_render_batch_variant(const CUtensorMap &low_map, int t, const RenderBatchArgs &a, dim3 grid, cudaStream_t s)
{
    const size_t smem = (size_t)Geo<MODE, TH>::kSW * Geo<MODE, TH>::kSH * sizeof(float);
    MEAO_LAUNCH((render_ao_batch_kernel<MODE, EXH, TH>), grid, kThreads, smem, s, low_map, a, t);
}
template <int MODE, bool EXH>
static cudaError_t launch_render_batch_th(const CUtensorMap &low_map, int t, const RenderBatchArgs &b, int gx, int rows, int frames, cudaStream_t s)
{
    switch (b.base.tile_h) {
        case kRenderTileHs[0]: launch_render_batch_variant<MODE, EXH, kRenderTileHs[0]>(low_map, t, b, dim3(gx, ceil_div(rows, kRenderTileHs[0]), frames), s); break;
        case kRenderTileHs[1]: launch_render_batch_variant<MODE, EXH, kRenderTileHs[1]>(low_map, t, b, dim3(gx, ceil_div(rows, kRenderTileHs[1]), frames), s); break;
        case kRenderTileHs[2]: launch_render_batch_variant<MODE, EXH, kRenderTileHs[2]>(low_map, t, b, dim3(gx, ceil_div(rows, kRenderTileHs[2]), frames), s); break;
        default: return cudaErrorInvalidValue;
    }
    return cudaGetLastError();
}

cudaError_t launch_render_ao_batch(const CUtensorMap &low_map3, bool use_tma, const RenderBatchArgs &b, int frames, cudaStream_t s)
{
    const RenderArgs &a = b.base;
    if (a.row1 <= a.row0 || frames < 1) return cudaSuccess;
    const int ybase = a.row0 & ~3;
    const int gx = ceil_div(a.lw, kTW), rows = a.row1 - ybase;
    const int t = use_tma ? 1 : 0;
    if (!a.wide) return a.exhaustive ? launch_render_batch_th<0, true>(low_map3, t, b, gx, rows, frames, s) : launch_render_batch_th<0, false>(low_map3, t, b, gx, rows, frames, s);
    return a.exhaustive ? launch_render_batch_th<1, true>(low_map3, t, b, gx, rows, frames, s) : launch_render_batch_th<1, false>(low_map3, t, b, gx, rows, frames, s);
}

#ifndef MEAO_EMULATE
cudaError_t preload_render_ao_batch()
{
    cudaError_t e = cudaSuccess;
    auto t = [&](auto k) { if (e == cudaSuccess) e = preload_kernel(k); };
    t(render_ao_batch_kernel<0, false, 32>); t(render_ao_batch_kernel<0, false, 16>); t(render_ao_batch_kernel<0, false, 8>);
    t(render_ao_batch_kernel<0, true, 32>); t(render_ao_batch_kernel<0, true, 16>); t(render_ao_batch_kernel<0, true, 8>);
    t(render_ao_batch_kernel<1, false, 32>); t(render_ao_batch_kernel<1, false, 16>); t(render_ao_batch_kernel<1, false, 8>);
    t(render_ao_batch_kernel<1, true, 32>); t(render_ao_batch_kernel<1, true, 16>); t(render_ao_batch_kernel<1, true, 8>);
    return e;
}
#endif
#endif

}  // namespace meao
