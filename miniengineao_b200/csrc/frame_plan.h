// frame_plan.h -- the host-side layout of one frame and the argument blocks of its launches.
//
// Pure functions and plain structs: no CUDA runtime call, no device code.  libmeao (meao_api.cu) builds every launch of a
// single frame, a row band and a batch from these, and so does the host emulator of tests/emu (g++ -DMEAO_EMULATE), so
// the emulated tests run the kernels fed by the same host logic as the product.
#pragma once

#include <stddef.h>
#include <stdint.h>

#include "../../include/meao.h"
#include "kernels.h"

namespace meao {

struct Range { int lo, hi; };   // [lo, hi)

inline int align_up(int x, int a) { return (x + a - 1) / a * a; }
inline float host_f16_round(float x) { return __half2float(__float2half_rn(x)); }

// Per-dispatch constants: the CPU half of RebuildCommandBuffers (AO.cs:496-540), filled by meao_api.cu's build_plan.
struct Plan {
    // Render (per level 1..4) -- AO.cs:660-734
    float inv_thickness[5][12];
    float sample_weight[5][12];
    float inv_slice_dim[5][2];
    float reject_fadeoff;
    float intensity;
    float pad[5];
    float inv_thickness_wide[5][12];       // the same for a NON-tiled source LowDepth<k> (kernel "main", AO.cs:679)
    float inv_slice_dim_wide[5][2];
    // Upsample (per lo level 1..4) -- AO.cs:750-771
    float inv_low[5][2], inv_high[5][2];
    float noise_filter_strength[5], step_size[5], blur_tolerance[5], upsample_tolerance[5];
    float zb[4];
};

// Level sizes (AO.cs:276-281) and row pitches in elements: rows start on 128-byte boundaries.
struct FrameGeom {
    int W = 0, H = 0;
    int lw[7] = {0}, lh[7] = {0};
    int lin_pitch = 0;                      // LinearDepth, f16
    int low_pitch[5] = {0};                 // LowDepth1..4, f32
    int occ_pitch[5] = {0};                 // Occlusion<k>, Combined<k> and HighQuality<k>, unorm8
    int result_pitch = 0;                   // the AO texture, unorm8
};

inline FrameGeom frame_geom(int W, int H)
{
    FrameGeom g;
    g.W = W; g.H = H;
    for (int l = 0; l < 7; l++) {
        const int div = 1 << l;
        g.lw[l] = (W + div - 1) / div;
        g.lh[l] = (H + div - 1) / div;
    }
    g.lin_pitch = align_up(g.lw[0], 64);
    g.result_pitch = align_up(g.lw[0], 128);
    for (int k = 1; k <= 4; k++) { g.low_pitch[k] = align_up(g.lw[k], 32); g.occ_pitch[k] = align_up(g.lw[k], 128); }
    return g;
}

// Reserves `bytes` at `off` (rounded up to 256 bytes) and returns its offset.
inline size_t take(size_t &off, size_t bytes)
{
    const size_t o = off;
    off += (bytes + 255) / 256 * 256;
    return o;
}

// One frame slot: every per-frame intermediate, at byte offsets from the slot's base.
struct SlotLayout {
    size_t lin = 0, low[5] = {0}, occ[5] = {0}, comb[4] = {0}, hq[5] = {0};
    size_t slot_bytes = 0;                  // a multiple of 256
};

inline SlotLayout slot_layout(const FrameGeom &g)
{
    SlotLayout s;
    size_t off = 0;
    s.lin = take(off, (size_t)g.lin_pitch * g.lh[0] * sizeof(__half));
    for (int k = 1; k <= 4; k++) {
        s.low[k] = take(off, (size_t)g.low_pitch[k] * g.lh[k] * sizeof(float));
        s.occ[k] = take(off, (size_t)g.occ_pitch[k] * g.lh[k]);
        if (k <= 3) s.comb[k] = take(off, (size_t)g.occ_pitch[k] * g.lh[k]);
        s.hq[k] = take(off, (size_t)g.occ_pitch[k] * g.lh[k]);
    }
    s.slot_bytes = off;
    return s;
}

// The buffers of one frame slot.
struct FrameBufs {
    __half *lin = nullptr;                  // LinearDepth
    float *low[5] = {nullptr};              // LowDepth1..4
    uint8_t *occ[5] = {nullptr};            // Occlusion1..4
    uint8_t *comb[4] = {nullptr};           // Combined1..3
    uint8_t *hq[5] = {nullptr};             // HighQuality1..4 (kernel "main" output)
};

inline FrameBufs frame_bufs(void *base, const SlotLayout &s)
{
    char *p = (char *)base;
    FrameBufs b;
    b.lin = (__half *)(p + s.lin);
    for (int k = 1; k <= 4; k++) {
        b.low[k] = (float *)(p + s.low[k]);
        b.occ[k] = (uint8_t *)(p + s.occ[k]);
        if (k <= 3) b.comb[k] = (uint8_t *)(p + s.comb[k]);
        b.hq[k] = (uint8_t *)(p + s.hq[k]);
    }
    return b;
}

// Value of the TiledDepth<k> atlas padding texels, f16-rounded: Linearize(0) for a raw depth ingest, 0 for a linear one.
inline float atlas_pad(const Plan &p, int k, bool raw) { return host_f16_round(raw ? p.pad[k] : 0.0f); }

// Buffer <id> (MEAO_BUF_*, 1..21) in the reference layout.  A TiledDepth<k> atlas (6..9) is never materialised: it is
// synthesised from LowDepth<k>, so `ptr` / `pitch_bytes` / `level` describe that source and w / h / slices / elem the atlas.
struct BufferView {
    void *ptr;
    size_t pitch_bytes;
    int level;                              // mip level of `ptr`
    int w, h, slices, elem;
    size_t bytes() const { return (size_t)w * h * slices * elem; }
};

inline bool buffer_view(const FrameGeom &g, const FrameBufs &b, uint8_t *result, int id, BufferView *v)
{
    if (id >= 6 && id <= 9) {                                   // TiledDepth<k>: 16 slices of level k + 2, f16
        const int k = id - 5;
        *v = BufferView{b.low[k], (size_t)g.low_pitch[k] * 4, k, g.lw[k + 2], g.lh[k + 2], 16, 2};
        return true;
    }
    void *p; int l, pitch, elem = 1;
    if (id == 1) { l = 0; p = b.lin; pitch = g.lin_pitch; elem = 2; }
    else if (id >= 2 && id <= 5) { l = id - 1; p = b.low[l]; pitch = g.low_pitch[l]; elem = 4; }
    else if (id >= 10 && id <= 13) { l = id - 9; p = b.occ[l]; pitch = g.occ_pitch[l]; }
    else if (id >= 14 && id <= 16) { l = id - 13; p = b.comb[l]; pitch = g.occ_pitch[l]; }
    else if (id == 17) { l = 0; p = result; pitch = g.result_pitch; }
    else if (id >= 18 && id <= 21) { l = id - 17; p = b.hq[l]; pitch = g.occ_pitch[l]; }
    else return false;
    *v = BufferView{p, (size_t)pitch * elem, l, g.lw[l], g.lh[l], 1, elem};
    return true;
}

inline bool hq_level(const MeaoVariants &v, int k) { return ((v.high_quality_mask >> (k - 1)) & 1) != 0; }
inline int depth_in_format(int kind) { return kind == MEAO_DEPTH_RAW_D16_UNORM ? 1 : (kind == MEAO_DEPTH_RAW_D24S8 ? 2 : 0); }
inline int depth_elem_bytes(int in_format) { return in_format == 1 ? 2 : 4; }


// The debug view of buffer view v (PushDebugBlitCommands, AO.cs:810-819) into out[W x H]
inline DebugViewArgs debug_view_args(const FrameGeom &g, const Plan &p, const BufferView &v, bool raw, uint8_t *out)
{
    DebugViewArgs a{};
    a.W = g.W; a.H = g.H; a.out = out; a.out_pitch = g.W;
    a.src = v.ptr; a.sw = v.w; a.sh = v.h;
    if (v.slices == 16) {                   // AO.cs:810-814: Blit.shader pass 4 on the atlas, read from LowDepth<k>
        a.tiled = 1; a.elem = 4; a.spitch = (int)(v.pitch_bytes / 4);
        a.lw = g.lw[v.level]; a.lh = g.lh[v.level];
        a.pad = atlas_pad(p, v.level, raw);
    } else {                                // AO.cs:815-819
        a.elem = v.elem; a.spitch = (int)(v.pitch_bytes / v.elem);
    }
    return a;
}

// A batch (meao_render_batch): frame f of every slot buffer is at its frame-0 pointer + f * slot_bytes.
struct BatchRun {
    int frames;
    long long in_frame_bytes;               // depth stride between frames (W * H * element size)
    long long slot_bytes;
};

// Bytes between the frames of the output of upsample `lo` in a batch: the caller's tight W x H frames, or the slots.
inline long long ups_out_frame_bytes(const FrameGeom &g, int lo, const BatchRun &batch)
{
    return lo == 1 ? (long long)g.W * g.H : batch.slot_bytes;
}

// Tile-height variant (index into kRenderTileHs = {32, 16, 8}) of a render producing `rows` of a level `lw` wide, over
// `frames` frames.  The big levels keep the 64 x 32 tile (least apron overhead: throughput); a level whose grid would not even
// put one CTA on every SM is latency-bound -- one CTA's serial time IS the kernel time -- so it takes the tallest tile that
// still gives >= 148 CTAs, else 64 x 8.  A batch counts the CTAs of all its frames.
// (Measured at 4K: level 2, 255 CTAs of 64 x 32, is FASTER with the big tile -- 14.0 vs 15.7 us -- levels 3 / 4 gain ~0.5 us.)
inline int render_tile_variant(int lw, Range rows, int frames)
{
    const int n = rows.hi - (rows.lo & ~3);
    for (int t = 0; t < kRenderTileVariants; t++) {
        const long long ctas = (long long)((lw + 63) / 64) * ((n + kRenderTileHs[t] - 1) / kRenderTileHs[t]) * frames;
        if (ctas >= 148) return t;
    }
    return kRenderTileVariants - 1;
}

// PushDownsampleCommands, AO.cs:604-658: rows `band` of the frame, depth[0] = row band.lo.
inline PrepareArgs prepare_args(const FrameGeom &g, const FrameBufs &b, const Plan &p, const void *depth, int in_format, bool raw,
                                int reversed_z, Range band, const BatchRun *batch)
{
    PrepareArgs a{};
    a.depth = depth;
    a.in_format = in_format;
    a.W = g.W; a.H = g.H;
    a.depth_row0 = band.lo;
    a.row0 = band.lo; a.row1 = band.hi;
    a.lin = b.lin; a.lin_pitch = g.lin_pitch;
    for (int k = 1; k <= 4; k++) { a.low[k - 1] = b.low[k]; a.low_pitch[k - 1] = g.low_pitch[k]; }
    a.zbx = p.zb[0]; a.zby = p.zb[1];
    a.raw = raw;
    a.reversed_z = reversed_z;
    // 16-byte loads: the depth pointer, every row and (a batch) every frame start 16-byte aligned
    a.vec_ok = (((uintptr_t)depth & 15) == 0) && (g.W % (in_format == 1 ? 8 : 4) == 0) && (!batch || batch->in_frame_bytes % 16 == 0);
    return a;
}

// PushRenderCommands, AO.cs:660-748, producing `rows` of level k with tile variant `tv`.  wide = false: the call
// AmbientOcclusion.cs makes (tiled source, kernel main_interleaved) -> Occlusion<k>; wide = true: the same recorder for the
// non-tiled source LowDepth<k> (kernel main) -> HighQuality<k>.
inline RenderArgs render_args(const FrameGeom &g, const FrameBufs &b, const Plan &p, int k, bool wide, bool exhaustive, bool raw,
                              Range rows, int tv)
{
    static const int idx_checker[7] = {1, 3, 4, 8, 11, 6, 10};                       // Render.compute:162-168 table slots, call order
    static const int idx_exh[12] = {0, 1, 2, 3, 4, 8, 11, 5, 6, 7, 9, 10};           // Render.compute:148-159
    const int n = exhaustive ? 12 : 7;
    const int *idx = exhaustive ? idx_exh : idx_checker;
    RenderArgs a{};
    a.low = b.low[k]; a.lw = g.lw[k]; a.lh = g.lh[k]; a.lpitch = g.low_pitch[k];
    a.occ = wide ? b.hq[k] : b.occ[k]; a.opitch = g.occ_pitch[k];
    a.sw = g.lw[k + 2]; a.sh = g.lh[k + 2];
    a.pad = atlas_pad(p, k, raw);
    const float *it = wide ? p.inv_thickness_wide[k] : p.inv_thickness[k];
    for (int i = 0; i < n; i++) {
        a.inv_thickness[i] = it[idx[i]];
        a.neg_front[i] = -(a.inv_thickness[i] - 0.5f);                                               // Render.compute:85
        a.weight[i] = p.sample_weight[k][idx[i]];
    }
    a.reject_fadeoff = p.reject_fadeoff;
    a.intensity = p.intensity;
    a.row0 = rows.lo; a.row1 = rows.hi;
    a.wide = wide ? 1 : 0;
    a.exhaustive = exhaustive ? 1 : 0;
    a.tile_h = kRenderTileHs[tv];
    return a;
}

// LoResAO1 of upsample `lo`: Occlusion1 alone when single-scale (no coarser level contributes), else Occlusion4 or Combined<lo>.
inline uint8_t *lo_res_ao(const FrameBufs &b, int lo, bool single_scale)
{
    return (single_scale && lo == 1) ? b.occ[1] : (lo == 4) ? b.occ[4] : b.comb[lo];
}

// upsample_tolerance and noise_filter_strength allow the kernel's fast division (blur_upsample.cu)
inline bool fast_div_ok(float upsample_tolerance, float noise_filter_strength)
{
    auto safe = [](float x) { return x >= 8.673617379884035e-19f && x < 1152921504606846976.0f; };
    bool ok = safe(upsample_tolerance) && safe(noise_filter_strength);
#if MEAO_UPS_STATIC_GUARD || MEAO_UPS_V2
    // 2^-55, 2^-52, 2^59: with these bounds total / num of the final division are provably inside the fast-division range
    ok = ok && upsample_tolerance >= 2.7755575615628914e-17f && noise_filter_strength >= 2.220446049250313e-16f &&
         noise_filter_strength < 288230376151711744.0f;
#endif
    return ok;
}

// PushUpsampleCommands with the wiring of AO.cs:528-531, producing `hi_rows` of level lo - 1.  The final upsample (lo = 1)
// writes ao_out (rows from band0 on, pitch W) or, when ao_out is null, the context's AO texture `result`.  premin: LoResAO2 =
// HighQuality<lo> (kernels main_premin / main_premin_blendout).
inline UpsamplePreminArgs upsample_args(const FrameGeom &g, const FrameBufs &b, const Plan &p, const MeaoVariants &v, int lo, Range hi_rows,
                                        uint8_t *ao_out, uint8_t *result, int band0, uint32_t *tile_ctr, const BatchRun *batch)
{
    const int hi = lo - 1;
    UpsampleArgs a{};
    a.lo_depth = b.low[lo]; a.low = g.lw[lo]; a.loh = g.lh[lo]; a.lo_dpitch = g.low_pitch[lo];
    a.lo_ao = lo_res_ao(b, lo, v.single_scale != 0); a.lo_apitch = g.occ_pitch[lo];
    if (hi == 0) { a.hi_depth = b.lin; a.hi_is_half = 1; a.hi_dpitch = g.lin_pitch; a.hi_ao = nullptr; a.hi_apitch = 0; }
    else { a.hi_depth = b.low[hi]; a.hi_is_half = 0; a.hi_dpitch = g.low_pitch[hi]; a.hi_ao = b.occ[hi]; a.hi_apitch = g.occ_pitch[hi]; }
    if (hi > 0) { a.out = b.comb[hi]; a.out_pitch = g.occ_pitch[hi]; a.out_row_origin = 0; }
    else if (ao_out) { a.out = ao_out; a.out_pitch = g.W; a.out_row_origin = band0; }
    else { a.out = result; a.out_pitch = g.result_pitch; a.out_row_origin = 0; }
    a.out_vec_ok = (((uintptr_t)a.out & 7) == 0) && (a.out_pitch % 8 == 0) && (!batch || ups_out_frame_bytes(g, lo, *batch) % 8 == 0);
    a.hiw = g.lw[hi]; a.hih = g.lh[hi];
    a.noise_filter_strength = p.noise_filter_strength[lo];
    a.step_size = p.step_size[lo];
    a.blur_tolerance = p.blur_tolerance[lo];
    a.upsample_tolerance = p.upsample_tolerance[lo];
    a.fast_div_ok = fast_div_ok(a.upsample_tolerance, a.noise_filter_strength);
    a.row0 = hi_rows.lo; a.row1 = hi_rows.hi;
    a.tile_ctr = tile_ctr + 2 * (lo - 1);
    return UpsamplePreminArgs{a, hq_level(v, lo) ? b.hq[lo] : nullptr, g.occ_pitch[lo]};
}

// ---- TMA maps: what cuTensorMapEncodeTiled is given for each map family (elem 4: f32, 1: unorm8) ---------------------------
// libmeao encodes a 2-D map per spec for its single-frame arena, or a 3-D map (w, h, capacity) with the slot stride for the
// batch arena; the emulator builds its CUtensorMap stand-in from the same spec.
struct MapSpec { const void *base; int elem, w, h; size_t pitch_bytes; int bw, bh; };

inline MapSpec render_map(const FrameGeom &g, const FrameBufs &b, int k, int tv, bool wide)
{
    return MapSpec{b.low[k], 4, g.lw[k], g.lh[k], (size_t)g.low_pitch[k] * 4, wide ? kRenderWideBoxW : kRenderBoxW, render_box_h(kRenderTileHs[tv], wide)};
}
inline MapSpec ups_depth_map(const FrameGeom &g, const FrameBufs &b, int lo)
{
    return MapSpec{b.low[lo], 4, g.lw[lo], g.lh[lo], (size_t)g.low_pitch[lo] * 4, kUpsDepthBoxW, kUpsDepthBoxH};
}
// an AO buffer of level lo read by upsample lo (LoResAO1 or LoResAO2)
inline MapSpec ups_ao_map(const FrameGeom &g, const uint8_t *ao, int lo)
{
    return MapSpec{ao, 1, g.lw[lo], g.lh[lo], (size_t)g.occ_pitch[lo], kUpsAoBoxW, kUpsAoBoxH};
}

}  // namespace meao
