// emu_batch_driver.cpp -- runs a batch of frames through the HOST-compiled batched kernel sources (TEST INFRASTRUCTURE ONLY,
// see ../emu/cuda_emu.h and cuda_emu_3d.h).  It is the single-frame driver of tests/emu (included whole: the same context,
// constants and buffer read-back) plus the launches of meao_render_batch, with the argument blocks filled the way meao_api.cu's
// recorders fill them for a batch.
#include "../emu/emu_driver.cpp"

namespace {

// The batch arena, laid out like meao_api.cu's reserve_batch: one frame slot = LinearDepth, LowDepth1-4, Occlusion1-4,
// Combined1-3, HighQuality1-4 with the single-frame pitches, slot size a multiple of 256 bytes.  Kept until the next batch.
struct EmuBatch {
    char *arena = nullptr;
    int frames = 0;
    size_t slot = 0, off_lin = 0, off_low[5] = {0}, off_occ[5] = {0}, off_comb[4] = {0}, off_hq[5] = {0};
    uint32_t tile_ctr[8] = {0};         // its own persistent-loop counters
};
EmuBatch g_batch;

// `e` with its buffer pointers moved to frame `frame` of the batch arena
Emu at_frame(const Emu *e, int frame)
{
    Emu x = *e;
    char *p = g_batch.arena + (size_t)frame * g_batch.slot;
    x.lin = (__half *)(p + g_batch.off_lin);
    for (int k = 1; k <= 4; k++) {
        x.low[k] = (float *)(p + g_batch.off_low[k]); x.occ[k] = (uint8_t *)(p + g_batch.off_occ[k]); x.hq[k] = (uint8_t *)(p + g_batch.off_hq[k]);
        if (k <= 3) x.comb[k] = (uint8_t *)(p + g_batch.off_comb[k]);
    }
    return x;
}

// what meao_api.cu's reserve_batch builds with a 3-D cuTensorMapEncodeTiled (see cuda_emu_3d.h for the encoding)
CUtensorMap make_map3(const void *base, int elem, int w, int h, int pitch_elems, int bw, int bh)
{
    CUtensorMap m = make_map(base, elem, w, h, pitch_elems, bw, bh);
    m.pad_[0] = (uint64_t)g_batch.frames; m.pad_[1] = g_batch.slot;
    return m;
}

void batch_downsample(Emu *x, const void *depth, int in_format, int frames)
{
    PrepareArgs a{};
    a.depth = depth; a.in_format = in_format; a.W = x->W; a.H = x->H; a.depth_row0 = 0; a.row0 = 0; a.row1 = x->H;
    a.lin = x->lin; a.lin_pitch = x->lin_pitch;
    for (int k = 1; k <= 4; k++) { a.low[k - 1] = x->low[k]; a.low_pitch[k - 1] = x->low_pitch[k]; }
    a.zbx = x->zbx; a.zby = x->zby; a.raw = x->raw; a.reversed_z = x->reversed_z;
    const long long in_frame = (long long)x->W * x->H * (in_format == 1 ? 2 : 4);
    a.vec_ok = (((uintptr_t)depth & 15) == 0) && (x->W % (in_format == 1 ? 8 : 4) == 0) && (in_frame % 16 == 0);
    launch_prepare_depth_batch(PrepareBatchArgs{a, in_frame, (long long)g_batch.slot}, frames, nullptr);
}

void batch_render(Emu *x, int k, bool wide, int frames)
{
    static const int idx_checker[7] = {1, 3, 4, 8, 11, 6, 10}, idx_exh[12] = {0, 1, 2, 3, 4, 8, 11, 5, 6, 7, 9, 10};
    const int n = x->exhaustive ? 12 : 7; const int *idx = x->exhaustive ? idx_exh : idx_checker;
    RenderArgs a{};
    a.low = x->low[k]; a.lw = x->lw[k]; a.lh = x->lh[k]; a.lpitch = x->low_pitch[k];
    a.occ = wide ? x->hq[k] : x->occ[k]; a.opitch = x->occ_pitch[k];
    a.sw = x->lw[k + 2]; a.sh = x->lh[k + 2];
    a.pad = __half2float(__float2half_rn(x->pad[k]));
    const float *it = wide ? x->inv_thickness_wide[k] : x->inv_thickness[k];
    for (int i = 0; i < n; i++) { a.inv_thickness[i] = it[idx[i]]; a.neg_front[i] = -(a.inv_thickness[i] - 0.5f); a.weight[i] = x->sample_weight[k][idx[i]]; }
    a.reject_fadeoff = x->reject_fadeoff; a.intensity = x->intensity;
    a.row0 = 0; a.row1 = x->lh[k]; a.wide = wide; a.exhaustive = x->exhaustive;
    int tv = x->ren_tile;
    if (tv < 0)             // meao_api.cu render_tile_variant, on the CTAs of all frames
        for (tv = 0; tv < kRenderTileVariants - 1; tv++)
            if ((long long)((x->lw[k] + 63) / 64) * ((a.row1 + kRenderTileHs[tv] - 1) / kRenderTileHs[tv]) * frames >= 148) break;
    a.tile_h = kRenderTileHs[tv];
    const CUtensorMap m = make_map3(x->low[k], 4, x->lw[k], x->lh[k], x->low_pitch[k], wide ? kRenderWideBoxW : kRenderBoxW, render_box_h(a.tile_h, wide));
    launch_render_ao_batch(m, x->use_tma != 0, RenderBatchArgs{a, (long long)g_batch.slot}, frames, nullptr);
}

void batch_upsample(Emu *x, int lo, uint8_t *out, int frames)
{
    const int hi = lo - 1;
    UpsampleArgs a{};
    a.lo_depth = x->low[lo]; a.low = x->lw[lo]; a.loh = x->lh[lo]; a.lo_dpitch = x->low_pitch[lo];
    a.lo_ao = (x->single_scale && lo == 1) ? x->occ[1] : (lo == 4) ? x->occ[4] : x->comb[lo]; a.lo_apitch = x->occ_pitch[lo];
    long long out_frame = (long long)g_batch.slot;
    if (hi == 0) { a.hi_depth = x->lin; a.hi_is_half = 1; a.hi_dpitch = x->lin_pitch; a.out = out; a.out_pitch = x->W; out_frame = (long long)x->W * x->H; }
    else { a.hi_depth = x->low[hi]; a.hi_is_half = 0; a.hi_dpitch = x->low_pitch[hi]; a.hi_ao = x->occ[hi]; a.hi_apitch = x->occ_pitch[hi]; a.out = x->comb[hi]; a.out_pitch = x->occ_pitch[hi]; }
    a.out_row_origin = 0;
    a.out_vec_ok = (((uintptr_t)a.out & 7) == 0) && (a.out_pitch % 8 == 0) && (out_frame % 8 == 0);
    a.hiw = x->lw[hi]; a.hih = x->lh[hi];
    a.noise_filter_strength = x->nfs[lo]; a.step_size = x->step[lo]; a.blur_tolerance = x->kblur[lo]; a.upsample_tolerance = x->tol[lo];
    auto safe = [](float v) { return v >= 8.673617379884035e-19f && v < 1152921504606846976.0f; };
    a.fast_div_ok = safe(a.upsample_tolerance) && safe(a.noise_filter_strength);
#if MEAO_UPS_STATIC_GUARD || MEAO_UPS_V2
    a.fast_div_ok = a.fast_div_ok && a.upsample_tolerance >= 2.7755575615628914e-17f && a.noise_filter_strength >= 2.220446049250313e-16f &&
                    a.noise_filter_strength < 288230376151711744.0f;
#endif
    a.row0 = 0; a.row1 = x->lh[hi];
    a.tile_ctr = g_batch.tile_ctr + 2 * (lo - 1);
    const bool premin = ((x->hq_mask >> (lo - 1)) & 1) != 0;
    const CUtensorMap md = make_map3(x->low[lo], 4, x->lw[lo], x->lh[lo], x->low_pitch[lo], kUpsDepthBoxW, kUpsDepthBoxH);
    const CUtensorMap ma = make_map3(a.lo_ao, 1, x->lw[lo], x->lh[lo], x->occ_pitch[lo], kUpsAoBoxW, kUpsAoBoxH);
    const CUtensorMap mh = make_map3(x->hq[lo], 1, x->lw[lo], x->lh[lo], x->occ_pitch[lo], kUpsAoBoxW, kUpsAoBoxH);
    const UpsampleBatchArgs ba{UpsamplePreminArgs{a, premin ? x->hq[lo] : nullptr, x->occ_pitch[lo]}, (long long)g_batch.slot, out_frame, frames, 0};
    launch_blur_upsample_batch(md, ma, &mh, x->use_tma != 0, ba, nullptr);
}

}  // namespace

extern "C" {

// `frames` frames stacked tightly in depth (16-byte aligned) -> out (frames x W x H codes), in record_frame order
void emu_run_batch(void *h, const void *depth, int in_format, int frames, uint8_t *out)
{
    Emu *e = (Emu *)h;
    free(g_batch.arena);
    g_batch = EmuBatch{};
    size_t off = 0;
    auto take = [&](size_t bytes) { size_t o = off; off += (bytes + 255) / 256 * 256; return o; };
    g_batch.off_lin = take((size_t)e->lin_pitch * e->lh[0] * 2);
    for (int k = 1; k <= 4; k++) {
        g_batch.off_low[k] = take((size_t)e->low_pitch[k] * e->lh[k] * 4);
        g_batch.off_occ[k] = take((size_t)e->occ_pitch[k] * e->lh[k]);
        if (k <= 3) g_batch.off_comb[k] = take((size_t)e->occ_pitch[k] * e->lh[k]);
        g_batch.off_hq[k] = take((size_t)e->occ_pitch[k] * e->lh[k]);
    }
    g_batch.slot = off; g_batch.frames = frames;
    g_batch.arena = alloc<char>(g_batch.slot * frames);
    Emu x = at_frame(e, 0);
    batch_downsample(&x, depth, in_format, frames);
    if (x.single_scale) { batch_render(&x, 1, false, frames); batch_upsample(&x, 1, out, frames); }
    else {
        for (int k = 1; k <= 4; k++) batch_render(&x, k, false, frames);
        for (int k = 1; k <= 4; k++) if ((x.hq_mask >> (k - 1)) & 1) batch_render(&x, k, true, frames);
        for (int lo = 4; lo >= 1; lo--) batch_upsample(&x, lo, lo == 1 ? out : nullptr, frames);
    }
    for (uint32_t c : g_batch.tile_ctr) if (c != 0) abort();      // the last CTA of every persistent launch re-armed its counters
}

// buffer <id> (1..16, 18..21) of frame <frame> of the last batch, like emu_get_buffer
int emu_get_batch_buffer(void *h, int frame, int id, void *out)
{
    if (frame < 0 || frame >= g_batch.frames || id == 17) return -1;
    Emu x = at_frame((Emu *)h, frame);
    return emu_get_buffer(&x, id, out);
}

}  // extern "C"
