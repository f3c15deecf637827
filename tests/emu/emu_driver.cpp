// emu_driver.cpp -- runs one frame through the HOST-compiled kernel sources (TEST INFRASTRUCTURE ONLY, see cuda_emu.h).
// It lays out one frame slot and builds every argument block and TMA map with libmeao's own host logic
// (miniengineao_b200/csrc/frame_plan.h); the per-dispatch constants are handed in by the test (which reads them from a
// plan-only libmeao context), so the planner itself is not duplicated here.  tests/emu_batch compiles this file with the
// 3-D TMA emulation and drives the same functions over a batch arena.
#include <cstdlib>
#include <cstring>
#include <vector>

#include "../../miniengineao_b200/csrc/common.cuh"
#include "../../miniengineao_b200/csrc/kernels.h"
#include "../../miniengineao_b200/csrc/frame_plan.h"

using namespace meao;

namespace {

template <class T> T *alloc(size_t n) { void *p = nullptr; if (posix_memalign(&p, 256, (n * sizeof(T) + 255) / 256 * 256 + 256)) abort(); memset(p, 0, n * sizeof(T)); return (T *)p; }

// The buffers a launch works in: the frame's own slot, or slot 0 of a batch (batch != nullptr, tests/emu_batch only).
struct EmuArena { FrameBufs bufs; uint32_t *tile_ctr; const BatchRun *batch; };

struct Emu {
    FrameGeom g;
    char *slot = nullptr;                   // one frame slot (SlotLayout)
    uint8_t *result = nullptr;
    uint32_t tile_ctr[8] = {0, 0, 0, 0, 0, 0, 0, 0};   // persistent blur_upsample grid: tile cursor + finished-CTA count per level
    EmuArena arena{};                       // the slot, its counters
    // constants (set by emu_set_constants)
    Plan plan{};
    MeaoVariants v = {0, 0, 0, 0};
    int raw = 1, reversed_z = 1;
    int use_tma = 1;        // 1: interior tiles take the kernels' TMA path (emulated box loads), 0: every tile gathers
    // row band (meao_set_row_band): rows of level k to PRODUCE, k = 0..4 (meao_band_rows "produce"); default = whole frame
    Range band{0, 0}, need[5] = {};
    int ren_tile = -1;      // render tile-height variant (index into kRenderTileHs); -1 = the planner's rule (render_tile_variant)
    BandFlags flags{};      // native neighbour exchange (band_exchange.cu)
    uint32_t host_error = 0;
};

// what libmeao's encode_map hands to cuTensorMapEncodeTiled; a batch: the 3-D map of tests/emu_batch/cuda_emu_3d.h
CUtensorMap emu_map(const MapSpec &s, const BatchRun *batch = nullptr)
{
    CUtensorMap m{};
    m.base = s.base; m.elem = s.elem; m.w = s.w; m.h = s.h; m.pitch_bytes = s.pitch_bytes; m.bw = s.bw; m.bh = s.bh;
    if (batch) { m.pad_[0] = (uint64_t)batch->frames; m.pad_[1] = (uint64_t)batch->slot_bytes; }
    return m;
}

// The three recorders of meao_api.cu; the batch launchers exist only in the tests/emu_batch build.
void run_downsample(Emu *e, const EmuArena &ar, const void *depth, int in_format)
{
    const PrepareArgs a = prepare_args(e->g, ar.bufs, e->plan, depth, in_format, e->raw != 0, e->reversed_z, e->band, ar.batch);
#ifdef MEAO_EMU_TMA_3D
    if (ar.batch) { launch_prepare_depth_batch(PrepareBatchArgs{a, ar.batch->in_frame_bytes, ar.batch->slot_bytes}, ar.batch->frames, nullptr); return; }
#endif
    launch_prepare_depth(a, nullptr);
}

void run_render(Emu *e, const EmuArena &ar, int k, bool wide)
{
    const int frames = ar.batch ? ar.batch->frames : 1;
    const int tv = e->ren_tile >= 0 ? e->ren_tile : render_tile_variant(e->g.lw[k], e->need[k], frames);
    const RenderArgs a = render_args(e->g, ar.bufs, e->plan, k, wide, e->v.sample_exhaustively != 0, e->raw != 0, e->need[k], tv);
    const CUtensorMap m = emu_map(render_map(e->g, ar.bufs, k, tv, wide), ar.batch);
#ifdef MEAO_EMU_TMA_3D
    if (ar.batch) { launch_render_ao_batch(m, e->use_tma != 0, RenderBatchArgs{a, ar.batch->slot_bytes}, frames, nullptr); return; }
#endif
    launch_render_ao(m, e->use_tma != 0, a, nullptr);
}

void run_upsample(Emu *e, const EmuArena &ar, int lo, uint8_t *ao_out)
{
    const UpsamplePreminArgs pa = upsample_args(e->g, ar.bufs, e->plan, e->v, lo, e->need[lo - 1], ao_out, e->result, e->band.lo,
                                                ar.tile_ctr, ar.batch);
    const CUtensorMap md = emu_map(ups_depth_map(e->g, ar.bufs, lo), ar.batch);
    const CUtensorMap ma = emu_map(ups_ao_map(e->g, pa.base.lo_ao, lo), ar.batch);
    const CUtensorMap mh = emu_map(ups_ao_map(e->g, ar.bufs.hq[lo], lo), ar.batch);
#ifdef MEAO_EMU_TMA_3D
    if (ar.batch) {
        const UpsampleBatchArgs ba{pa, ar.batch->slot_bytes, ups_out_frame_bytes(e->g, lo, *ar.batch), ar.batch->frames, 0};
        launch_blur_upsample_batch(md, ma, &mh, e->use_tma != 0, ba, nullptr);
        return;
    }
#endif
    launch_blur_upsample(md, ma, &mh, e->use_tma != 0, pa.base, pa.lo_ao2, pa.lo_a2pitch, nullptr);
}

// everything after the downsample, in meao_api.cu's record_frame order; ao_out = nullptr: the AO texture
void run_renders_upsamples(Emu *e, const EmuArena &ar, uint8_t *ao_out)
{
    const int kmax = e->v.single_scale ? 1 : 4;       // single-scale: Render level 1 + the final-style Upsample only
    for (int k = 1; k <= kmax; k++) run_render(e, ar, k, false);
    for (int k = 1; k <= kmax; k++) if (hq_level(e->v, k)) run_render(e, ar, k, true);
    for (int lo = kmax; lo >= 1; lo--) run_upsample(e, ar, lo, lo == 1 ? ao_out : nullptr);
}

// a buffer view in the reference layout / native type (meao_get_buffer)
void read_view(const Emu *e, const BufferView &v, void *out)
{
    if (v.slices == 16) {
        const int k = v.level;
        launch_synth_tiled((const float *)v.ptr, e->g.lw[k], e->g.lh[k], e->g.low_pitch[k], v.w, v.h, atlas_pad(e->plan, k, e->raw != 0), (__half *)out, nullptr);
        return;
    }
    for (int y = 0; y < v.h; y++) memcpy((char *)out + (size_t)y * v.w * v.elem, (const char *)v.ptr + (size_t)y * v.pitch_bytes, (size_t)v.w * v.elem);
}

}  // namespace

extern "C" {

void *emu_create(int W, int H)
{
    Emu *e = new Emu();
    e->g = frame_geom(W, H);
    const SlotLayout s = slot_layout(e->g);
    e->slot = alloc<char>(s.slot_bytes);
    e->result = alloc<uint8_t>((size_t)e->g.result_pitch * H);
    e->arena = EmuArena{frame_bufs(e->slot, s), e->tile_ctr, nullptr};
    e->band = Range{0, H};
    for (int k = 0; k <= 4; k++) e->need[k] = Range{0, e->g.lh[k]};
    return e;
}

void emu_destroy(void *h)
{
    Emu *e = (Emu *)h;
    free(e->slot); free(e->result);
    delete e;
}

// rc[k], rcw[k]: the 28 floats of meao_render_constants / meao_render_constants_wide (k = 1..4 at index k-1);
// uc[lo]: the 8 floats of meao_upsample_constants; zb: ZBufferParams; pad12: value of the DS1-written atlas padding texels
void emu_set_constants(void *h, const float *rc, const float *rcw, const float *uc, const float *zb, float pad12,
                       int raw, int reversed_z, int hq_mask, int exhaustive)
{
    Emu *e = (Emu *)h;
    Plan &p = e->plan;
    for (int k = 1; k <= 4; k++) {
        memcpy(p.inv_thickness[k], rc + 28 * (k - 1), 48);
        memcpy(p.sample_weight[k], rc + 28 * (k - 1) + 12, 48);
        memcpy(p.inv_thickness_wide[k], rcw + 28 * (k - 1), 48);
        p.pad[k] = (k <= 2) ? pad12 : 0.0f;
        const float *u = uc + 8 * (k - 1);
        p.noise_filter_strength[k] = u[4]; p.step_size[k] = u[5]; p.blur_tolerance[k] = u[6]; p.upsample_tolerance[k] = u[7];
    }
    p.reject_fadeoff = rc[26]; p.intensity = rc[27];
    memcpy(p.zb, zb, sizeof p.zb);
    e->raw = raw; e->reversed_z = reversed_z; e->v.high_quality_mask = hq_mask; e->v.sample_exhaustively = exhaustive;
}

// aborts (on purpose) with the emulated TMA's alignment complaint: an f32 box starting at x = 3
int emu_selfcheck_unaligned_tma()
{
    alignas(128) static float src[64 * 8], dst[16 * 4];
    const CUtensorMap m = emu_map(MapSpec{src, 4, 64, 8, 64 * 4, 16, 4});
    meao_emu::tma_load_2d(dst, &m, 3, 0);
    return 0;
}

long long emu_tma_box_loads() { return meao_emu::tma_box_loads; }

void emu_set_tma(void *h, int use_tma) { ((Emu *)h)->use_tma = use_tma; }
void emu_set_render_tile(void *h, int variant) { ((Emu *)h)->ren_tile = variant; }
void emu_set_single_scale(void *h, int on) { ((Emu *)h)->v.single_scale = on; }

// in_format: 0 = f32, 1 = D16 codes, 2 = D24S8 words (PrepareArgs.in_format); depth must be 16-byte aligned
void emu_run(void *h, const void *depth, int in_format)
{
    Emu *e = (Emu *)h;
    run_downsample(e, e->arena, depth, in_format);
    run_renders_upsamples(e, e->arena, nullptr);
}

// ---- native neighbour exchange: band_exchange_kernel with the segments meao_api.cu's record_exchange builds (whole pitched rows
// copied to the same position in the neighbour's LowDepth buffers).  up / down: the neighbours' Emu handles (NULL = none);
// rows_up8 / rows_down8 = meao_halo_rows(side, send = 1).  The fiber emulator runs one grid at a time, so the test presets the
// flags a concurrently running neighbour would have written (emu_band_flags).  Returns the kernel's sticky error.
int emu_band_exchange(void *h, void *up, void *down, const int *rows_up8, const int *rows_down8, int timeout_polls)
{
    Emu *e = (Emu *)h;
    Emu *peer[2] = {(Emu *)up, (Emu *)down};
    const int *rows8[2] = {rows_up8, rows_down8};
    if (e->flags.epoch == 0) e->flags.epoch = 1;
    XchgArgs a{}; a.nseg = 0;
    a.local = &e->flags; a.host_error = &e->host_error;
    a.timeout_ns = (unsigned long long)timeout_polls * 1000ull;       // the emulated global timer advances 1000 "ns" per read
    for (int side = 0; side < 2; side++) {
        if (!peer[side]) continue;
        if (peer[side]->flags.epoch == 0) peer[side]->flags.epoch = 1;
        a.peer[side] = &peer[side]->flags;
        for (int k = 1; k <= 4; k++) {
            const int lo = rows8[side][2 * (k - 1)], rows = rows8[side][2 * (k - 1) + 1] - lo;
            if (rows <= 0) continue;
            XchgSeg &g = a.seg[a.nseg++];
            g.src = (const uint4 *)(e->arena.bufs.low[k] + (size_t)lo * e->g.low_pitch[k]);
            g.dst = (uint4 *)(peer[side]->arena.bufs.low[k] + (size_t)lo * e->g.low_pitch[k]);
            g.n16 = (uint32_t)((size_t)rows * e->g.low_pitch[k] * sizeof(float) / 16); g.side = side;
        }
    }
    launch_band_exchange(a, nullptr);
    return (int)e->flags.error;
}
// out8 = ready[2], ack[2], epoch, done, error, host_error;  set8 (may be NULL) overwrites ready / ack first
void emu_band_flags(void *h, const int *set_ready_ack4, int *out8)
{
    Emu *e = (Emu *)h;
    if (set_ready_ack4) { for (int i = 0; i < 2; i++) { e->flags.ready[i] = set_ready_ack4[i]; e->flags.ack[i] = set_ready_ack4[2 + i]; } }
    if (out8) {
        out8[0] = e->flags.ready[0]; out8[1] = e->flags.ready[1]; out8[2] = e->flags.ack[0]; out8[3] = e->flags.ack[1];
        out8[4] = e->flags.epoch; out8[5] = e->flags.done; out8[6] = e->flags.error; out8[7] = e->host_error;
    }
}

// ---- row bands: the two phases of meao_band_phase_a / _b around the neighbour exchange ----------------------------------
// produce10 = meao_band_rows()[0..9]: rows of level k = 0..4 to produce; [row0, row1) = the band itself
void emu_set_band(void *h, int row0, int row1, const int *produce10)
{
    Emu *e = (Emu *)h;
    e->band = Range{row0, row1};
    for (int k = 0; k <= 4; k++) e->need[k] = Range{produce10[2 * k], produce10[2 * k + 1]};
}

// every LowDepth texel becomes NaN: rows this band neither produces nor receives must never reach an output
void emu_poison_low(void *h)
{
    Emu *e = (Emu *)h;
    for (int k = 1; k <= 4; k++) for (size_t i = 0; i < (size_t)e->g.low_pitch[k] * e->g.lh[k]; i++) e->arena.bufs.low[k][i] = __uint_as_float(0x7fc00000u);
}

// depth_band: the band's rows only (row1 - row0 rows), like meao_render_band_prepare
void emu_band_phase_a(void *h, const void *depth_band, int in_format) { Emu *e = (Emu *)h; run_downsample(e, e->arena, depth_band, in_format); }

// rows8 = meao_halo_rows(side, send): {lo1,hi1, ..., lo4,hi4}; packed message layout of meao_halo_pack (level 1 first, tight rows)
void emu_halo(void *h, const int *rows8, float *packed, int pack)
{
    Emu *e = (Emu *)h;
    HaloArgs a{}; a.nseg = 0;
    float *p = packed;
    for (int k = 1; k <= 4; k++) {
        const int lo = rows8[2 * (k - 1)], rows = rows8[2 * (k - 1) + 1] - lo;
        if (rows <= 0) continue;
        float *buf = e->arena.bufs.low[k] + (size_t)lo * e->g.low_pitch[k];
        HaloSeg &g = a.seg[a.nseg++];
        if (pack) g = HaloSeg{buf, p, e->g.low_pitch[k], e->g.lw[k], e->g.lw[k], rows};
        else      g = HaloSeg{p, buf, e->g.lw[k], e->g.low_pitch[k], e->g.lw[k], rows};
        p += (size_t)rows * e->g.lw[k];
    }
    launch_halo_copy(a, nullptr);
}

void emu_band_phase_b(void *h)
{
    Emu *e = (Emu *)h;
    run_renders_upsamples(e, e->arena, nullptr);
}

// buffer <id> (1..21) in the reference layout / native type, like meao_get_buffer
int emu_get_buffer(void *h, int id, void *out)
{
    Emu *e = (Emu *)h;
    BufferView v;
    if (!buffer_view(e->g, e->arena.bufs, e->result, id, &v)) return -1;
    read_view(e, v, out);
    return 0;
}

// the debug view of buffer <id> (meao_debug_view) into out[W * H]
int emu_debug_view(void *h, int id, uint8_t *out)
{
    Emu *e = (Emu *)h;
    BufferView v;
    if (!buffer_view(e->g, e->arena.bufs, e->result, id, &v)) return -1;
    launch_debug_view(debug_view_args(e->g, e->plan, v, e->raw != 0, out), nullptr);
    return 0;
}

// Blit.shader passes 1 / 2 on host buffers (launch_composite): color updated in place
void emu_composite(const uint8_t *ao, void *color, long long npix, int half, int rgb, int alpha, int one_minus)
{
    launch_composite(ao, color, npix, half, rgb, alpha, one_minus, nullptr);
}

void emu_composite_debug(const uint8_t *view, void *color, long long npix, int half) { launch_debug_composite(view, color, npix, half, nullptr); }

}  // extern "C"
