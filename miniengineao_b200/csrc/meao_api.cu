// meao_api.cu -- context, planner and C ABI of libmeao.so (see include/meao.h).
//
// Host-side mirror of the parts of AmbientOcclusion.cs that own the hot path:
//   RTHandle geometry/formats (AO.cs:124-282), the CPU constant math of the three Push*Commands
//   recorders (AO.cs:561-593, 660-734, 750-771), the record order of RebuildCommandBuffers
//   (AO.cs:511-531) and the re-plan triggers of LateUpdate (AO.cs:329-350).
// "Plan once, replay per frame" maps to: constants + TMA descriptors are rebuilt only when a
// parameter, the camera or the size changes; a frame is then ten kernel launches (or one CUDA
// graph launch) on one stream.
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <cmath>
#include <functional>
#include <map>
#include <mutex>
#include <string>
#include <vector>
#include <unistd.h>

#include <nvtx3/nvToolsExt.h>

#include "../../include/meao.h"
#include "common.cuh"
#include "kernels.h"

using namespace meao;

namespace {

thread_local std::string g_create_error;

struct Range { int lo, hi; };   // [lo, hi)
inline Range clampr(Range r, int n) { Range o{r.lo < 0 ? 0 : r.lo, r.hi > n ? n : r.hi}; if (o.hi < o.lo) o.hi = o.lo; return o; }
inline int align_up(int x, int a) { return (x + a - 1) / a * a; }

// cuTensorMapEncodeTiled is fetched through the runtime so libmeao.so has no link-time
// dependency on libcuda (it must load on a machine without a driver for the ABI tests).
typedef CUresult (*PFN_encodeTiled)(CUtensorMap *, CUtensorMapDataType, cuuint32_t, void *, const cuuint64_t *,
                                    const cuuint64_t *, const cuuint32_t *, const cuuint32_t *, CUtensorMapInterleave,
                                    CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

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

// Batch arena (meao_render_batch): `capacity` frame slots of every intermediate, apart from the single-frame arena so that a
// batch never disturbs meao_get_buffer / debug views / stage calls / the band flags.  Frame f of a buffer is at ptr + f * slot_bytes.
struct BatchArena {
    void *base = nullptr;
    size_t bytes = 0, slot_bytes = 0;
    int capacity = 0;
    int last_frames = 0;                    // frames of the last batch (meao_get_batch_buffer)
    int last_kind = MEAO_DEPTH_RAW_F32;
    uint32_t *tile_ctr = nullptr;           // its own persistent-loop counters: a batch and a single frame never share a word
    __half *lin = nullptr;
    float *low[5] = {nullptr};
    uint8_t *occ[5] = {nullptr}, *comb[4] = {nullptr}, *hq[5] = {nullptr};
    bool tma_ok = false;
    // 3-D maps (w, h, capacity), strides (pitch, slot_bytes); same boxes as the single-frame maps
    CUtensorMap map_low_ren[kRenderTileVariants][5], map_low_wide[kRenderTileVariants][5];
    CUtensorMap map_low_ups[5], map_ao_ups[5], map_hq_ups[5], map_occ1_ups;
};

// what the recorders need to know about a batched launch (nullptr: the single-frame path, today's launches)
struct BatchRun {
    int frames;
    long long in_frame_bytes;               // depth stride between frames (W * H * element size)
};

}  // namespace

struct MeaoCtx {
    int device = 0;
    bool plan_only = false;                 // device < 0: host-side planning only (no CUDA calls at all)
    uint32_t flags = 0;
    std::string error;
    cudaStream_t stream = nullptr;
    cudaStream_t branch[3] = {nullptr, nullptr, nullptr};   // forked capture streams: the graph runs independent levels side by side
    cudaEvent_t ev[5] = {nullptr, nullptr, nullptr, nullptr, nullptr};
    PFN_encodeTiled encode = nullptr;

    MeaoParams params;
    MeaoCamera camera;
    MeaoVariants variants = {0, 0, 0, 0};
    bool plan_dirty = true;
    Plan plan;

    int W = 0, H = 0;
    int lw[7] = {0}, lh[7] = {0};
    // band (global L0 rows) + neighbours
    int band0 = 0, band1 = 0, prev0 = -1, next1 = -1;

    // device buffers (natural layout, pitched, global coordinates)
    void *arena = nullptr;
    size_t arena_bytes = 0;
    __half *lin = nullptr; int lin_pitch = 0;
    float *low[5] = {nullptr}; int low_pitch[5] = {0};
    uint8_t *occ[5] = {nullptr}; int occ_pitch[5] = {0};
    uint8_t *comb[4] = {nullptr};           // same pitch as occ of that level
    uint8_t *hq[5] = {nullptr};             // HighQuality<k> (kernel "main" output), same pitch as occ of that level
    uint8_t *result = nullptr; int result_pitch = 0;
    // staging for the host path: two slots so that the H2D copy of frame i+1 overlaps the kernels and the
    // D2H copy of frame i (meao_render_host_async)
    float *depth_stage[2] = {nullptr, nullptr};     // device, W*H each
    uint8_t *ao_stage[2] = {nullptr, nullptr};      // device, W*H each
    cudaStream_t slot_stream[2] = {nullptr, nullptr};
    cudaEvent_t slot_done[2] = {nullptr, nullptr};
    cudaEvent_t compute_done = nullptr;
    bool compute_done_valid = false;

    bool tma_ok = false;
    CUtensorMap map_low_ren[kRenderTileVariants][5];    // LowDepth<k> with the render box of tile height kRenderTileHs[t]
    CUtensorMap map_low_ups[5];             // LowDepth<k> with the upsample depth box
    CUtensorMap map_ao_ups[5];              // lo AO of upsample lo level k (Occlusion4 / Combined k)
    CUtensorMap map_low_wide[kRenderTileVariants][5];   // LowDepth<k> with the wide-render box
    CUtensorMap map_hq_ups[5];              // HighQuality<k> as LoResAO2 of upsample lo level k
    CUtensorMap map_occ1_ups;               // Occlusion1 as LoResAO1 of the final upsample (MeaoVariants.single_scale)

    // native neighbour exchange (meao_band_export / _connect / _step)
    BandFlags *band_flags = nullptr;        // first 256 bytes of the arena
    uint32_t *tile_ctr = nullptr;           // 2 words per upsample level: tile cursor + finished-CTA count of the persistent blur_upsample grid (zero between launches)
    void *peer_base[2] = {nullptr, nullptr};    // the neighbours' arenas through a peer mapping (same layout as ours)
    bool peer_ipc[2] = {false, false};      // mapping came from cudaIpcOpenMemHandle (must be closed)
    unsigned long long band_timeout_ns = 2000000000ull;
    uint32_t *host_error = nullptr;         // pinned + mapped: the exchange kernel mirrors its sticky error here (read by meao_band_step without a CUDA call)
    uint32_t *host_error_dev = nullptr;     // device alias of host_error
    int pdl_level = -1;                     // programmatic dependent launch in the captured graphs: -1 untried, 0 none, 1 plain chains, 2 all same-stream edges

    // row ranges (per level) for this band
    Range need_c[5];                        // rows of Occlusion<k>/Combined<k> to produce (k=1..4); [0] = final rows
    Range need_low[5];                      // rows of LowDepth<k> required
    Range own_low[5];                       // rows of LowDepth<k> this band produces

    int64_t launches = 0;
    BatchArena batch;

    // CUDA graph cache: one instantiated graph per (depth, out, kind), LRU; when it is full the least recently used
    // executable graph is RE-TARGETED in place with cudaGraphExecUpdate (same topology, new pointers: no device
    // synchronisation, launches already enqueued are unaffected).  Dropped as a whole only when the plan changes.
    struct GraphKey { const void *p[4]; int kind; bool operator<(const GraphKey &o) const {
        for (int i = 0; i < 4; i++) if (p[i] != o.p[i]) return p[i] < o.p[i];
        return kind < o.kind; } };
    struct GraphEntry { cudaGraphExec_t exec; uint64_t last_use; };
    std::map<GraphKey, GraphEntry> graphs;
    std::vector<cudaGraphExec_t> retired;   // executable graphs replaced while possibly in flight: destroyed at the next drop_graph
    uint64_t graph_clock = 0;
    bool graphs_stale = false;              // set by the device-less getters: dropped by the next ensure_ready (on the right device)
    void *last_out = nullptr;               // where the last final upsample wrote (nullptr: c->result)
    int last_kind = MEAO_DEPTH_RAW_F32;     // ingest kind of the last downsample (selects the atlas padding value)

    std::vector<std::pair<std::string, float>> last_profile;
    int profile_repeats = 1;                // launches per kernel inside one event pair of meao_profile_frame
};

namespace {

int fail(MeaoCtx *c, int code, const char *fmt, ...)
{
    char buf[512];
    va_list ap; va_start(ap, fmt); vsnprintf(buf, sizeof buf, fmt, ap); va_end(ap);
    if (c) c->error = buf; else g_create_error = buf;
    return code;
}
#define CUDA_TRY(c, expr) do { cudaError_t e__ = (expr); if (e__ != cudaSuccess) \
    return fail((c), MEAO_ERR_CUDA, "%s failed: %s (%s:%d)", #expr, cudaGetErrorString(e__), __FILE__, __LINE__); } while (0)

// Mathf.Sqrt / Mathf.Pow are (float)Math.X((double)...) in Unity
float mathf_sqrt(float f) { return (float)std::sqrt((double)f); }
float mathf_pow(float f, float p) { return (float)std::pow((double)f, (double)p); }

float host_f16_round(float x) { return __half2float(__float2half_rn(x)); }

// AO.cs:577-590
void sample_thickness(float t[12])
{
    t[0] = mathf_sqrt(1 - 0.2f * 0.2f);                 t[1] = mathf_sqrt(1 - 0.4f * 0.4f);
    t[2] = mathf_sqrt(1 - 0.6f * 0.6f);                 t[3] = mathf_sqrt(1 - 0.8f * 0.8f);
    t[4] = mathf_sqrt(1 - 0.2f * 0.2f - 0.2f * 0.2f);   t[5] = mathf_sqrt(1 - 0.2f * 0.2f - 0.4f * 0.4f);
    t[6] = mathf_sqrt(1 - 0.2f * 0.2f - 0.6f * 0.6f);   t[7] = mathf_sqrt(1 - 0.2f * 0.2f - 0.8f * 0.8f);
    t[8] = mathf_sqrt(1 - 0.4f * 0.4f - 0.4f * 0.4f);   t[9] = mathf_sqrt(1 - 0.4f * 0.4f - 0.6f * 0.6f);
    t[10] = mathf_sqrt(1 - 0.4f * 0.4f - 0.8f * 0.8f);  t[11] = mathf_sqrt(1 - 0.6f * 0.6f - 0.6f * 0.6f);
}

// Rebuild the per-dispatch constants (the CPU half of RebuildCommandBuffers, AO.cs:496-540).
void build_plan(MeaoCtx *c)
{
    Plan &p = c->plan;
    // AO.cs:561-568
    const float fpn = c->camera.far_clip / c->camera.near_clip;
    if (c->camera.reversed_z) { p.zb[0] = fpn - 1; p.zb[1] = 1; } else { p.zb[0] = 1 - fpn; p.zb[1] = fpn; }
    p.zb[2] = p.zb[3] = 0;

    float thick[12];
    sample_thickness(thick);
    for (int k = 1; k <= 4; k++) {
        const int src_w = c->lw[k + 2], src_h = c->lh[k + 2];
        const float ScreenspaceDiameter = 10;                                                        // AO.cs:669
        float ThicknessMultiplier = 2 * c->camera.tan_half_fov_h * ScreenspaceDiameter / src_w;     // AO.cs:678
        if (c->variants.single_pass_stereo) ThicknessMultiplier *= 2;                                // AO.cs:680
        float InverseRangeFactor = 1 / ThicknessMultiplier;                                          // AO.cs:683
        for (int i = 0; i < 12; i++) p.inv_thickness[k][i] = InverseRangeFactor / thick[i];          // AO.cs:687-688
        {   // the same recorder fed a non-tiled source (LowDepth<k>): kernel "main"
            float tm = 2 * c->camera.tan_half_fov_h * ScreenspaceDiameter / c->lw[k];               // AO.cs:678
            tm *= 2;                                                                                 // AO.cs:679 (!source.isTiled)
            if (c->variants.single_pass_stereo) tm *= 2;                                             // AO.cs:680
            const float irf = 1 / tm;                                                                // AO.cs:683
            for (int i = 0; i < 12; i++) p.inv_thickness_wide[k][i] = irf / thick[i];
            p.inv_slice_dim_wide[k][0] = 1.0f / c->lw[k]; p.inv_slice_dim_wide[k][1] = 1.0f / c->lh[k];
        }
        static const float mult[12] = {4, 4, 4, 4, 4, 8, 8, 8, 4, 8, 8, 4};                          // AO.cs:696-707
        float *w = p.sample_weight[k];
        for (int i = 0; i < 12; i++) w[i] = mult[i] * thick[i];
        if (!c->variants.sample_exhaustively) { w[0] = 0; w[2] = 0; w[5] = 0; w[7] = 0; w[9] = 0; }  // AO.cs:709-715
        float total = 0.0f;
        for (int i = 0; i < 12; i++) total += w[i];                                                  // AO.cs:718-721
        for (int i = 0; i < 12; i++) w[i] /= total;                                                  // AO.cs:723-724
        p.inv_slice_dim[k][0] = 1.0f / src_w; p.inv_slice_dim[k][1] = 1.0f / src_h;                  // AO.cs:732
        // value of the atlas padding texels (SURVEY.md P3): Downsample1 writes Linearize(OOB load = 0),
        // Downsample2 writes 0 (its OOB load of DS4x)
        float pad = 0.0f;
        if (k <= 2) {
            // raw depth 0 through Linearize (DS1:40-45); linear ingest: 0
            pad = c->camera.reversed_z ? 1e5f : 1.0f / std::fmaf(p.zb[0], 0.0f, p.zb[1]);
        }
        p.pad[k] = pad;   // the depth-kind dependent part (linear ingest -> 0) is applied at launch
    }
    p.reject_fadeoff = -1 / c->params.thickness_modifier;                                            // AO.cs:733
    p.intensity = c->params.intensity;                                                               // AO.cs:734

    for (int lo = 1; lo <= 4; lo++) {
        const int lo_w = c->lw[lo], lo_h = c->lh[lo], hi_w = c->lw[lo - 1], hi_h = c->lh[lo - 1];
        float stepSize = 1920.0f / lo_w;                                                             // AO.cs:760
        float blurTolerance = 1 - mathf_pow(10, c->params.blur_tolerance) * stepSize;                // AO.cs:761
        blurTolerance *= blurTolerance;                                                              // AO.cs:762
        float upsampleTolerance = mathf_pow(10, c->params.upsample_tolerance);                       // AO.cs:763
        float noiseFilterWeight = 1 / (mathf_pow(10, c->params.noise_filter_tolerance) + upsampleTolerance);   // AO.cs:764
        p.inv_low[lo][0] = 1.0f / lo_w; p.inv_low[lo][1] = 1.0f / lo_h;                              // AO.cs:766
        p.inv_high[lo][0] = 1.0f / hi_w; p.inv_high[lo][1] = 1.0f / hi_h;                            // AO.cs:767
        p.noise_filter_strength[lo] = noiseFilterWeight;
        p.step_size[lo] = stepSize;
        p.blur_tolerance[lo] = blurTolerance;
        p.upsample_tolerance[lo] = upsampleTolerance;
    }
    c->plan_dirty = false;
}

// Caller must have made c->device current (ensure_ready / meao_resize / meao_destroy do).
void drop_graph(MeaoCtx *c)
{
    c->graphs_stale = false;
    if (c->graphs.empty() && c->retired.empty()) return;
    cudaDeviceSynchronize();            // a re-plan is rare; never destroy an executable graph that may still be in flight
    for (auto &kv : c->graphs) cudaGraphExecDestroy(kv.second.exec);
    for (auto ge : c->retired) cudaGraphExecDestroy(ge);
    c->graphs.clear();
    c->retired.clear();
}

void disconnect_peers(MeaoCtx *c)
{
    for (int side = 0; side < 2; side++) {
        if (c->peer_base[side] && c->peer_ipc[side]) cudaIpcCloseMemHandle(c->peer_base[side]);
        c->peer_base[side] = nullptr; c->peer_ipc[side] = false;
    }
}

void free_batch(MeaoCtx *c)
{
    if (c->batch.base) cudaFree(c->batch.base);
    c->batch = BatchArena{};
}

void free_buffers(MeaoCtx *c)
{
    drop_graph(c);
    free_batch(c);
    disconnect_peers(c);
    c->band_flags = nullptr;
    if (c->arena) cudaFree(c->arena);
    c->arena = nullptr; c->arena_bytes = 0;
    c->depth_stage[0] = c->depth_stage[1] = nullptr; c->ao_stage[0] = c->ao_stage[1] = nullptr;
    c->compute_done_valid = false;
}

int make_map(MeaoCtx *c, CUtensorMap *m, CUtensorMapDataType dt, int elem, void *base, int w, int h, int pitch_elems, int bw, int bh)
{
    cuuint64_t dims[2] = {(cuuint64_t)w, (cuuint64_t)h};
    cuuint64_t strides[1] = {(cuuint64_t)pitch_elems * elem};
    cuuint32_t box[2] = {(cuuint32_t)bw, (cuuint32_t)bh};
    cuuint32_t estr[2] = {1, 1};
    CUresult r = c->encode(m, dt, 2, base, dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                           CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    return r == CUDA_SUCCESS ? 0 : -1;
}

int make_map3(MeaoCtx *c, CUtensorMap *m, CUtensorMapDataType dt, int elem, void *base, int w, int h, int pitch_elems, int frames,
              size_t slot_bytes, int bw, int bh)
{
    cuuint64_t dims[3] = {(cuuint64_t)w, (cuuint64_t)h, (cuuint64_t)frames};
    cuuint64_t strides[2] = {(cuuint64_t)pitch_elems * elem, (cuuint64_t)slot_bytes};
    cuuint32_t box[3] = {(cuuint32_t)bw, (cuuint32_t)bh, 1};
    cuuint32_t estr[3] = {1, 1, 1};
    CUresult r = c->encode(m, dt, 3, base, dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                           CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    return r == CUDA_SUCCESS ? 0 : -1;
}

// rows of the low level (after clamping) that an upsample producing hi rows [a,b) reads
Range ups_lo_rows(Range hi, int loh)
{
    if (hi.hi <= hi.lo) return Range{0, 0};
    const int ymin = (hi.lo + 1) >> 1, ymax = hi.hi >> 1;      // Y = (py+1)>>1 for py in [a, b-1]
    return clampr(Range{ymin - 3, ymax + 3}, loh);             // quad rows Y-1..Y, blur radius 2
}
// rows of LowDepth<k> that a render producing rows [a,b) of level k reads (slice texel +-4 => +-16 rows, slice aligned)
Range ren_low_rows(Range out, int lh)
{
    if (out.hi <= out.lo) return Range{0, 0};
    return clampr(Range{4 * ((out.lo >> 2) - 4), 4 * (((out.hi - 1) >> 2) + 4) + 4}, lh);
}

struct BandNeeds { Range need_c[5]; Range need_low[5]; Range own_low[5]; };

BandNeeds compute_needs(const MeaoCtx *c, int b0, int b1)
{
    BandNeeds n;
    n.need_c[0] = Range{b0, b1};
    for (int k = 1; k <= 4; k++) n.need_c[k] = ups_lo_rows(n.need_c[k - 1], c->lh[k]);
    for (int k = 1; k <= 4; k++) {
        Range r = ren_low_rows(n.need_c[k], c->lh[k]);
        // the upsample also reads LowDepth<k> on need_c[k] (as lo depth) -- a subset of r
        if (n.need_c[k].lo < r.lo) r.lo = n.need_c[k].lo;
        if (n.need_c[k].hi > r.hi) r.hi = n.need_c[k].hi;
        n.need_low[k] = r;
        n.own_low[k] = Range{b0 >> k, (b1 + (1 << k) - 1) >> k};
    }
    n.need_low[0] = n.own_low[0] = Range{b0, b1};
    return n;
}

int setup_band(MeaoCtx *c)
{
    BandNeeds n = compute_needs(c, c->band0, c->band1);
    for (int k = 0; k <= 4; k++) { c->need_c[k] = n.need_c[k]; c->need_low[k] = n.need_low[k]; c->own_low[k] = n.own_low[k]; }
    for (int k = 1; k <= 4; k++) {
        if (c->need_low[k].lo < c->own_low[k].lo) {
            if (c->prev0 < 0 || c->need_low[k].lo < (c->prev0 >> k))
                return fail(c, MEAO_ERR_UNSUPPORTED, "halo of level %d reaches beyond the band above", k);
        }
        if (c->need_low[k].hi > c->own_low[k].hi) {
            if (c->next1 < 0 || c->need_low[k].hi > ((c->next1 + (1 << k) - 1) >> k))
                return fail(c, MEAO_ERR_UNSUPPORTED, "halo of level %d reaches beyond the band below", k);
        }
    }
    return 0;
}

int allocate(MeaoCtx *c)
{
    const int W = c->W, H = c->H;
    for (int l = 0; l < 7; l++) {                         // AO.cs:276-281
        const int div = 1 << l;
        c->lw[l] = (W + div - 1) / div;
        c->lh[l] = (H + div - 1) / div;
    }
    c->band0 = 0; c->band1 = H; c->prev0 = -1; c->next1 = -1;
    c->plan_dirty = true;
    if (c->plan_only) return setup_band(c);
    free_buffers(c);
    // pitches: rows start on 128-byte boundaries
    c->lin_pitch = align_up(c->lw[0], 64);
    c->result_pitch = align_up(c->lw[0], 128);
    size_t off = 0;
    auto take = [&](size_t bytes) { size_t o = off; off += (bytes + 255) / 256 * 256; return o; };
    take(sizeof(BandFlags));            // offset 0 in EVERY context's arena (the neighbours address it through their peer mapping)
    const size_t o_ctr = take(8 * sizeof(uint32_t));
    size_t o_lin = take((size_t)c->lin_pitch * c->lh[0] * sizeof(__half));
    size_t o_res = take((size_t)c->result_pitch * c->lh[0]);
    size_t o_low[5], o_occ[5], o_comb[4], o_hq[5];
    for (int k = 1; k <= 4; k++) {
        c->low_pitch[k] = align_up(c->lw[k], 32);
        c->occ_pitch[k] = align_up(c->lw[k], 128);
        o_low[k] = take((size_t)c->low_pitch[k] * c->lh[k] * sizeof(float));
        o_occ[k] = take((size_t)c->occ_pitch[k] * c->lh[k]);
        if (k <= 3) o_comb[k] = take((size_t)c->occ_pitch[k] * c->lh[k]);
        o_hq[k] = take((size_t)c->occ_pitch[k] * c->lh[k]);
    }
    size_t o_dst[2], o_ast[2];
    for (int i = 0; i < 2; i++) { o_dst[i] = take((size_t)W * H * sizeof(float)); o_ast[i] = take((size_t)W * H); }
    cudaError_t e = cudaMalloc(&c->arena, off);
    if (e != cudaSuccess) return fail(c, e == cudaErrorMemoryAllocation ? MEAO_ERR_NOMEM : MEAO_ERR_CUDA,
                                      "cudaMalloc(%zu) failed: %s", off, cudaGetErrorString(e));
    c->arena_bytes = off;
    CUDA_TRY(c, cudaMemsetAsync(c->arena, 0, off, c->stream));
    CUDA_TRY(c, cudaStreamSynchronize(c->stream));
    char *b = (char *)c->arena;
    c->band_flags = (BandFlags *)b;
    c->tile_ctr = (uint32_t *)(b + o_ctr);          // zeroed by the memset above
    {
        BandFlags init{}; init.epoch = 1;
        CUDA_TRY(c, cudaMemcpy(c->band_flags, &init, sizeof init, cudaMemcpyHostToDevice));
        if (c->host_error) *c->host_error = 0;
    }
    c->lin = (__half *)(b + o_lin);
    c->result = (uint8_t *)(b + o_res);
    for (int k = 1; k <= 4; k++) {
        c->low[k] = (float *)(b + o_low[k]);
        c->occ[k] = (uint8_t *)(b + o_occ[k]);
        if (k <= 3) c->comb[k] = (uint8_t *)(b + o_comb[k]);
        c->hq[k] = (uint8_t *)(b + o_hq[k]);
    }
    for (int i = 0; i < 2; i++) { c->depth_stage[i] = (float *)(b + o_dst[i]); c->ao_stage[i] = (uint8_t *)(b + o_ast[i]); }

    c->tma_ok = false;
    if (c->encode) {
        bool ok = true;
        for (int k = 1; k <= 4 && ok; k++) {
            for (int t = 0; t < kRenderTileVariants; t++) {
                ok &= make_map(c, &c->map_low_ren[t][k], CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 4, c->low[k], c->lw[k], c->lh[k], c->low_pitch[k], kRenderBoxW, render_box_h(kRenderTileHs[t], false)) == 0;
                ok &= make_map(c, &c->map_low_wide[t][k], CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 4, c->low[k], c->lw[k], c->lh[k], c->low_pitch[k], kRenderWideBoxW, render_box_h(kRenderTileHs[t], true)) == 0;
            }
            ok &= make_map(c, &c->map_low_ups[k], CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 4, c->low[k], c->lw[k], c->lh[k], c->low_pitch[k], kUpsDepthBoxW, kUpsDepthBoxH) == 0;
            uint8_t *ao = (k == 4) ? c->occ[4] : c->comb[k];
            ok &= make_map(c, &c->map_ao_ups[k], CU_TENSOR_MAP_DATA_TYPE_UINT8, 1, ao, c->lw[k], c->lh[k], c->occ_pitch[k], kUpsAoBoxW, kUpsAoBoxH) == 0;
            ok &= make_map(c, &c->map_hq_ups[k], CU_TENSOR_MAP_DATA_TYPE_UINT8, 1, c->hq[k], c->lw[k], c->lh[k], c->occ_pitch[k], kUpsAoBoxW, kUpsAoBoxH) == 0;
        }
        ok &= make_map(c, &c->map_occ1_ups, CU_TENSOR_MAP_DATA_TYPE_UINT8, 1, c->occ[1], c->lw[1], c->lh[1], c->occ_pitch[1], kUpsAoBoxW, kUpsAoBoxH) == 0;
        c->tma_ok = ok;
    }
    if (!c->tma_ok) {
        memset(&c->map_occ1_ups, 0, sizeof c->map_occ1_ups);
        memset(c->map_low_ren, 0, sizeof c->map_low_ren);
        memset(c->map_low_ups, 0, sizeof c->map_low_ups);
        memset(c->map_ao_ups, 0, sizeof c->map_ao_ups);
        memset(c->map_low_wide, 0, sizeof c->map_low_wide);
        memset(c->map_hq_ups, 0, sizeof c->map_hq_ups);
    }
    return setup_band(c);
}

int ensure_ready(MeaoCtx *c)
{
    if (!c) return MEAO_ERR_INVALID;
    if (c->W <= 0) return fail(c, MEAO_ERR_INVALID, "meao_resize has not been called");
    if (c->plan_only) return fail(c, MEAO_ERR_CUDA, "plan-only context (device < 0): no CUDA device bound, and libmeao has no CPU fallback");
    CUDA_TRY(c, cudaSetDevice(c->device));
    if (c->plan_dirty) { build_plan(c); c->graphs_stale = true; }
    if (c->graphs_stale) drop_graph(c);
    return 0;
}

// Grows the batch arena to >= frames slots.  Synchronous (device synchronise, cudaFree, cudaMalloc): callers keep it out of
// timed regions with meao_reserve_batch.  The captured batch graphs point into the old arena and are dropped with it.
int reserve_batch(MeaoCtx *c, int frames)
{
    BatchArena &b = c->batch;
    if (frames <= b.capacity) return 0;
    CUDA_TRY(c, cudaDeviceSynchronize());
    for (auto it = c->graphs.begin(); it != c->graphs.end();) {
        if (it->first.kind >= 400) { cudaGraphExecDestroy(it->second.exec); it = c->graphs.erase(it); } else ++it;
    }
    free_batch(c);
    size_t off = 0;
    auto take = [&](size_t bytes) { size_t o = off; off += (bytes + 255) / 256 * 256; return o; };
    const size_t o_lin = take((size_t)c->lin_pitch * c->lh[0] * sizeof(__half));
    size_t o_low[5], o_occ[5], o_comb[4], o_hq[5];
    for (int k = 1; k <= 4; k++) {
        o_low[k] = take((size_t)c->low_pitch[k] * c->lh[k] * sizeof(float));
        o_occ[k] = take((size_t)c->occ_pitch[k] * c->lh[k]);
        if (k <= 3) o_comb[k] = take((size_t)c->occ_pitch[k] * c->lh[k]);
        o_hq[k] = take((size_t)c->occ_pitch[k] * c->lh[k]);
    }
    const size_t slot = off;                        // a multiple of 256 bytes
    const size_t head = 256;                        // persistent-loop tile counters
    const size_t total = head + slot * (size_t)frames;
    cudaError_t e = cudaMalloc(&b.base, total);
    if (e != cudaSuccess) {
        b.base = nullptr; cudaGetLastError();
        return fail(c, e == cudaErrorMemoryAllocation ? MEAO_ERR_NOMEM : MEAO_ERR_CUDA, "batch arena cudaMalloc(%zu) failed: %s", total, cudaGetErrorString(e));
    }
    CUDA_TRY(c, cudaMemset(b.base, 0, head));
    b.bytes = total; b.slot_bytes = slot; b.capacity = frames;
    char *p = (char *)b.base;
    b.tile_ctr = (uint32_t *)p;
    p += head;
    b.lin = (__half *)(p + o_lin);
    for (int k = 1; k <= 4; k++) {
        b.low[k] = (float *)(p + o_low[k]);
        b.occ[k] = (uint8_t *)(p + o_occ[k]);
        if (k <= 3) b.comb[k] = (uint8_t *)(p + o_comb[k]);
        b.hq[k] = (uint8_t *)(p + o_hq[k]);
    }
    b.tma_ok = false;
    if (c->encode) {
        bool ok = true;
        for (int k = 1; k <= 4 && ok; k++) {
            for (int t = 0; t < kRenderTileVariants; t++) {
                ok &= make_map3(c, &b.map_low_ren[t][k], CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 4, b.low[k], c->lw[k], c->lh[k], c->low_pitch[k], frames, slot, kRenderBoxW, render_box_h(kRenderTileHs[t], false)) == 0;
                ok &= make_map3(c, &b.map_low_wide[t][k], CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 4, b.low[k], c->lw[k], c->lh[k], c->low_pitch[k], frames, slot, kRenderWideBoxW, render_box_h(kRenderTileHs[t], true)) == 0;
            }
            ok &= make_map3(c, &b.map_low_ups[k], CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 4, b.low[k], c->lw[k], c->lh[k], c->low_pitch[k], frames, slot, kUpsDepthBoxW, kUpsDepthBoxH) == 0;
            uint8_t *ao = (k == 4) ? b.occ[4] : b.comb[k];
            ok &= make_map3(c, &b.map_ao_ups[k], CU_TENSOR_MAP_DATA_TYPE_UINT8, 1, ao, c->lw[k], c->lh[k], c->occ_pitch[k], frames, slot, kUpsAoBoxW, kUpsAoBoxH) == 0;
            ok &= make_map3(c, &b.map_hq_ups[k], CU_TENSOR_MAP_DATA_TYPE_UINT8, 1, b.hq[k], c->lw[k], c->lh[k], c->occ_pitch[k], frames, slot, kUpsAoBoxW, kUpsAoBoxH) == 0;
        }
        ok &= make_map3(c, &b.map_occ1_ups, CU_TENSOR_MAP_DATA_TYPE_UINT8, 1, b.occ[1], c->lw[1], c->lh[1], c->occ_pitch[1], frames, slot, kUpsAoBoxW, kUpsAoBoxH) == 0;
        b.tma_ok = ok;
    }
    return 0;
}

struct NvtxRange { explicit NvtxRange(const char *n) { nvtxRangePushA(n); } ~NvtxRange() { nvtxRangePop(); } };

// Tile-height variant (index into kRenderTileHs = {32, 16, 8}) of a render launch.  The big levels keep the 64 x 32 tile
// (least apron overhead: throughput); a level whose grid would not even put one CTA on every SM is latency-bound -- one
// CTA's serial time IS the kernel time -- so it takes the tallest tile that still gives >= 148 CTAs, else 64 x 8.
// (Measured at 4K: level 2, 255 CTAs of 64 x 32, is FASTER with the big tile -- 14.0 vs 15.7 us -- levels 3 / 4 gain ~0.5 us.)
int render_tile_variant(const MeaoCtx *c, int k, int rows, int frames = 1)
{
    const char *force = getenv("MEAO_REN_TILE");               // tuning aid: 0 / 1 / 2 forces a variant for every level
    if (force && force[0] >= '0' && force[0] < '0' + kRenderTileVariants) return force[0] - '0';
    for (int t = 0; t < kRenderTileVariants; t++) {
        const long long ctas = (long long)((c->lw[k] + 63) / 64) * ((rows + kRenderTileHs[t] - 1) / kRenderTileHs[t]) * frames;   // a batch: all its frames
        if (ctas >= 148) return t;
    }
    return kRenderTileVariants - 1;
}

// ---- the three recorders ---------------------------------------------------------------------

// PushDownsampleCommands, AO.cs:604-658
int record_downsample(MeaoCtx *c, const void *depth, int kind, cudaStream_t s, const BatchRun *batch = nullptr)
{
    if (kind < MEAO_DEPTH_RAW_F32 || kind > MEAO_DEPTH_RAW_D24S8) return fail(c, MEAO_ERR_INVALID, "bad depth kind %d", kind);
    NvtxRange nv("meao::prepare_depth");
    PrepareArgs a{};
    a.depth = depth;
    a.in_format = (kind == MEAO_DEPTH_RAW_D16_UNORM) ? 1 : (kind == MEAO_DEPTH_RAW_D24S8 ? 2 : 0);
    a.W = c->W; a.H = c->H;
    a.depth_row0 = c->band0;
    a.row0 = c->band0; a.row1 = c->band1;
    a.lin = c->lin; a.lin_pitch = c->lin_pitch;
    for (int k = 1; k <= 4; k++) { a.low[k - 1] = c->low[k]; a.low_pitch[k - 1] = c->low_pitch[k]; }
    a.zbx = c->plan.zb[0]; a.zby = c->plan.zb[1];
    a.raw = (kind != MEAO_DEPTH_LINEAR_F32);
    a.reversed_z = c->camera.reversed_z;
    a.vec_ok = (((uintptr_t)depth & 15) == 0) && (c->W % (a.in_format == 1 ? 8 : 4) == 0);
    if (batch) {
        const BatchArena &b = c->batch;
        a.lin = b.lin;
        for (int k = 1; k <= 4; k++) a.low[k - 1] = b.low[k];
        a.vec_ok = a.vec_ok && (batch->in_frame_bytes % 16 == 0);     // every frame's base stays 16-byte aligned
        c->batch.last_kind = kind;
        CUDA_TRY(c, launch_prepare_depth_batch(PrepareBatchArgs{a, batch->in_frame_bytes, (long long)b.slot_bytes}, batch->frames, s));
        c->launches++;
        return 0;
    }
    c->last_kind = kind;
    CUDA_TRY(c, launch_prepare_depth(a, s));
    c->launches++;
    return 0;
}

// PushRenderCommands, AO.cs:660-748.  wide = false: the call AmbientOcclusion.cs makes (tiled source, kernel main_interleaved);
// wide = true: the same recorder for the non-tiled source LowDepth<k> (kernel main) -> HighQuality<k>.
int record_render(MeaoCtx *c, int k, int kind, cudaStream_t s, bool wide = false, const BatchRun *batch = nullptr)
{
    static const int idx_checker[7] = {1, 3, 4, 8, 11, 6, 10};                       // Render.compute:162-168 table slots, call order
    static const int idx_exh[12] = {0, 1, 2, 3, 4, 8, 11, 5, 6, 7, 9, 10};           // Render.compute:148-159
    const bool exh = c->variants.sample_exhaustively != 0;
    const int n = exh ? 12 : 7;
    const int *idx = exh ? idx_exh : idx_checker;
    NvtxRange nv(wide ? "meao::render_ao_wide" : "meao::render_ao");
    RenderArgs a{};
    a.low = c->low[k]; a.lw = c->lw[k]; a.lh = c->lh[k]; a.lpitch = c->low_pitch[k];
    a.occ = wide ? c->hq[k] : c->occ[k]; a.opitch = c->occ_pitch[k];
    a.sw = c->lw[k + 2]; a.sh = c->lh[k + 2];
    a.pad = host_f16_round((kind != MEAO_DEPTH_LINEAR_F32) ? c->plan.pad[k] : 0.0f);
    const float *it = wide ? c->plan.inv_thickness_wide[k] : c->plan.inv_thickness[k];
    for (int i = 0; i < n; i++) {
        a.inv_thickness[i] = it[idx[i]];
        a.neg_front[i] = -(a.inv_thickness[i] - 0.5f);                                               // Render.compute:85
        a.weight[i] = c->plan.sample_weight[k][idx[i]];
    }
    a.reject_fadeoff = c->plan.reject_fadeoff;
    a.intensity = c->plan.intensity;
    a.row0 = c->need_c[k].lo; a.row1 = c->need_c[k].hi;
    a.wide = wide ? 1 : 0;
    a.exhaustive = exh ? 1 : 0;
    const int tv = render_tile_variant(c, k, a.row1 - (a.row0 & ~3), batch ? batch->frames : 1);
    a.tile_h = kRenderTileHs[tv];
    if (batch) {
        const BatchArena &b = c->batch;
        a.low = b.low[k]; a.occ = wide ? b.hq[k] : b.occ[k];
        CUDA_TRY(c, launch_render_ao_batch(wide ? b.map_low_wide[tv][k] : b.map_low_ren[tv][k], b.tma_ok, RenderBatchArgs{a, (long long)b.slot_bytes}, batch->frames, s));
        c->launches++;
        return 0;
    }
    CUDA_TRY(c, launch_render_ao(wide ? c->map_low_wide[tv][k] : c->map_low_ren[tv][k], c->tma_ok, a, s));
    c->launches++;
    return 0;
}
inline bool hq_level(const MeaoCtx *c, int k) { return ((c->variants.high_quality_mask >> (k - 1)) & 1) != 0; }

// PushUpsampleCommands with the wiring of AO.cs:528-531
int record_upsample(MeaoCtx *c, int lo, void *ao_out, cudaStream_t s, const BatchRun *batch = nullptr)
{
    const int hi = lo - 1;
    NvtxRange nv("meao::blur_upsample");
    const bool single = c->variants.single_scale != 0 && lo == 1;      // LoResAO1 = Occlusion1: no coarser level contributes
    UpsampleArgs a{};
    a.lo_depth = c->low[lo]; a.low = c->lw[lo]; a.loh = c->lh[lo]; a.lo_dpitch = c->low_pitch[lo];
    a.lo_ao = single ? c->occ[1] : (lo == 4) ? c->occ[4] : c->comb[lo]; a.lo_apitch = c->occ_pitch[lo];
    if (hi == 0) { a.hi_depth = c->lin; a.hi_is_half = 1; a.hi_dpitch = c->lin_pitch; a.hi_ao = nullptr; a.hi_apitch = 0; }
    else { a.hi_depth = c->low[hi]; a.hi_is_half = 0; a.hi_dpitch = c->low_pitch[hi]; a.hi_ao = c->occ[hi]; a.hi_apitch = c->occ_pitch[hi]; }
    if (hi == 0) {
        if (ao_out) { a.out = (uint8_t *)ao_out; a.out_pitch = c->W; a.out_row_origin = c->band0; }
        else { a.out = c->result; a.out_pitch = c->result_pitch; a.out_row_origin = 0; }
        if (!batch) c->last_out = ao_out;
    } else { a.out = c->comb[hi]; a.out_pitch = c->occ_pitch[hi]; a.out_row_origin = 0; }
    a.out_vec_ok = (((uintptr_t)a.out & 7) == 0) && (a.out_pitch % 8 == 0);
    a.hiw = c->lw[hi]; a.hih = c->lh[hi];
    a.noise_filter_strength = c->plan.noise_filter_strength[lo];
    a.step_size = c->plan.step_size[lo];
    a.blur_tolerance = c->plan.blur_tolerance[lo];
    a.upsample_tolerance = c->plan.upsample_tolerance[lo];
    {
        auto safe = [](float x) { return x >= 8.673617379884035e-19f && x < 1152921504606846976.0f; };
        a.fast_div_ok = safe(a.upsample_tolerance) && safe(a.noise_filter_strength);
#if MEAO_UPS_STATIC_GUARD || MEAO_UPS_V2
        // 2^-55, 2^-52, 2^59: with these bounds total / num of the final division are provably inside the fast-division range
        a.fast_div_ok = a.fast_div_ok && a.upsample_tolerance >= 2.7755575615628914e-17f &&
                        a.noise_filter_strength >= 2.220446049250313e-16f && a.noise_filter_strength < 288230376151711744.0f;
#endif
    }
    a.row0 = c->need_c[hi].lo; a.row1 = c->need_c[hi].hi;
    a.tile_ctr = c->tile_ctr + 2 * (lo - 1);
    const uint8_t *lo_ao2 = hq_level(c, lo) ? c->hq[lo] : nullptr;                   // kernels main_premin / main_premin_blendout
    if (batch) {
        const BatchArena &b = c->batch;
        a.lo_depth = b.low[lo];
        a.lo_ao = single ? b.occ[1] : (lo == 4) ? b.occ[4] : b.comb[lo];
        if (hi == 0) a.hi_depth = b.lin;
        else { a.hi_depth = b.low[hi]; a.hi_ao = b.occ[hi]; }
        long long out_frame_bytes = (long long)b.slot_bytes;
        if (hi == 0) { a.out = (uint8_t *)ao_out; a.out_pitch = c->W; a.out_row_origin = 0; out_frame_bytes = (long long)c->W * c->H; }
        else a.out = b.comb[hi];
        a.out_vec_ok = (((uintptr_t)a.out & 7) == 0) && (a.out_pitch % 8 == 0) && (out_frame_bytes % 8 == 0);
        a.tile_ctr = b.tile_ctr + 2 * (lo - 1);
        UpsampleBatchArgs ba{UpsamplePreminArgs{a, hq_level(c, lo) ? b.hq[lo] : nullptr, c->occ_pitch[lo]}, (long long)b.slot_bytes, out_frame_bytes, batch->frames, 0};
        CUDA_TRY(c, launch_blur_upsample_batch(b.map_low_ups[lo], single ? b.map_occ1_ups : b.map_ao_ups[lo], &b.map_hq_ups[lo], b.tma_ok, ba, s));
        c->launches++;
        return 0;
    }
    CUDA_TRY(c, launch_blur_upsample(c->map_low_ups[lo], single ? c->map_occ1_ups : c->map_ao_ups[lo], &c->map_hq_ups[lo], c->tma_ok, a, lo_ao2, c->occ_pitch[lo], s));
    c->launches++;
    return 0;
}

// RAII: launches issued while one of these is alive (and `on`) carry the programmatic-dependent-launch attribute.
struct PdlScope { bool prev; explicit PdlScope(bool on) : prev(g_launch_pdl) { g_launch_pdl = on; } ~PdlScope() { g_launch_pdl = prev; } };

// The same nine launches as record_frame, recorded as a DAG on forked streams (for graph capture): the four
// render levels are independent (SURVEY.md 3.2), the coarse upsample chain 4->3->2 only needs Occlusion2..4,
// and only the last two upsamples wait for the big level-1 render.
// pdl: 0 = plain edges; 1 = programmatic dependent launch on the kernels whose ONLY predecessor is the kernel before them in
// the same stream; 2 = also on kernels that additionally wait for an event of another branch.  after_exchange: the node
// before this DAG is the neighbour-exchange kernel, which spins on remote flags -- nothing may be scheduled "early" behind it
// (a grid parked in griddepcontrol.wait holds SM resources that the neighbour band's kernels may need: see DESIGN.md 4).
int record_frame_dag(MeaoCtx *c, const void *depth, int kind, void *ao_out, cudaStream_t s, bool do_prepare = true, int pdl = 0,
                     bool after_exchange = false, const BatchRun *batch = nullptr)
{
    int rc;
    if (c->variants.single_scale) {     // BASELINE.json configs[0]: Downsample1 -> Render level 1 -> final-style Upsample on Occlusion1
        if (do_prepare && (rc = record_downsample(c, depth, kind, s, batch))) return rc;
        { PdlScope p(pdl >= 1 && !after_exchange); if ((rc = record_render(c, 1, kind, s, false, batch))) return rc; }
        { PdlScope p(pdl >= 1); if ((rc = record_upsample(c, 1, ao_out, s, batch))) return rc; }
        return 0;
    }
    cudaStream_t b1 = c->branch[0], b2 = c->branch[1], b3 = c->branch[2];
    if (do_prepare && (rc = record_downsample(c, depth, kind, s, batch))) return rc;
    CUDA_TRY(c, cudaEventRecord(c->ev[0], s));
    CUDA_TRY(c, cudaStreamWaitEvent(b1, c->ev[0], 0));
    CUDA_TRY(c, cudaStreamWaitEvent(b2, c->ev[0], 0));
    CUDA_TRY(c, cudaStreamWaitEvent(b3, c->ev[0], 0));
    // the optional high-quality render of a level (kernel "main") rides on the branch of that level's interleaved render
    { PdlScope p(pdl >= 1 && !after_exchange); if ((rc = record_render(c, 1, kind, s, false, batch))) return rc; }
    { PdlScope p(pdl >= 1); if (hq_level(c, 1) && (rc = record_render(c, 1, kind, s, true, batch))) return rc; }
    if ((rc = record_render(c, 2, kind, b1, false, batch))) return rc;
    { PdlScope p(pdl >= 1); if (hq_level(c, 2) && (rc = record_render(c, 2, kind, b1, true, batch))) return rc; }
    CUDA_TRY(c, cudaEventRecord(c->ev[1], b1));
    if ((rc = record_render(c, 3, kind, b2, false, batch))) return rc;
    { PdlScope p(pdl >= 1); if (hq_level(c, 3) && (rc = record_render(c, 3, kind, b2, true, batch))) return rc; }
    CUDA_TRY(c, cudaEventRecord(c->ev[2], b2));
    if ((rc = record_render(c, 4, kind, b3, false, batch))) return rc;
    { PdlScope p(pdl >= 1); if (hq_level(c, 4) && (rc = record_render(c, 4, kind, b3, true, batch))) return rc; }
    CUDA_TRY(c, cudaStreamWaitEvent(b3, c->ev[2], 0));
    { PdlScope p(pdl >= 2); if ((rc = record_upsample(c, 4, nullptr, b3, batch))) return rc; }
    CUDA_TRY(c, cudaStreamWaitEvent(b3, c->ev[1], 0));
    { PdlScope p(pdl >= 2); if ((rc = record_upsample(c, 3, nullptr, b3, batch))) return rc; }
    CUDA_TRY(c, cudaEventRecord(c->ev[3], b3));
    CUDA_TRY(c, cudaStreamWaitEvent(s, c->ev[3], 0));
    { PdlScope p(pdl >= 2); if ((rc = record_upsample(c, 2, nullptr, s, batch))) return rc; }
    { PdlScope p(pdl >= 1); if ((rc = record_upsample(c, 1, ao_out, s, batch))) return rc; }
    return 0;
}

// record order of RebuildCommandBuffers, AO.cs:511-531
int record_frame(MeaoCtx *c, const void *depth, int kind, void *ao_out, cudaStream_t s, bool profile, const BatchRun *batch = nullptr)
{
    static const char *ren_names[5] = {"", "render_ao L1", "render_ao L2", "render_ao L3", "render_ao L4"};
    static const char *hq_names[5] = {"", "render_ao_wide L1", "render_ao_wide L2", "render_ao_wide L3", "render_ao_wide L4"};
    static const char *ups_names[5] = {"", "blur_upsample L1->L0", "blur_upsample L2->L1", "blur_upsample L3->L2", "blur_upsample L4->L3"};
    std::vector<const char *> names;
    std::vector<cudaEvent_t> ev;
    auto mark = [&]() { if (profile) { cudaEvent_t e; cudaEventCreate(&e); cudaEventRecord(e, s); ev.push_back(e); } };
    const int reps = profile ? c->profile_repeats : 1;         // every kernel is idempotent (out of place), so repeating it is harmless
    int rc = 0;
    mark();
    for (int r = 0; r < reps && !rc; r++) rc = record_downsample(c, depth, kind, s, batch);
    if (rc) return rc;
    names.push_back("prepare_depth"); mark();
    const int kmax = c->variants.single_scale ? 1 : 4;       // single-scale: Render level 1 + the final-style Upsample only
    for (int k = 1; k <= kmax; k++) { for (int r = 0; r < reps && !rc; r++) rc = record_render(c, k, kind, s, false, batch); if (rc) return rc; names.push_back(ren_names[k]); mark(); }
    for (int k = 1; k <= kmax; k++) if (hq_level(c, k)) { for (int r = 0; r < reps && !rc; r++) rc = record_render(c, k, kind, s, true, batch); if (rc) return rc; names.push_back(hq_names[k]); mark(); }
    for (int lo = kmax; lo >= 1; lo--) { for (int r = 0; r < reps && !rc; r++) rc = record_upsample(c, lo, lo == 1 ? ao_out : nullptr, s, batch); if (rc) return rc; names.push_back(ups_names[lo]); mark(); }
    if (profile) {
        CUDA_TRY(c, cudaStreamSynchronize(s));
        c->last_profile.clear();
        for (size_t i = 0; i + 1 < ev.size(); i++) {
            float ms = 0; cudaEventElapsedTime(&ms, ev[i], ev[i + 1]);
            c->last_profile.push_back({names[i], ms / (float)reps});
        }
        for (auto e : ev) cudaEventDestroy(e);
    }
    return 0;
}

int buffer_info(const MeaoCtx *c, int id, int *lvl, int *slices, int *elem)
{
    if (id == 1) { *lvl = 0; *slices = 1; *elem = 2; }
    else if (id >= 2 && id <= 5) { *lvl = id - 1; *slices = 1; *elem = 4; }
    else if (id >= 6 && id <= 9) { *lvl = id - 5 + 2; *slices = 16; *elem = 2; }
    else if (id >= 10 && id <= 13) { *lvl = id - 9; *slices = 1; *elem = 1; }
    else if (id >= 14 && id <= 16) { *lvl = id - 13; *slices = 1; *elem = 1; }
    else if (id == 17) { *lvl = 0; *slices = 1; *elem = 1; }
    else if (id >= 18 && id <= 21) { *lvl = id - 17; *slices = 1; *elem = 1; }      // HighQuality1..4 (extension)
    else return -1;
    (void)c;
    return 0;
}

// device pointer + pitch (bytes) of a non-tiled buffer
int buffer_ptr(MeaoCtx *c, int id, void **p, size_t *pitch_bytes)
{
    if (id == 1) { *p = c->lin; *pitch_bytes = (size_t)c->lin_pitch * 2; }
    else if (id >= 2 && id <= 5) { *p = c->low[id - 1]; *pitch_bytes = (size_t)c->low_pitch[id - 1] * 4; }
    else if (id >= 10 && id <= 13) { *p = c->occ[id - 9]; *pitch_bytes = c->occ_pitch[id - 9]; }
    else if (id >= 14 && id <= 16) { *p = c->comb[id - 13]; *pitch_bytes = c->occ_pitch[id - 13]; }
    else if (id == 17) { *p = c->result; *pitch_bytes = c->result_pitch; }
    else if (id >= 18 && id <= 21) { *p = c->hq[id - 17]; *pitch_bytes = c->occ_pitch[id - 17]; }
    else return -1;
    return 0;
}

std::mutex g_event_mutex;
struct EventBinding { MeaoCtx *ctx; const void *depth; int kind; void *out; void *stream; };
std::map<int, EventBinding> g_events;

}  // namespace

// =================================================================================================
// C ABI
// =================================================================================================
extern "C" {

int meao_abi_version(void) { return MEAO_ABI_VERSION; }

void meao_default_params(MeaoParams *p)
{
    if (!p) return;
    p->noise_filter_tolerance = 0.0f;   // AO.cs:20
    p->blur_tolerance = -4.6f;          // AO.cs:28
    p->upsample_tolerance = -12.0f;     // AO.cs:36
    p->thickness_modifier = 1.0f;       // AO.cs:44
    p->intensity = 1.0f;                // AO.cs:52
    p->debug = 0;                       // AO.cs:60
    p->ambient_only = 1;                // AO.cs:68
}

int meao_create(const MeaoDeviceCfg *cfg, MeaoCtx **out)
{
    if (!out) return fail(nullptr, MEAO_ERR_INVALID, "out_ctx is NULL");
    *out = nullptr;
    if (cfg && cfg->device < 0) {       // host-side planner only: constants, geometry, band/halo ranges
        MeaoCtx *c = new MeaoCtx();
        c->device = -1; c->plan_only = true; c->flags = cfg->flags;
        meao_default_params(&c->params);
        c->camera = MeaoCamera{0.3f, 1000.0f, 1.0f, 1};
        *out = c;
        return MEAO_OK;
    }
    int ndev = 0;
    cudaError_t e = cudaGetDeviceCount(&ndev);
    if (e != cudaSuccess || ndev == 0)
        return fail(nullptr, MEAO_ERR_CUDA, "no CUDA device available (%s); libmeao has no CPU fallback",
                    e != cudaSuccess ? cudaGetErrorString(e) : "device count 0");
    const int dev = cfg ? cfg->device : 0;
    if (dev < 0 || dev >= ndev) return fail(nullptr, MEAO_ERR_INVALID, "device %d out of range (0..%d)", dev, ndev - 1);
    cudaDeviceProp prop;
    e = cudaGetDeviceProperties(&prop, dev);
    if (e != cudaSuccess) return fail(nullptr, MEAO_ERR_CUDA, "cudaGetDeviceProperties: %s", cudaGetErrorString(e));
    if (prop.major != 10)
        return fail(nullptr, MEAO_ERR_CUDA, "device %d is sm_%d%d; libmeao is built for sm_100a (B200) only", dev, prop.major, prop.minor);
    e = cudaSetDevice(dev);
    if (e != cudaSuccess) return fail(nullptr, MEAO_ERR_CUDA, "cudaSetDevice: %s", cudaGetErrorString(e));
    MeaoCtx *c = new MeaoCtx();
    c->device = dev;
    c->flags = cfg ? cfg->flags : 0;
    meao_default_params(&c->params);
    c->camera = MeaoCamera{0.3f, 1000.0f, 1.0f, 1};
    e = cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking);
    for (int i = 0; i < 3 && e == cudaSuccess; i++) e = cudaStreamCreateWithFlags(&c->branch[i], cudaStreamNonBlocking);
    for (int i = 0; i < 5 && e == cudaSuccess; i++) e = cudaEventCreateWithFlags(&c->ev[i], cudaEventDisableTiming);
    for (int i = 0; i < 2 && e == cudaSuccess; i++) e = cudaStreamCreateWithFlags(&c->slot_stream[i], cudaStreamNonBlocking);
    for (int i = 0; i < 2 && e == cudaSuccess; i++) e = cudaEventCreateWithFlags(&c->slot_done[i], cudaEventDisableTiming);
    if (e == cudaSuccess) e = cudaEventCreateWithFlags(&c->compute_done, cudaEventDisableTiming);
    if (e != cudaSuccess) { delete c; return fail(nullptr, MEAO_ERR_CUDA, "cudaStreamCreate: %s", cudaGetErrorString(e)); }
    if (cudaHostAlloc((void **)&c->host_error, 64, cudaHostAllocMapped) == cudaSuccess) {
        *c->host_error = 0;
        if (cudaHostGetDevicePointer((void **)&c->host_error_dev, c->host_error, 0) != cudaSuccess) c->host_error_dev = nullptr;
    } else c->host_error = nullptr;
    cudaGetLastError();
    {   // load every kernel of the library on this device NOW (kernels.h "eager loading"): a lazy load later could wait for a
        // spinning exchange kernel that in turn waits for the very launch that triggered the load
        static std::mutex preload_mutex;
        static std::map<int, bool> preloaded;
        std::lock_guard<std::mutex> g(preload_mutex);
        if (!preloaded[dev]) {
            cudaError_t pe = preload_prepare_depth();
            if (pe == cudaSuccess) pe = preload_render_ao();
            if (pe == cudaSuccess) pe = preload_blur_upsample();
            if (pe == cudaSuccess) pe = preload_blur_upsample_batch();
            if (pe == cudaSuccess) pe = preload_prepare_depth_batch();
            if (pe == cudaSuccess) pe = preload_render_ao_batch();
            if (pe == cudaSuccess) pe = preload_band_kernels();
            if (pe == cudaSuccess) pe = preload_aux_kernels();
            if (pe != cudaSuccess) { cudaGetLastError(); meao_destroy(c); return fail(nullptr, MEAO_ERR_CUDA, "loading the kernels failed: %s", cudaGetErrorString(pe)); }
            preloaded[dev] = true;
        }
    }
    void *fn = nullptr;
    cudaDriverEntryPointQueryResult qres;
    const char *no_tma = getenv("MEAO_DISABLE_TMA");     // debugging aid: force the gather path in every tile
    if (!(no_tma && no_tma[0] == '1') &&
        cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &qres) == cudaSuccess && qres == cudaDriverEntryPointSuccess)
        c->encode = (PFN_encodeTiled)fn;
    cudaGetLastError();
    *out = c;
    return MEAO_OK;
}

void meao_destroy(MeaoCtx *c)
{
    if (!c) return;
    {
        std::lock_guard<std::mutex> g(g_event_mutex);
        for (auto it = g_events.begin(); it != g_events.end();) { if (it->second.ctx == c) it = g_events.erase(it); else ++it; }
    }
    if (c->plan_only) { delete c; return; }
    cudaSetDevice(c->device);
    if (c->stream) cudaStreamSynchronize(c->stream);
    free_buffers(c);
    if (c->stream) cudaStreamDestroy(c->stream);
    for (auto b : c->branch) if (b) cudaStreamDestroy(b);
    for (auto e : c->ev) if (e) cudaEventDestroy(e);
    for (auto b : c->slot_stream) if (b) { cudaStreamSynchronize(b); cudaStreamDestroy(b); }
    for (auto e : c->slot_done) if (e) cudaEventDestroy(e);
    if (c->compute_done) cudaEventDestroy(c->compute_done);
    if (c->host_error) cudaFreeHost(c->host_error);
    delete c;
}

const char *meao_last_error(const MeaoCtx *c) { return c ? c->error.c_str() : g_create_error.c_str(); }

int meao_set_params(MeaoCtx *c, const MeaoParams *p)
{
    if (!c || !p) return MEAO_ERR_INVALID;
    // CheckPropertiesChanged, AO.cs:104-113 (ambient_only is not part of the change detection there either)
    bool changed = c->params.noise_filter_tolerance != p->noise_filter_tolerance || c->params.blur_tolerance != p->blur_tolerance ||
                   c->params.upsample_tolerance != p->upsample_tolerance || c->params.thickness_modifier != p->thickness_modifier ||
                   c->params.intensity != p->intensity || c->params.debug != p->debug;
    if (!(p->thickness_modifier > 0.0f)) return fail(c, MEAO_ERR_INVALID, "thickness_modifier must be > 0");
    c->params = *p;
    if (changed) c->plan_dirty = true;
    return changed ? 1 : 0;
}

int meao_get_params(const MeaoCtx *c, MeaoParams *out)
{
    if (!c || !out) return MEAO_ERR_INVALID;
    *out = c->params;
    return MEAO_OK;
}

int meao_set_variants(MeaoCtx *c, const MeaoVariants *v)
{
    if (!c || !v) return MEAO_ERR_INVALID;
    if (v->high_quality_mask < 0 || v->high_quality_mask > 15) return fail(c, MEAO_ERR_INVALID, "high_quality_mask %d not in 0..15", v->high_quality_mask);
    if (v->single_scale && v->high_quality_mask) return fail(c, MEAO_ERR_INVALID, "single_scale excludes high_quality_mask");
    MeaoVariants n{v->single_pass_stereo ? 1 : 0, v->sample_exhaustively ? 1 : 0, v->high_quality_mask, v->single_scale ? 1 : 0};
    const bool changed = memcmp(&c->variants, &n, sizeof n) != 0;
    c->variants = n;
    if (changed) c->plan_dirty = true;          // re-plan + drop the captured graphs (ensure_ready)
    return changed ? 1 : 0;
}

int meao_get_variants(const MeaoCtx *c, MeaoVariants *out)
{
    if (!c || !out) return MEAO_ERR_INVALID;
    *out = c->variants;
    return MEAO_OK;
}

int meao_set_camera(MeaoCtx *c, const MeaoCamera *cam)
{
    if (!c || !cam) return MEAO_ERR_INVALID;
    if (!(cam->near_clip > 0) || !(cam->far_clip > cam->near_clip) || !(cam->tan_half_fov_h > 0))
        return fail(c, MEAO_ERR_INVALID, "bad camera (near %g far %g tanHalfFovH %g)", cam->near_clip, cam->far_clip, cam->tan_half_fov_h);
    if (memcmp(&c->camera, cam, sizeof *cam) != 0) { c->camera = *cam; c->plan_dirty = true; }
    return MEAO_OK;
}

int meao_resize(MeaoCtx *c, int32_t w, int32_t h)
{
    if (!c) return MEAO_ERR_INVALID;
    if (w <= 0 || h <= 0 || w > 32768 || h > 32768) return fail(c, MEAO_ERR_INVALID, "bad size %dx%d", w, h);
    if (w == c->W && h == c->H && (c->arena || c->plan_only)) return 0;       // RTHandle.CheckBaseDimensions, AO.cs:145-148
    if (!c->plan_only) {
        CUDA_TRY(c, cudaSetDevice(c->device));
        CUDA_TRY(c, cudaStreamSynchronize(c->stream));
    }
    c->W = w; c->H = h;
    int rc = allocate(c);
    if (rc) { c->W = c->H = 0; return rc; }
    return 1;
}

int meao_set_row_band(MeaoCtx *c, int32_t row0, int32_t row1, int32_t prev_row0, int32_t next_row1)
{
    if (!c || c->W <= 0) return MEAO_ERR_INVALID;
    if (row0 < 0 || row1 > c->H || row0 >= row1 || (row0 % 16) || ((row1 % 16) && row1 != c->H))
        return fail(c, MEAO_ERR_INVALID, "band [%d,%d) must be 16-row aligned inside [0,%d)", row0, row1, c->H);
    if ((prev_row0 >= 0 && (prev_row0 % 16 || prev_row0 >= row0)) || (next_row1 >= 0 && (next_row1 <= row1 || next_row1 > c->H)))
        return fail(c, MEAO_ERR_INVALID, "bad neighbour extents");
    if ((row0 > 0) != (prev_row0 >= 0) || (row1 < c->H) != (next_row1 >= 0))
        return fail(c, MEAO_ERR_INVALID, "neighbour extents must be given exactly where the band is interior");
    // validate against temporaries; the context keeps its old band when the new one is refused
    {
        const BandNeeds n = compute_needs(c, row0, row1);
        for (int k = 1; k <= 4; k++) {
            if (n.need_low[k].lo < n.own_low[k].lo && (prev_row0 < 0 || n.need_low[k].lo < (prev_row0 >> k)))
                return fail(c, MEAO_ERR_UNSUPPORTED, "halo of level %d reaches beyond the band above", k);
            if (n.need_low[k].hi > n.own_low[k].hi && (next_row1 < 0 || n.need_low[k].hi > ((next_row1 + (1 << k) - 1) >> k)))
                return fail(c, MEAO_ERR_UNSUPPORTED, "halo of level %d reaches beyond the band below", k);
        }
    }
    if (!c->plan_only) {
        CUDA_TRY(c, cudaSetDevice(c->device));
        drop_graph(c);
        disconnect_peers(c);        // the halo ranges change: the host exports / connects again
    }
    c->band0 = row0; c->band1 = row1; c->prev0 = prev_row0; c->next1 = next_row1;
    return setup_band(c);
}

static void halo_ranges(MeaoCtx *c, int side, bool send, Range out[5])
{
    // send up:   rows of my own range that the band above needs  = [own.lo, above.need.hi)
    // recv up:   [need.lo, own.lo)
    for (int k = 1; k <= 4; k++) out[k] = Range{0, 0};
    if (side == 0 && c->prev0 < 0) return;
    if (side == 1 && c->next1 < 0) return;
    if (!send) {
        for (int k = 1; k <= 4; k++) {
            if (side == 0) out[k] = Range{c->need_low[k].lo, c->own_low[k].lo};
            else out[k] = Range{c->own_low[k].hi, c->need_low[k].hi};
            if (out[k].hi < out[k].lo) out[k].hi = out[k].lo;
        }
        return;
    }
    BandNeeds nb = (side == 0) ? compute_needs(c, c->prev0, c->band0) : compute_needs(c, c->band1, c->next1);
    for (int k = 1; k <= 4; k++) {
        if (side == 0) out[k] = Range{c->own_low[k].lo, nb.need_low[k].hi};
        else out[k] = Range{nb.need_low[k].lo, c->own_low[k].hi};
        if (out[k].hi < out[k].lo) out[k].hi = out[k].lo;
    }
}

static int64_t halo_size(MeaoCtx *c, int side, bool send)
{
    if (!c || c->W <= 0 || (side != 0 && side != 1)) return MEAO_ERR_INVALID;
    Range r[5]; halo_ranges(c, side, send, r);
    int64_t bytes = 0;
    for (int k = 1; k <= 4; k++) bytes += (int64_t)(r[k].hi - r[k].lo) * c->lw[k] * 4;
    return bytes;
}
int64_t meao_halo_bytes(MeaoCtx *c, int32_t side) { return halo_size(c, side, true); }
int meao_halo_rows(MeaoCtx *c, int32_t side, int32_t send, int32_t out8[8])
{
    if (!c || c->W <= 0 || (side != 0 && side != 1) || !out8) return MEAO_ERR_INVALID;
    Range r[5]; halo_ranges(c, side, send != 0, r);
    for (int k = 1; k <= 4; k++) { out8[2 * (k - 1)] = r[k].lo; out8[2 * (k - 1) + 1] = r[k].hi; }
    return MEAO_OK;
}
int meao_band_rows(MeaoCtx *c, int32_t out30[30])
{
    if (!c || c->W <= 0 || !out30) return MEAO_ERR_INVALID;
    for (int k = 0; k <= 4; k++) {
        out30[2 * k] = c->need_c[k].lo; out30[2 * k + 1] = c->need_c[k].hi;
        out30[10 + 2 * k] = c->need_low[k].lo; out30[10 + 2 * k + 1] = c->need_low[k].hi;
        out30[20 + 2 * k] = c->own_low[k].lo; out30[20 + 2 * k + 1] = c->own_low[k].hi;
    }
    return MEAO_OK;
}
int64_t meao_halo_recv_bytes(MeaoCtx *c, int32_t side) { return halo_size(c, side, false); }

static int halo_copy(MeaoCtx *c, int side, void *packed, bool pack, void *stream)
{
    int rc = ensure_ready(c); if (rc) return rc;
    if (side != 0 && side != 1) return fail(c, MEAO_ERR_INVALID, "side must be 0 or 1");
    cudaStream_t s = (cudaStream_t)stream;
    Range r[5]; halo_ranges(c, side, pack, r);
    char *p = (char *)packed;
    for (int k = 1; k <= 4; k++) {
        const int rows = r[k].hi - r[k].lo;
        if (rows <= 0) continue;
        const size_t wb = (size_t)c->lw[k] * 4, pb = (size_t)c->low_pitch[k] * 4;
        char *buf = (char *)(c->low[k] + (size_t)r[k].lo * c->low_pitch[k]);
        if (pack) CUDA_TRY(c, cudaMemcpy2DAsync(p, wb, buf, pb, wb, rows, cudaMemcpyDeviceToDevice, s));
        else      CUDA_TRY(c, cudaMemcpy2DAsync(buf, pb, p, wb, wb, rows, cudaMemcpyDeviceToDevice, s));
        p += wb * rows;
    }
    return MEAO_OK;
}
int meao_halo_pack(MeaoCtx *c, int32_t side, void *packed, void *stream) { return halo_copy(c, side, packed, true, stream); }
int meao_halo_unpack(MeaoCtx *c, int32_t side, const void *packed, void *stream) { return halo_copy(c, side, (void *)packed, false, stream); }

int meao_render_band_prepare(MeaoCtx *c, const void *depth, int32_t kind, void *stream)
{
    int rc = ensure_ready(c); if (rc) return rc;
    if (!depth) return fail(c, MEAO_ERR_INVALID, "depth is NULL");
    return record_downsample(c, depth, kind, (cudaStream_t)stream);
}

int meao_render_band_finish(MeaoCtx *c, void *ao_out, void *stream)
{
    int rc = ensure_ready(c); if (rc) return rc;
    cudaStream_t s = (cudaStream_t)stream;
    const int kind = c->last_kind;
    for (int k = 1; k <= 4; k++) if ((rc = record_render(c, k, kind, s))) return rc;
    for (int k = 1; k <= 4; k++) if (hq_level(c, k) && (rc = record_render(c, k, kind, s, true))) return rc;
    for (int lo = 4; lo >= 1; lo--) if ((rc = record_upsample(c, lo, lo == 1 ? ao_out : nullptr, s))) return rc;
    return MEAO_OK;
}

static int halo_kernel(MeaoCtx *c, void *up, void *down, bool pack, cudaStream_t s)
{
    HaloArgs a{}; a.nseg = 0;
    void *bufs[2] = {up, down};
    for (int side = 0; side < 2; side++) {
        if (!bufs[side]) continue;
        Range r[5]; halo_ranges(c, side, pack, r);
        float *p = (float *)bufs[side];
        for (int k = 1; k <= 4; k++) {
            const int rows = r[k].hi - r[k].lo;
            if (rows <= 0) continue;
            float *buf = c->low[k] + (size_t)r[k].lo * c->low_pitch[k];
            HaloSeg &g = a.seg[a.nseg++];
            if (pack) g = HaloSeg{buf, p, c->low_pitch[k], c->lw[k], c->lw[k], rows};
            else      g = HaloSeg{p, buf, c->lw[k], c->low_pitch[k], c->lw[k], rows};
            p += (size_t)rows * c->lw[k];
        }
    }
    CUDA_TRY(c, launch_halo_copy(a, s));
    if (a.nseg) c->launches++;
    return 0;
}

// ---- graph cache ----------------------------------------------------------------------------------------------------
// record(stream, pdl) issues the launches; it is captured into a graph, with the highest programmatic-dependent-launch
// level the runtime accepts (tried once per context: 2, then 1, then 0 = plain edges).
static int capture_graph(MeaoCtx *c, const std::function<int(cudaStream_t, int)> &record, cudaGraph_t *out)
{
    const char *env = getenv("MEAO_PDL");                           // tuning / debugging aid: cap the level (0 disables)
    const int cap = (env && env[0] >= '0' && env[0] <= '2') ? env[0] - '0' : 2;
    for (int level = (c->pdl_level >= 0 ? c->pdl_level : cap); level >= 0; level--) {
        cudaGraph_t g = nullptr;
        CUDA_TRY(c, cudaStreamBeginCapture(c->stream, cudaStreamCaptureModeThreadLocal));
        const int64_t before = c->launches;
        const int rc = record(c->stream, level);
        c->launches = before;
        const cudaError_t e = cudaStreamEndCapture(c->stream, &g);
        if (rc == 0 && e == cudaSuccess) { c->pdl_level = level; *out = g; return 0; }
        if (g) cudaGraphDestroy(g);
        cudaGetLastError();
        if (level == 0) {
            if (rc) return rc;
            return fail(c, MEAO_ERR_CUDA, "cudaStreamEndCapture: %s", cudaGetErrorString(e));
        }
        // a capture that failed with PDL edges is retried one level lower (mixed programmatic + event dependencies may be refused)
    }
    return fail(c, MEAO_ERR_CUDA, "graph capture failed");
}

static int launch_cached(MeaoCtx *c, const MeaoCtx::GraphKey &key, cudaStream_t s, int nk, const std::function<int(cudaStream_t, int)> &record)
{
    if (c->flags & MEAO_FLAG_NO_GRAPH) return record(s, 0);
    constexpr size_t kMaxGraphs = 64;
    auto it = c->graphs.find(key);
    if (it == c->graphs.end()) {
        cudaGraph_t g = nullptr;
        int rc = capture_graph(c, record, &g);
        if (rc) return rc;
        cudaGraphExec_t ge = nullptr;
        if (c->graphs.size() >= kMaxGraphs) {
            // a caller that rotates more buffers than the cache holds: re-target the least recently used executable graph
            // (same topology, new kernel arguments) instead of synchronising the device and instantiating again
            auto victim = c->graphs.begin();
            for (auto j = c->graphs.begin(); j != c->graphs.end(); ++j) if (j->second.last_use < victim->second.last_use) victim = j;
            cudaGraphExecUpdateResultInfo info;
            ge = victim->second.exec;
            if (cudaGraphExecUpdate(ge, g, &info) != cudaSuccess) { cudaGetLastError(); c->retired.push_back(ge); ge = nullptr; }
            c->graphs.erase(victim);
        }
        if (!ge) {
            cudaError_t e = cudaGraphInstantiate(&ge, g, 0);
            if (e != cudaSuccess && c->pdl_level > 0) {             // be conservative: fall back to plain edges once and for all
                cudaGetLastError();
                cudaGraphDestroy(g); g = nullptr;
                c->pdl_level = 0;
                if ((rc = capture_graph(c, record, &g))) return rc;
                e = cudaGraphInstantiate(&ge, g, 0);
            }
            if (e != cudaSuccess) { if (g) cudaGraphDestroy(g); return fail(c, MEAO_ERR_CUDA, "cudaGraphInstantiate: %s", cudaGetErrorString(e)); }
        }
        cudaGraphDestroy(g);
        it = c->graphs.emplace(key, MeaoCtx::GraphEntry{ge, 0}).first;
    }
    it->second.last_use = ++c->graph_clock;
    CUDA_TRY(c, cudaGraphLaunch(it->second.exec, s));
    c->launches += nk;
    return 0;
}

int meao_band_phase_a(MeaoCtx *c, const void *depth, int32_t kind, void *send_up, void *send_down, void *stream)
{
    int rc = ensure_ready(c); if (rc) return rc;
    if (!depth) return fail(c, MEAO_ERR_INVALID, "depth is NULL");
    c->last_kind = kind;
    const MeaoCtx::GraphKey key{{depth, send_up, send_down, nullptr}, 100 + kind};
    const int nk = 1 + ((send_up || send_down) ? 1 : 0);
    return launch_cached(c, key, (cudaStream_t)stream, nk, [&](cudaStream_t s, int pdl) {
        int r = record_downsample(c, depth, kind, s);
        if (r) return r;
        PdlScope p(pdl >= 1);
        return halo_kernel(c, send_up, send_down, true, s);
    });
}

int meao_band_phase_b(MeaoCtx *c, const void *recv_up, const void *recv_down, void *ao_out, void *stream)
{
    int rc = ensure_ready(c); if (rc) return rc;
    if (!ao_out) return fail(c, MEAO_ERR_INVALID, "ao_out is NULL");
    const int kind = c->last_kind;
    const MeaoCtx::GraphKey key{{recv_up, recv_down, ao_out, nullptr}, 200 + kind};
    const int nk = meao_kernels_per_frame(c) - 1 + ((recv_up || recv_down) ? 1 : 0);
    c->last_out = ao_out;
    return launch_cached(c, key, (cudaStream_t)stream, nk, [&](cudaStream_t s, int pdl) {
        int r = halo_kernel(c, (void *)recv_up, (void *)recv_down, false, s);
        if (r) return r;
        return record_frame_dag(c, nullptr, kind, ao_out, s, false, pdl);
    });
}

// ---- native neighbour exchange (include/meao.h) -----------------------------------------------------------------------
namespace {
struct PeerHandlePod {              // what MeaoPeerHandle carries (<= MEAO_PEER_HANDLE_BYTES)
    uint32_t magic;                 // 'MEAO'
    int32_t device;
    int64_t pid;
    int32_t W, H;
    uint64_t arena_bytes;
    uint64_t arena_ptr;             // valid in the exporting process only
    cudaIpcMemHandle_t ipc;         // valid in every other process on this node
};
static_assert(sizeof(PeerHandlePod) <= MEAO_PEER_HANDLE_BYTES, "MeaoPeerHandle too small");
constexpr uint32_t kPeerMagic = 0x4d45414fu;
}  // namespace

int meao_band_export(MeaoCtx *c, MeaoPeerHandle *out)
{
    int rc = ensure_ready(c); if (rc) return rc;
    if (!out) return fail(c, MEAO_ERR_INVALID, "out is NULL");
    PeerHandlePod h{};
    h.magic = kPeerMagic; h.device = c->device; h.pid = (int64_t)getpid(); h.W = c->W; h.H = c->H;
    h.arena_bytes = c->arena_bytes; h.arena_ptr = (uint64_t)(uintptr_t)c->arena;
    const cudaError_t e = cudaIpcGetMemHandle(&h.ipc, c->arena);
    if (e != cudaSuccess) { cudaGetLastError(); memset(&h.ipc, 0, sizeof h.ipc); }     // in-process peers still work without IPC
    memset(out, 0, sizeof *out);
    memcpy(out->bytes, &h, sizeof h);
    return MEAO_OK;
}

int meao_band_connect(MeaoCtx *c, int32_t side, const MeaoPeerHandle *peer)
{
    int rc = ensure_ready(c); if (rc) return rc;
    if (side != 0 && side != 1) return fail(c, MEAO_ERR_INVALID, "side must be 0 (up) or 1 (down)");
    drop_graph(c);                                  // captured band steps carry the old peer pointers
    if (c->peer_base[side] && c->peer_ipc[side]) cudaIpcCloseMemHandle(c->peer_base[side]);
    c->peer_base[side] = nullptr; c->peer_ipc[side] = false;
    if (!peer) return MEAO_OK;
    if ((side == 0 && c->prev0 < 0) || (side == 1 && c->next1 < 0)) return fail(c, MEAO_ERR_INVALID, "this band has no neighbour on side %d", side);
    {   // The epoch counters of neighbouring bands advance in lock step from 1.  A context that has already stepped can only be
        // (re)connected as a whole: with the other side still attached its epoch cannot restart, and the new neighbour starts at 1.
        BandFlags f{};
        CUDA_TRY(c, cudaMemcpy(&f, c->band_flags, sizeof f, cudaMemcpyDeviceToHost));
        if (f.epoch != 1 || f.error != 0) {
            if (c->peer_base[side ^ 1])
                return fail(c, MEAO_ERR_INVALID, "this band has stepped (epoch %u): disconnect BOTH sides, then connect them again -- every band of the frame restarts at epoch 1", f.epoch);
            BandFlags init{}; init.epoch = 1;
            CUDA_TRY(c, cudaMemcpy(c->band_flags, &init, sizeof init, cudaMemcpyHostToDevice));
            if (c->host_error) *c->host_error = 0;
        }
    }
    PeerHandlePod h;
    memcpy(&h, peer->bytes, sizeof h);
    if (h.magic != kPeerMagic) return fail(c, MEAO_ERR_INVALID, "not a MeaoPeerHandle");
    if (h.W != c->W || h.H != c->H || h.arena_bytes != c->arena_bytes)
        return fail(c, MEAO_ERR_INVALID, "neighbour frame %dx%d (arena %llu B) differs from this context's %dx%d (%zu B)", h.W, h.H,
                    (unsigned long long)h.arena_bytes, c->W, c->H, c->arena_bytes);
    if (h.pid == (int64_t)getpid()) {
        if (h.device != c->device) {
            int can = 0;
            CUDA_TRY(c, cudaDeviceCanAccessPeer(&can, c->device, h.device));
            if (!can) return fail(c, MEAO_ERR_UNSUPPORTED, "device %d cannot access device %d", c->device, h.device);
            const cudaError_t e = cudaDeviceEnablePeerAccess(h.device, 0);
            if (e != cudaSuccess && e != cudaErrorPeerAccessAlreadyEnabled) return fail(c, MEAO_ERR_CUDA, "cudaDeviceEnablePeerAccess: %s", cudaGetErrorString(e));
            cudaGetLastError();
        }
        c->peer_base[side] = (void *)(uintptr_t)h.arena_ptr;
    } else {
        void *p = nullptr;
        const cudaError_t e = cudaIpcOpenMemHandle(&p, h.ipc, cudaIpcMemLazyEnablePeerAccess);
        if (e != cudaSuccess) { cudaGetLastError(); return fail(c, MEAO_ERR_CUDA, "cudaIpcOpenMemHandle: %s", cudaGetErrorString(e)); }
        c->peer_base[side] = p; c->peer_ipc[side] = true;
    }
    const char *t = getenv("MEAO_BAND_TIMEOUT_MS");
    if (t && atof(t) > 0) c->band_timeout_ns = (unsigned long long)(atof(t) * 1e6);
    return MEAO_OK;
}

// prepare_depth on the band has run: push my border rows into the neighbours' LowDepth1..4, signal, wait for theirs
static int record_exchange(MeaoCtx *c, cudaStream_t s)
{
    NvtxRange nv("meao::band_exchange");
    XchgArgs a{}; a.nseg = 0;
    a.local = c->band_flags;
    a.host_error = c->host_error_dev;
    a.timeout_ns = c->band_timeout_ns;
    for (int side = 0; side < 2; side++) {
        a.peer[side] = (BandFlags *)c->peer_base[side];                 // BandFlags sit at offset 0 of every arena
        if (!c->peer_base[side]) continue;
        Range r[5]; halo_ranges(c, side, true, r);
        for (int k = 1; k <= 4; k++) {
            const int rows = r[k].hi - r[k].lo;
            if (rows <= 0) continue;
            const size_t off = (size_t)((char *)(c->low[k] + (size_t)r[k].lo * c->low_pitch[k]) - (char *)c->arena);
            const size_t bytes = (size_t)rows * c->low_pitch[k] * sizeof(float);          // whole pitched rows: contiguous, 128 B aligned
            XchgSeg &g = a.seg[a.nseg++];
            g.src = (const uint4 *)((char *)c->arena + off);
            g.dst = (uint4 *)((char *)c->peer_base[side] + off);
            g.n16 = (uint32_t)(bytes / 16); g.side = side;
        }
    }
    if (a.nseg == 0) return 0;
    CUDA_TRY(c, launch_band_exchange(a, s));
    c->launches++;
    return 0;
}

int meao_band_step(MeaoCtx *c, const void *depth, int32_t kind, void *ao_out, void *stream)
{
    int rc = ensure_ready(c); if (rc) return rc;
    if (!depth || !ao_out) return fail(c, MEAO_ERR_INVALID, "depth / ao_out is NULL");
    if ((c->prev0 >= 0 && !c->peer_base[0]) || (c->next1 >= 0 && !c->peer_base[1]))
        return fail(c, MEAO_ERR_INVALID, "meao_band_step: connect every neighbour first (meao_band_export / meao_band_connect)");
    // a time-out of an earlier step is sticky; the kernel mirrors it into a mapped host word, so this costs no CUDA call
    if (c->host_error && *(volatile uint32_t *)c->host_error != 0)
        return fail(c, MEAO_ERR_PEER, "neighbour exchange timed out earlier (error %u): see meao_band_status", *(volatile uint32_t *)c->host_error);
    NvtxRange nv("meao::band_step");
    c->last_kind = kind; c->last_out = ao_out;
    const MeaoCtx::GraphKey key{{depth, ao_out, c->peer_base[0], c->peer_base[1]}, 300 + kind};
    const bool has_peer = c->peer_base[0] || c->peer_base[1];
    const int nk = meao_kernels_per_frame(c) + (has_peer ? 1 : 0);
    return launch_cached(c, key, (cudaStream_t)stream, nk, [&](cudaStream_t s, int pdl) {
        int r = record_downsample(c, depth, kind, s);
        if (r) return r;
        { PdlScope p(pdl >= 1); if ((r = record_exchange(c, s))) return r; }
        return record_frame_dag(c, nullptr, kind, ao_out, s, false, pdl, has_peer);
    });
}

int meao_band_step_host(MeaoCtx *c, const void *depth_host, int32_t kind, uint8_t *ao_host)
{
    int rc = ensure_ready(c); if (rc) return rc;
    if (!depth_host || !ao_host) return fail(c, MEAO_ERR_INVALID, "depth / ao_out is NULL");
    if (kind < MEAO_DEPTH_RAW_F32 || kind > MEAO_DEPTH_RAW_D24S8) return fail(c, MEAO_ERR_INVALID, "bad depth kind %d", kind);
    const size_t rows = (size_t)(c->band1 - c->band0);
    cudaStream_t s = c->slot_stream[0];
    const size_t esz = (kind == MEAO_DEPTH_RAW_D16_UNORM) ? 2 : 4;
    CUDA_TRY(c, cudaMemcpyAsync(c->depth_stage[0], depth_host, rows * c->W * esz, cudaMemcpyHostToDevice, s));
    if ((rc = meao_band_step(c, c->depth_stage[0], kind, c->ao_stage[0], s))) return rc;
    CUDA_TRY(c, cudaMemcpyAsync(ao_host, c->ao_stage[0], rows * c->W, cudaMemcpyDeviceToHost, s));
    return MEAO_OK;
}

int meao_band_status(MeaoCtx *c, int32_t out4[4])
{
    if (!c || !out4 || c->plan_only || !c->band_flags) return MEAO_ERR_INVALID;
    CUDA_TRY(c, cudaSetDevice(c->device));
    BandFlags f{};
    // a dedicated non-blocking stream: never waits for (or delays) the frames in flight
    CUDA_TRY(c, cudaMemcpyAsync(&f, c->band_flags, sizeof f, cudaMemcpyDeviceToHost, c->slot_stream[1]));
    CUDA_TRY(c, cudaStreamSynchronize(c->slot_stream[1]));
    out4[0] = (int32_t)f.epoch; out4[1] = (int32_t)f.error; out4[2] = c->peer_base[0] ? 1 : 0; out4[3] = c->peer_base[1] ? 1 : 0;
    return MEAO_OK;
}

int meao_render(MeaoCtx *c, const void *depth, int32_t kind, void *ao_out, void *stream)
{
    int rc = ensure_ready(c); if (rc) return rc;
    if (!depth || !ao_out) return fail(c, MEAO_ERR_INVALID, "depth / ao_out is NULL");
    if (kind < MEAO_DEPTH_RAW_F32 || kind > MEAO_DEPTH_RAW_D24S8) return fail(c, MEAO_ERR_INVALID, "bad depth kind %d", kind);
    if (c->need_low[1].lo < c->own_low[1].lo || c->need_low[1].hi > c->own_low[1].hi)
        return fail(c, MEAO_ERR_INVALID, "interior row band: use meao_render_band_prepare / halo exchange / meao_render_band_finish");
    cudaStream_t s = (cudaStream_t)stream;
    if (c->flags & MEAO_FLAG_NO_GRAPH) return record_frame(c, depth, kind, ao_out, s, false);

    // plan-once / replay: one captured graph per (depth, out, kind), like the reference's command buffer
    // that is re-recorded only when something changed (AO.cs:334-347)
    NvtxRange nv("meao::frame");
    const MeaoCtx::GraphKey key{{depth, ao_out, nullptr, nullptr}, kind};
    c->last_kind = kind; c->last_out = ao_out;
    return launch_cached(c, key, s, meao_kernels_per_frame(c), [&](cudaStream_t cs, int pdl) {
        return record_frame_dag(c, depth, kind, ao_out, cs, true, pdl);
    });
}

int meao_reserve_batch(MeaoCtx *c, int32_t frames)
{
    int rc = ensure_ready(c); if (rc) return rc;
    if (frames < 1 || frames > 65535) return fail(c, MEAO_ERR_INVALID, "frames %d not in 1..65535", frames);
    return reserve_batch(c, frames);
}

int meao_render_batch(MeaoCtx *c, const void *depth, int32_t kind, int32_t frames, void *ao_out, void *stream)
{
    int rc = ensure_ready(c); if (rc) return rc;
    if (!depth || !ao_out) return fail(c, MEAO_ERR_INVALID, "depth / ao_out is NULL");
    if (kind < MEAO_DEPTH_RAW_F32 || kind > MEAO_DEPTH_RAW_D24S8) return fail(c, MEAO_ERR_INVALID, "bad depth kind %d", kind);
    if (frames < 1 || frames > 65535) return fail(c, MEAO_ERR_INVALID, "frames %d not in 1..65535", frames);
    if (c->band0 != 0 || c->band1 != c->H) return fail(c, MEAO_ERR_UNSUPPORTED, "batched frames need a whole-frame context (no row band)");
    if ((rc = reserve_batch(c, frames))) return rc;
    cudaStream_t s = (cudaStream_t)stream;
    const size_t esz = (kind == MEAO_DEPTH_RAW_D16_UNORM) ? 2 : 4;
    const BatchRun run{frames, (long long)c->W * c->H * (long long)esz};
    c->batch.last_frames = frames;
    if (c->flags & MEAO_FLAG_NO_GRAPH) return record_frame(c, depth, kind, ao_out, s, false, &run);
    // one graph replay for the whole batch: the DAG of record_frame_dag, every node covering all frames
    NvtxRange nv("meao::batch");
    const MeaoCtx::GraphKey key{{depth, ao_out, (const void *)(uintptr_t)frames, c->batch.base}, 400 + kind};
    return launch_cached(c, key, s, meao_kernels_per_frame(c), [&](cudaStream_t cs, int pdl) {
        return record_frame_dag(c, depth, kind, ao_out, cs, true, pdl, false, &run);
    });
}

int meao_get_batch_buffer(MeaoCtx *c, int32_t frame, int32_t id, void *host_out, size_t host_bytes)
{
    int rc = ensure_ready(c); if (rc) return rc;
    int lvl, slices, elem;
    if (!host_out || id == MEAO_BUF_AMBIENT_OCCLUSION || buffer_info(c, id, &lvl, &slices, &elem))
        return fail(c, MEAO_ERR_INVALID, "bad batch buffer id %d (the AO of a batch is in the caller's buffer)", id);
    const BatchArena &b = c->batch;
    if (frame < 0 || frame >= b.last_frames) return fail(c, MEAO_ERR_INVALID, "frame %d not in the last batch (%d frames)", frame, b.last_frames);
    const size_t need = (size_t)c->lw[lvl] * c->lh[lvl] * slices * elem;
    if (host_bytes < need) return fail(c, MEAO_ERR_INVALID, "buffer %d needs %zu bytes, got %zu", id, need, host_bytes);
    CUDA_TRY(c, cudaDeviceSynchronize());     // debug path: batches may be in flight on any caller stream
    const size_t fo = (size_t)frame * b.slot_bytes;
    if (slices == 16) {
        const int k = id - 5;
        __half *tmp = nullptr;
        CUDA_TRY(c, cudaMalloc(&tmp, need));
        const float pad = host_f16_round((b.last_kind != MEAO_DEPTH_LINEAR_F32) ? c->plan.pad[k] : 0.0f);
        cudaError_t e = launch_synth_tiled((const float *)((const char *)b.low[k] + fo), c->lw[k], c->lh[k], c->low_pitch[k], c->lw[k + 2], c->lh[k + 2], pad, tmp, c->stream);
        if (e == cudaSuccess) e = cudaMemcpyAsync(host_out, tmp, need, cudaMemcpyDeviceToHost, c->stream);
        if (e == cudaSuccess) e = cudaStreamSynchronize(c->stream);
        cudaFree(tmp);
        if (e != cudaSuccess) return fail(c, MEAO_ERR_CUDA, "tiled view: %s", cudaGetErrorString(e));
        return MEAO_OK;
    }
    const void *p; size_t pitch;
    if (id == 1) { p = b.lin; pitch = (size_t)c->lin_pitch * 2; }
    else if (id >= 2 && id <= 5) { p = b.low[id - 1]; pitch = (size_t)c->low_pitch[id - 1] * 4; }
    else if (id >= 10 && id <= 13) { p = b.occ[id - 9]; pitch = c->occ_pitch[id - 9]; }
    else if (id >= 14 && id <= 16) { p = b.comb[id - 13]; pitch = c->occ_pitch[id - 13]; }
    else { p = b.hq[id - 17]; pitch = c->occ_pitch[id - 17]; }
    const size_t wb = (size_t)c->lw[lvl] * elem;
    CUDA_TRY(c, cudaMemcpy2DAsync(host_out, wb, (const char *)p + fo, pitch, wb, c->lh[lvl], cudaMemcpyDeviceToHost, c->stream));
    CUDA_TRY(c, cudaStreamSynchronize(c->stream));
    return MEAO_OK;
}

int meao_render_host_async(MeaoCtx *c, const void *depth_host, int32_t kind, uint8_t *ao_host, int32_t slot)
{
    int rc = ensure_ready(c); if (rc) return rc;
    if (!depth_host || !ao_host) return fail(c, MEAO_ERR_INVALID, "depth / ao_out is NULL");
    if (slot != 0 && slot != 1) return fail(c, MEAO_ERR_INVALID, "slot must be 0 or 1");
    const size_t rows = (size_t)(c->band1 - c->band0);
    cudaStream_t s = c->slot_stream[slot];
    const size_t esz = (kind == MEAO_DEPTH_RAW_D16_UNORM) ? 2 : 4;
    CUDA_TRY(c, cudaMemcpyAsync(c->depth_stage[slot], depth_host, rows * c->W * esz, cudaMemcpyHostToDevice, s));
    // the two slots share the context's intermediates: kernels of consecutive frames are serialised, copies are not
    if (c->compute_done_valid) CUDA_TRY(c, cudaStreamWaitEvent(s, c->compute_done, 0));
    if ((rc = meao_render(c, c->depth_stage[slot], kind, c->ao_stage[slot], s))) return rc;
    CUDA_TRY(c, cudaEventRecord(c->compute_done, s));
    c->compute_done_valid = true;
    CUDA_TRY(c, cudaMemcpyAsync(ao_host, c->ao_stage[slot], rows * c->W, cudaMemcpyDeviceToHost, s));
    CUDA_TRY(c, cudaEventRecord(c->slot_done[slot], s));
    return MEAO_OK;
}

int meao_host_wait(MeaoCtx *c, int32_t slot)
{
    if (!c || (slot != 0 && slot != 1)) return MEAO_ERR_INVALID;
    if (c->plan_only) return MEAO_OK;
    CUDA_TRY(c, cudaSetDevice(c->device));
    CUDA_TRY(c, cudaStreamSynchronize(c->slot_stream[slot]));
    return MEAO_OK;
}

int meao_render_host(MeaoCtx *c, const void *depth_host, int32_t kind, uint8_t *ao_host)
{
    int rc = meao_render_host_async(c, depth_host, kind, ao_host, 0);
    if (rc) return rc;
    return meao_host_wait(c, 0);
}

int meao_synchronize(MeaoCtx *c)
{
    if (!c) return MEAO_ERR_INVALID;
    if (c->plan_only) return MEAO_OK;
    CUDA_TRY(c, cudaSetDevice(c->device));
    CUDA_TRY(c, cudaStreamSynchronize(c->stream));
    for (auto st : c->slot_stream) CUDA_TRY(c, cudaStreamSynchronize(st));
    return MEAO_OK;
}

void *meao_host_alloc(size_t bytes)
{
    void *p = nullptr;
    if (cudaHostAlloc(&p, bytes, cudaHostAllocDefault) != cudaSuccess) { cudaGetLastError(); return nullptr; }
    return p;
}
void meao_host_free(void *p) { if (p) cudaFreeHost(p); }

int meao_stage_downsample(MeaoCtx *c, const void *depth, int32_t kind, void *stream)
{
    int rc = ensure_ready(c); if (rc) return rc;
    if (!depth) return fail(c, MEAO_ERR_INVALID, "depth is NULL");
    return record_downsample(c, depth, kind, (cudaStream_t)stream);
}

int meao_stage_render(MeaoCtx *c, int32_t level, void *stream)
{
    int rc = ensure_ready(c); if (rc) return rc;
    if (level < 1 || level > 4) return fail(c, MEAO_ERR_INVALID, "render level %d not in 1..4", level);
    return record_render(c, level, c->last_kind, (cudaStream_t)stream);
}

int meao_stage_render_wide(MeaoCtx *c, int32_t level, void *stream)
{
    int rc = ensure_ready(c); if (rc) return rc;
    if (level < 1 || level > 4) return fail(c, MEAO_ERR_INVALID, "render level %d not in 1..4", level);
    return record_render(c, level, c->last_kind, (cudaStream_t)stream, true);
}

int meao_stage_upsample(MeaoCtx *c, int32_t lo_level, void *ao_out, void *stream)
{
    int rc = ensure_ready(c); if (rc) return rc;
    if (lo_level < 1 || lo_level > 4) return fail(c, MEAO_ERR_INVALID, "upsample lo level %d not in 1..4", lo_level);
    return record_upsample(c, lo_level, lo_level == 1 ? ao_out : nullptr, (cudaStream_t)stream);
}

int meao_buffer_desc(const MeaoCtx *c, int32_t id, MeaoBufferDesc *out)
{
    if (!c || !out || c->W <= 0) return MEAO_ERR_INVALID;
    int lvl, slices, elem;
    if (buffer_info(c, id, &lvl, &slices, &elem)) return MEAO_ERR_INVALID;
    out->width = c->lw[lvl]; out->height = c->lh[lvl]; out->slices = slices; out->elem_bytes = elem;
    return MEAO_OK;
}

int meao_get_buffer(MeaoCtx *c, int32_t id, void *host_out, size_t host_bytes)
{
    int rc = ensure_ready(c); if (rc) return rc;
    int lvl, slices, elem;
    if (!host_out || buffer_info(c, id, &lvl, &slices, &elem)) return fail(c, MEAO_ERR_INVALID, "bad buffer id %d", id);
    const size_t need = (size_t)c->lw[lvl] * c->lh[lvl] * slices * elem;
    if (host_bytes < need) return fail(c, MEAO_ERR_INVALID, "buffer %d needs %zu bytes, got %zu", id, need, host_bytes);
    CUDA_TRY(c, cudaDeviceSynchronize());     // debug path: frames may be in flight on any caller stream
    if (slices == 16) {
        const int k = id - 5;
        __half *tmp = nullptr;
        CUDA_TRY(c, cudaMalloc(&tmp, need));
        const float pad = host_f16_round((c->last_kind != MEAO_DEPTH_LINEAR_F32) ? c->plan.pad[k] : 0.0f);
        cudaError_t e = launch_synth_tiled(c->low[k], c->lw[k], c->lh[k], c->low_pitch[k], c->lw[k + 2], c->lh[k + 2], pad, tmp, c->stream);
        if (e == cudaSuccess) e = cudaMemcpyAsync(host_out, tmp, need, cudaMemcpyDeviceToHost, c->stream);
        if (e == cudaSuccess) e = cudaStreamSynchronize(c->stream);
        cudaFree(tmp);
        if (e != cudaSuccess) return fail(c, MEAO_ERR_CUDA, "tiled view: %s", cudaGetErrorString(e));
        return MEAO_OK;
    }
    void *p; size_t pitch;
    buffer_ptr(c, id, &p, &pitch);
    const size_t wb = (size_t)c->lw[lvl] * elem;
    if (id == MEAO_BUF_AMBIENT_OCCLUSION && c->last_out) {
        // the last frame wrote the AO texture straight into the caller's buffer; regenerate the debug view
        // from the (still resident) Combined1 / LowDepth1 / LinearDepth with the same kernel
        const int64_t before = c->launches;
        if ((rc = record_upsample(c, 1, nullptr, c->stream))) return rc;
        c->launches = before;
    }
    CUDA_TRY(c, cudaMemcpy2DAsync(host_out, wb, p, pitch, wb, c->lh[lvl], cudaMemcpyDeviceToHost, c->stream));
    CUDA_TRY(c, cudaStreamSynchronize(c->stream));
    return MEAO_OK;
}

int meao_debug_view(MeaoCtx *c, int32_t id, void *out, void *stream)
{
    int rc = ensure_ready(c); if (rc) return rc;
    int lvl, slices, elem;
    if (!out || buffer_info(c, id, &lvl, &slices, &elem)) return fail(c, MEAO_ERR_INVALID, "bad buffer id %d / out is NULL", id);
    if (c->band0 != 0 || c->band1 != c->H) return fail(c, MEAO_ERR_UNSUPPORTED, "debug views need a whole-frame context (no row band)");
    cudaStream_t s = (cudaStream_t)stream;
    DebugViewArgs a{};
    a.W = c->W; a.H = c->H; a.out = (uint8_t *)out; a.out_pitch = c->W;
    if (slices == 16) {                                             // AO.cs:810-814: Blit.shader pass 4
        const int k = id - 5;
        a.tiled = 1; a.src = c->low[k]; a.elem = 4; a.spitch = c->low_pitch[k];
        a.sw = c->lw[k + 2]; a.sh = c->lh[k + 2]; a.lw = c->lw[k]; a.lh = c->lh[k];
        a.pad = host_f16_round((c->last_kind != MEAO_DEPTH_LINEAR_F32) ? c->plan.pad[k] : 0.0f);
    } else {                                                        // AO.cs:815-819
        if (id == MEAO_BUF_AMBIENT_OCCLUSION && c->last_out) {
            // the last frame wrote the AO texture straight into the caller's buffer: regenerate the context's own copy
            const int64_t before = c->launches;
            if ((rc = record_upsample(c, 1, nullptr, s))) return rc;
            c->launches = before;
        }
        void *p; size_t pitch;
        buffer_ptr(c, id, &p, &pitch);
        a.src = p; a.elem = elem; a.spitch = (int)(pitch / elem); a.sw = c->lw[lvl]; a.sh = c->lh[lvl];
    }
    CUDA_TRY(c, launch_debug_view(a, s));
    c->launches++;
    return MEAO_OK;
}

int meao_set_buffer(MeaoCtx *c, int32_t id, const void *host_in, size_t host_bytes)
{
    int rc = ensure_ready(c); if (rc) return rc;
    int lvl, slices, elem;
    if (!host_in || buffer_info(c, id, &lvl, &slices, &elem) || slices != 1)
        return fail(c, MEAO_ERR_INVALID, "buffer id %d cannot be set", id);
    const size_t need = (size_t)c->lw[lvl] * c->lh[lvl] * elem;
    if (host_bytes < need) return fail(c, MEAO_ERR_INVALID, "buffer %d needs %zu bytes, got %zu", id, need, host_bytes);
    void *p; size_t pitch;
    buffer_ptr(c, id, &p, &pitch);
    const size_t wb = (size_t)c->lw[lvl] * elem;
    CUDA_TRY(c, cudaDeviceSynchronize());
    CUDA_TRY(c, cudaMemcpy2DAsync(p, pitch, host_in, wb, wb, c->lh[lvl], cudaMemcpyHostToDevice, c->stream));
    CUDA_TRY(c, cudaStreamSynchronize(c->stream));
    return MEAO_OK;
}

// The constant getters work without a device context being current: they only need the plan.
static int plan_only(MeaoCtx *c)
{
    if (!c || c->W <= 0) return MEAO_ERR_INVALID;
    if (c->plan_dirty) { build_plan(c); c->graphs_stale = true; }    // the captured graphs are dropped by the next ensure_ready, on c->device
    return 0;
}

int meao_render_constants(MeaoCtx *c, int32_t level, float out[28])
{
    if (plan_only(c) || !out || level < 1 || level > 4) return MEAO_ERR_INVALID;
    memcpy(out, c->plan.inv_thickness[level], 48);
    memcpy(out + 12, c->plan.sample_weight[level], 48);
    out[24] = c->plan.inv_slice_dim[level][0]; out[25] = c->plan.inv_slice_dim[level][1];
    out[26] = c->plan.reject_fadeoff; out[27] = c->plan.intensity;
    return MEAO_OK;
}

int meao_render_constants_wide(MeaoCtx *c, int32_t level, float out[28])
{
    if (plan_only(c) || !out || level < 1 || level > 4) return MEAO_ERR_INVALID;
    memcpy(out, c->plan.inv_thickness_wide[level], 48);
    memcpy(out + 12, c->plan.sample_weight[level], 48);
    out[24] = c->plan.inv_slice_dim_wide[level][0]; out[25] = c->plan.inv_slice_dim_wide[level][1];
    out[26] = c->plan.reject_fadeoff; out[27] = c->plan.intensity;
    return MEAO_OK;
}

int meao_upsample_constants(MeaoCtx *c, int32_t lo, float out[8])
{
    if (plan_only(c) || !out || lo < 1 || lo > 4) return MEAO_ERR_INVALID;
    out[0] = c->plan.inv_low[lo][0]; out[1] = c->plan.inv_low[lo][1];
    out[2] = c->plan.inv_high[lo][0]; out[3] = c->plan.inv_high[lo][1];
    out[4] = c->plan.noise_filter_strength[lo]; out[5] = c->plan.step_size[lo];
    out[6] = c->plan.blur_tolerance[lo]; out[7] = c->plan.upsample_tolerance[lo];
    return MEAO_OK;
}

int meao_zbuffer_params(MeaoCtx *c, float out[4])
{
    if (plan_only(c) || !out) return MEAO_ERR_INVALID;
    memcpy(out, c->plan.zb, 16);
    return MEAO_OK;
}

static int composite_args(MeaoCtx *c, const void *ao, const void *color, int fmt)
{
    if (!ao || !color) return fail(c, MEAO_ERR_INVALID, "ao / colour target is NULL");
    if (fmt != MEAO_FMT_RGBA8_UNORM && fmt != MEAO_FMT_RGBA16_FLOAT) return fail(c, MEAO_ERR_INVALID, "bad colour format %d", fmt);
    if (((uintptr_t)ao & 3) || ((uintptr_t)color & 15)) return fail(c, MEAO_ERR_INVALID, "composite needs a 4-byte aligned AO and a 16-byte aligned colour pointer");
    return 0;
}

int meao_composite_framebuffer(MeaoCtx *c, const void *ao, void *color, int32_t fmt, void *stream)
{
    int rc = ensure_ready(c); if (rc) return rc;
    if ((rc = composite_args(c, ao, color, fmt))) return rc;
    const long long npix = (long long)c->W * (c->band1 - c->band0);
    CUDA_TRY(c, launch_composite((const uint8_t *)ao, color, npix, fmt == MEAO_FMT_RGBA16_FLOAT, 1, 1, 0, (cudaStream_t)stream));
    c->launches++;
    return MEAO_OK;
}

int meao_composite_gbuffer(MeaoCtx *c, const void *ao, void *g0, void *g3, int32_t fmt3, void *stream)
{
    int rc = ensure_ready(c); if (rc) return rc;
    if ((rc = composite_args(c, ao, g0, MEAO_FMT_RGBA8_UNORM)) || (rc = composite_args(c, ao, g3, fmt3))) return rc;
    const long long npix = (long long)c->W * (c->band1 - c->band0);
    CUDA_TRY(c, launch_composite((const uint8_t *)ao, g0, npix, 0, 0, 1, 1, (cudaStream_t)stream));                               // gbuffer0.a
    CUDA_TRY(c, launch_composite((const uint8_t *)ao, g3, npix, fmt3 == MEAO_FMT_RGBA16_FLOAT, 1, 0, 1, (cudaStream_t)stream));   // gbuffer3.rgb
    c->launches += 2;
    return MEAO_OK;
}

int meao_composite_debug(MeaoCtx *c, const void *view, void *color, int32_t fmt, void *stream)
{
    int rc = ensure_ready(c); if (rc) return rc;
    if ((rc = composite_args(c, view, color, fmt))) return rc;
    const long long npix = (long long)c->W * (c->band1 - c->band0);
    CUDA_TRY(c, launch_debug_composite((const uint8_t *)view, color, npix, fmt == MEAO_FMT_RGBA16_FLOAT, (cudaStream_t)stream));
    c->launches++;
    return MEAO_OK;
}

int meao_bind_event(MeaoCtx *c, int32_t event_id, const void *depth, int32_t kind, void *ao_out, void *stream)
{
    if (!c) return MEAO_ERR_INVALID;
    std::lock_guard<std::mutex> g(g_event_mutex);
    if (!depth && !ao_out) { g_events.erase(event_id); return MEAO_OK; }
    g_events[event_id] = EventBinding{c, depth, kind, ao_out, stream};
    return MEAO_OK;
}

void meao_render_event(int event_id)
{
    EventBinding b;
    {
        std::lock_guard<std::mutex> g(g_event_mutex);
        auto it = g_events.find(event_id);
        if (it == g_events.end()) return;
        b = it->second;
    }
    meao_render(b.ctx, b.depth, b.kind, b.out, b.stream);
}

MeaoRenderEventFunc meao_get_render_event_func(void) { return meao_render_event; }

int64_t meao_launch_count(const MeaoCtx *c) { return c ? c->launches : 0; }
int meao_pdl_level(const MeaoCtx *c) { return c ? c->pdl_level : -1; }
int meao_kernels_per_frame(const MeaoCtx *c)
{
    if (c && c->variants.single_scale) return 3;      // Downsample1 + Render level 1 + the final-style Upsample
    int n = 9;
    if (c) for (int k = 1; k <= 4; k++) n += hq_level(c, k) ? 1 : 0;
    return n;
}

int64_t meao_algorithmic_bytes(const MeaoCtx *c, int32_t stage)
{
    if (!c || c->W <= 0) return MEAO_ERR_INVALID;
    auto px = [&](int l) { return (int64_t)c->lw[l] * c->lh[l]; };
    // SURVEY.md 8(d): every buffer of the reference data-flow read once per consuming stage, written once
    const int64_t ds1 = 6 * px(0) + 4 * px(1) + 4 * px(2) + 32 * px(3) + 32 * px(4);
    const int64_t ds2 = 4 * px(2) + 4 * px(3) + 4 * px(4) + 32 * px(5) + 32 * px(6);
    int64_t ren = 0, ups = 0, ups_final = 0;
    for (int k = 1; k <= 4; k++) ren += 32 * px(k + 2) + px(k);
    for (int lo = 4; lo >= 1; lo--) {
        const int hi = lo - 1;
        const int64_t b = 5 * px(lo) + (hi == 0 ? 2 : 5) * px(hi) + px(hi);
        ups += b;
        if (lo == 1) ups_final = b;
    }
    switch (stage) {
        case 0: return ds1 + ds2 + ren + ups;
        case 1: return ds1;
        case 2: return ds2;
        case 3: return ren;
        case 4: return ups;
        case 5: return ups_final;
        default: return MEAO_ERR_INVALID;
    }
}

int meao_selftest_div(MeaoCtx *c, uint64_t n, uint32_t seed, uint64_t *mismatches)
{
    int rc = ensure_ready(c); if (rc) return rc;
    if (!mismatches) return fail(c, MEAO_ERR_INVALID, "mismatches is NULL");
    unsigned long long *d = nullptr;
    CUDA_TRY(c, cudaMalloc(&d, sizeof *d));
    cudaError_t e = cudaMemsetAsync(d, 0, sizeof *d, c->stream);
    if (e == cudaSuccess) e = launch_selftest_div(n, seed, d, c->stream);
    unsigned long long h = 0;
    if (e == cudaSuccess) e = cudaMemcpyAsync(&h, d, sizeof h, cudaMemcpyDeviceToHost, c->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(c->stream);
    cudaFree(d);
    if (e != cudaSuccess) return fail(c, MEAO_ERR_CUDA, "selftest: %s", cudaGetErrorString(e));
    *mismatches = h;
    return MEAO_OK;
}

int meao_set_profile_repeats(MeaoCtx *c, int32_t n)
{
    if (!c || n < 1 || n > 1000) return MEAO_ERR_INVALID;
    c->profile_repeats = n;
    return MEAO_OK;
}

int meao_profile_frame(MeaoCtx *c, const void *depth, int32_t kind, void *ao_out, float *ms_out, const char **names_out, int32_t capacity)
{
    int rc = ensure_ready(c); if (rc) return rc;
    if (!depth || !ao_out) return fail(c, MEAO_ERR_INVALID, "depth / ao_out is NULL");
    CUDA_TRY(c, cudaDeviceSynchronize());
    if ((rc = record_frame(c, depth, kind, ao_out, c->stream, true))) return rc;
    const int n = (int)c->last_profile.size();
    for (int i = 0; i < n && i < capacity; i++) {
        if (ms_out) ms_out[i] = c->last_profile[i].second;
        if (names_out) names_out[i] = c->last_profile[i].first.c_str();
    }
    return n;
}

}  // extern "C"
