/*
 * meao.h -- C ABI of libmeao.so: the B200-native multi-scale SSAO pipeline that stands in for
 * the compute path of keijiro/MiniEngineAO's AmbientOcclusion component.
 *
 * The reference has no FFI seam: its boundary is the set of CommandBuffer calls
 * AmbientOcclusion.cs makes against four ComputeShader assets.  Each entry point below names
 * the reference interface it replaces (paths relative to /root/reference/Assets/MiniEngineAO/).
 * The C# P/Invoke binding a maintainer would add is host/AmbientOcclusionNative.cs and is
 * described in INTEGRATION.md.
 *
 * Conventions: plain C types only; every call returns 0 on success or a negative MeaoStatus;
 * meao_last_error() gives the text.  A context is owned by one thread at a time (the reference
 * records on Unity's main thread and replays on one render thread); distinct contexts are
 * independent.  The caller owns the depth input and the AO output memory; the context owns the
 * 16 intermediate buffers (LinearDepth, LowDepth1-4, Occlusion1-4, Combined1-3; the four
 * TiledDepth atlases are virtual, see DESIGN.md).
 * There is NO CPU fallback: every compute entry point fails with MEAO_ERR_CUDA when no
 * sm_100 device is usable.
 */
#ifndef MEAO_H
#define MEAO_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif
#if defined(__GNUC__)
#pragma GCC visibility push(default)
#endif

#define MEAO_ABI_VERSION 3   /* 2: + MeaoVariants, meao_stage_render_wide, meao_debug_view, meao_composite_debug, buffer ids 18..21
                              * 3: + MeaoVariants.single_scale, native peer halo exchange (meao_band_export / _connect / _step / _status),
                              *      meao_bind_event takes the stream;
                              *      later (backward compatible): batched frames (meao_reserve_batch / meao_render_batch / meao_get_batch_buffer) */

typedef struct MeaoCtx MeaoCtx;

typedef enum {
    MEAO_OK = 0,
    MEAO_ERR_INVALID = -1,      /* bad argument / call order */
    MEAO_ERR_CUDA = -2,         /* CUDA runtime or driver error, or no usable device */
    MEAO_ERR_UNSUPPORTED = -3,  /* e.g. halo deeper than the neighbouring band */
    MEAO_ERR_NOMEM = -4,
    MEAO_ERR_PEER = -5          /* native halo exchange: a neighbour did not arrive within the time-out (meao_band_status) */
} MeaoStatus;

/* AmbientOcclusion.cs:20-68 -- the serialized parameter surface, same names, ranges, defaults. */
typedef struct {
    float noise_filter_tolerance;   /* Range(-8, 0)    default 0      AO.cs:20-26 */
    float blur_tolerance;           /* Range(-8, -1)   default -4.6   AO.cs:28-34 */
    float upsample_tolerance;       /* Range(-12, -1)  default -12    AO.cs:36-42 */
    float thickness_modifier;       /* Range(1, 10)    default 1      AO.cs:44-50 */
    float intensity;                /* Range(0, 2)     default 1      AO.cs:52-58 */
    int32_t debug;                  /* Range(0, 17)    default 0      AO.cs:60    (carried; selects nothing on the compute path) */
    int32_t ambient_only;           /* default 1       AO.cs:62-68   (carried; composite is out of scope) */
} MeaoParams;

/* Camera inputs of the CPU-side constant math: AO.cs:561-573. */
typedef struct {
    float near_clip;        /* camera.nearClipPlane                         AO.cs:563 */
    float far_clip;         /* camera.farClipPlane                          AO.cs:563 */
    float tan_half_fov_h;   /* 1 / camera.projectionMatrix[0,0]             AO.cs:570-573 */
    int32_t reversed_z;     /* SystemInfo.usesReversedZBuffer (D3D11/12: 1) AO.cs:564, Downsample1.compute:41-45 */
} MeaoCamera;

typedef struct {
    int32_t device;         /* CUDA device ordinal; < 0 = host-side PLANNING context only (constants, geometry,
                               band / halo row ranges) -- every compute call on it fails with MEAO_ERR_CUDA */
    uint32_t flags;         /* MEAO_FLAG_* */
} MeaoDeviceCfg;

#define MEAO_FLAG_NONE        0u
#define MEAO_FLAG_NO_GRAPH    1u   /* launch the kernels on the stream instead of replaying the captured CUDA graph */

typedef enum {
    MEAO_DEPTH_RAW_F32 = 0,     /* camera depth, linearised by Downsample1.compute:37-48 (reference behaviour) */
    MEAO_DEPTH_LINEAR_F32 = 1,  /* already-linear depth (Linearize becomes the identity; not in the reference) */
    /* native depth-buffer formats (what Blit.shader pass 0 :48-64 samples; SURVEY.md 8f.1): the UNORM code is
     * converted with the D3D rule (float)code * (1 / (2^n - 1)) and then linearised like RAW_F32 */
    MEAO_DEPTH_RAW_D16_UNORM = 2,   /* uint16 codes, 2 bytes / pixel */
    MEAO_DEPTH_RAW_D24S8 = 3        /* uint32 words, depth in the low 24 bits (D24_UNORM_S8_UINT), stencil ignored */
} MeaoDepthKind;

/* Debug buffer ids, numbering of AmbientOcclusion.cs:787-808. */
typedef enum {
    MEAO_BUF_LINEAR_DEPTH = 1,                                  /* L0, f16 */
    MEAO_BUF_LOW_DEPTH1 = 2, MEAO_BUF_LOW_DEPTH2 = 3,           /* L1..L4, f32 */
    MEAO_BUF_LOW_DEPTH3 = 4, MEAO_BUF_LOW_DEPTH4 = 5,
    MEAO_BUF_TILED_DEPTH1 = 6, MEAO_BUF_TILED_DEPTH2 = 7,       /* L3..L6 x 16 slices, f16 */
    MEAO_BUF_TILED_DEPTH3 = 8, MEAO_BUF_TILED_DEPTH4 = 9,
    MEAO_BUF_OCCLUSION1 = 10, MEAO_BUF_OCCLUSION2 = 11,         /* L1..L4, unorm8 */
    MEAO_BUF_OCCLUSION3 = 12, MEAO_BUF_OCCLUSION4 = 13,
    MEAO_BUF_COMBINED1 = 14, MEAO_BUF_COMBINED2 = 15, MEAO_BUF_COMBINED3 = 16,   /* L1..L3, unorm8 */
    MEAO_BUF_AMBIENT_OCCLUSION = 17,                            /* L0, unorm8 */
    /* extension ids (not in AO.cs:787-808): output of Render.compute kernel "main" (MeaoVariants.high_quality_mask) */
    MEAO_BUF_HIGH_QUALITY1 = 18, MEAO_BUF_HIGH_QUALITY2 = 19,   /* L1..L4, unorm8 */
    MEAO_BUF_HIGH_QUALITY3 = 20, MEAO_BUF_HIGH_QUALITY4 = 21
} MeaoBufferId;

typedef struct {
    int32_t width, height, slices;  /* reference texture dimensions (AO.cs:276-281; slices = 16 when tiled, AO.cs:154) */
    int32_t elem_bytes;             /* 1 = unorm8, 2 = f16 bits, 4 = f32  (AO.cs:262-273) */
} MeaoBufferDesc;

/* Shader / host variants that the reference SHIPS but never selects (SURVEY.md 8f.2, 8f.4).  All zero = exactly what
 * AmbientOcclusion.cs records; every field is a plan input like MeaoParams (a change re-plans, AO.cs:334-347). */
typedef struct {
    int32_t single_pass_stereo;   /* singlePassStereoEnabled (AO.cs:392-401): ThicknessMultiplier *= 2 (AO.cs:680).  The caller passes the
                                     DOUBLE-WIDE eye pair to meao_resize, as LateUpdate / RebuildCommandBuffers do (AO.cs:338-341, 501-504). */
    int32_t sample_exhaustively;  /* Render.compute:144-159 "#define SAMPLE_EXHAUSTIVELY": 68 taps instead of the 36-tap checker, and the
                                     weight zeroing of AO.cs:709-715 ("FIXME: should we support SAMPLE_EXHAUSTIVELY mode?") is skipped */
    int32_t high_quality_mask;    /* bit k-1 (k = 1..4): level k ALSO runs Render.compute kernel "main" (WIDE_SAMPLING, :22,27-29,46-50,79-82:
                                     non-tiled source LowDepth<k>, so PushRenderCommands takes the "!source.isTiled" branch AO.cs:679) into
                                     HighQuality<k>, and the upsample whose LOW level is k runs Upsample.compute kernel "main_premin" /
                                     "main_premin_blendout" (:23,25,32-34,58-60) with LoResAO2 = HighQuality<k>.  E.g. 8 = coarsest level
                                     only, 15 = every level (the quality ladder of the upstream MiniEngine sample, which is not vendored). */
    int32_t single_scale;         /* BASELINE.json configs[0] "single-scale AO": the frame is Downsample1 -> Render level 1 -> the FINAL-style
                                     Upsample (kernel "main", AO.cs:531's dispatch with LoResAO1 = Occlusion1 instead of Combined1): three of
                                     the ten dispatches of AO.cs:511-531, no coarser level contributes.  Requires high_quality_mask == 0. */
} MeaoVariants;

/* ---- lifetime ------------------------------------------------------------------------------ */
/* replaces: component construction + DoLazyInitialization (AO.cs:440-494). */
int meao_create(const MeaoDeviceCfg *cfg, MeaoCtx **out_ctx);
/* replaces: OnDestroy (AO.cs:357-381). */
void meao_destroy(MeaoCtx *ctx);
const char *meao_last_error(const MeaoCtx *ctx);   /* ctx may be NULL: error of the last failed meao_create on this thread */
int meao_abi_version(void);

/* ---- parameters (plan inputs) ---------------------------------------------------------------- */
/* replaces: the property setters AO.cs:22-66.  Marks the plan dirty iff a value changed
 * (CheckPropertiesChanged, AO.cs:104-113); returns 1 if the plan was dirtied, 0 if not. */
int meao_set_params(MeaoCtx *ctx, const MeaoParams *params);
int meao_get_params(const MeaoCtx *ctx, MeaoParams *out);
void meao_default_params(MeaoParams *out);          /* AO.cs:20-68 defaults */
/* Selects the undispatched shader variants above; returns 1 if the plan was dirtied, 0 if not. */
int meao_set_variants(MeaoCtx *ctx, const MeaoVariants *variants);
int meao_get_variants(const MeaoCtx *ctx, MeaoVariants *out);
/* replaces: CalculateZBufferParams / CalculateTanHalfFovHeight inputs (AO.cs:561-573). */
int meao_set_camera(MeaoCtx *ctx, const MeaoCamera *camera);
/* replaces: RTHandle.SetBaseDimensions + AllocateNow + the rebuild it triggers (AO.cs:338-341, 501-506).
 * Allocates the intermediates for width x height.  Returns 1 if dimensions changed, 0 if not.
 * A size change RESETS the row band to the whole frame and drops the neighbour connections (meao_set_row_band,
 * meao_band_connect): a band host must set its band again after every call that returned 1. */
int meao_resize(MeaoCtx *ctx, int32_t width, int32_t height);

/* ---- the frame ------------------------------------------------------------------------------- */
/* replaces: replay of the "SSAO" command buffer, steps 1-10 of RebuildCommandBuffers (AO.cs:511-531):
 * Downsample1+2, Render x4, Upsample x4.  depth: device pointer, width*height f32, rows contiguous
 * (row pitch = width*4).  ao_out: device pointer, width*height bytes (R8, AO.cs:475).
 * stream: a cudaStream_t, used as given (NULL = the CUDA legacy default stream).  Asynchronous.  Re-plans first if dirty
 * (LateUpdate, AO.cs:329-350). */
int meao_render(MeaoCtx *ctx, const void *depth_dev, int32_t depth_kind, void *ao_out_dev, void *stream);
/* Same with HOST buffers: H2D copy of depth, the ten passes, D2H copy of the AO texture, then a
 * stream synchronise.  Use meao_host_alloc for pinned memory. */
int meao_render_host(MeaoCtx *ctx, const void *depth_host, int32_t depth_kind, uint8_t *ao_out_host);
/* Pipelined form of meao_render_host for frame streams: enqueues H2D + kernels + D2H of one frame on staging slot
 * `slot` (0 or 1) and returns; meao_host_wait(slot) blocks until that frame's AO is in ao_out_host.  Alternating the
 * two slots overlaps the H2D copy of frame i+1 with the kernels and the D2H copy of frame i (the kernels of
 * consecutive frames stay serialised: they share the context's intermediates).  Host buffers must be pinned
 * (meao_host_alloc) for the copies to be asynchronous, and must stay valid until the matching wait. */
int meao_render_host_async(MeaoCtx *ctx, const void *depth_host, int32_t depth_kind, uint8_t *ao_out_host, int32_t slot);
int meao_host_wait(MeaoCtx *ctx, int32_t slot);

/* ---- batched frames ---------------------------------------------------------------------------- */
/* Batched frames: `frames` independent frames of the size set by meao_resize, stacked tightly:
 * frame f of depth_dev starts at element f*W*H, frame f of ao_out_dev at byte f*W*H (R8).
 * Every frame gives exactly what meao_render gives for it.  With graphs on, a batch is ONE graph replay (the DAG of a frame, every
 * kernel covering all frames); MEAO_FLAG_NO_GRAPH issues the same launches directly.  Re-plans first if dirty, like meao_render.
 * The intermediates of a batch live in a batch arena of their own: meao_get_buffer, meao_debug_view, the stage and band calls
 * do not see a batch.  meao_resize and meao_destroy free it.
 * meao_render_batch grows the arena on demand; growing is a synchronous allocation (device synchronise + cudaMalloc), so
 * reserve the largest batch with meao_reserve_batch outside any timed region.
 * MEAO_ERR_INVALID: frames < 1 or > 65535, NULL pointers, bad depth kind.  MEAO_ERR_UNSUPPORTED: a row band is set.
 * MEAO_ERR_CUDA: plan-only context.  meao_launch_count grows by meao_kernels_per_frame per batch. */
int meao_reserve_batch(MeaoCtx *ctx, int32_t frames);   /* allocate batch intermediates for >= frames (optional; render_batch grows on demand) */
int meao_render_batch(MeaoCtx *ctx, const void *depth_dev, int32_t depth_kind, int32_t frames, void *ao_out_dev, void *stream);
/* Buffer ids 1-16 and 18-21 of frame `frame` of the last batch, in the layout of meao_get_buffer (TiledDepth synthesised the
 * same way; synchronises the device).  Id 17 is refused: the AO of a batch is in the caller's buffer. */
int meao_get_batch_buffer(MeaoCtx *ctx, int32_t frame, int32_t buffer_id, void *host_out, size_t host_bytes);
int meao_synchronize(MeaoCtx *ctx);
void *meao_host_alloc(size_t bytes);                /* cudaHostAlloc; NULL on failure */
void meao_host_free(void *p);

/* ---- per-stage entry points (stage parity; mirror the three Push*Commands recorders) ----------- */
/* replaces: PushDownsampleCommands (AO.cs:604-658) -> LinearDepth, LowDepth1..4 (+ virtual TiledDepth1..4) */
int meao_stage_downsample(MeaoCtx *ctx, const void *depth_dev, int32_t depth_kind, void *stream);
/* replaces: PushRenderCommands (AO.cs:660-748) for TiledDepth<level> -> Occlusion<level>, level 1..4 */
int meao_stage_render(MeaoCtx *ctx, int32_t level, void *stream);
/* PushRenderCommands (AO.cs:660-748) for a NON-tiled source: LowDepth<level> -> HighQuality<level> with Render.compute kernel
 * "main" (FindKernel would name it instead of "main_interleaved", AO.cs:728; thread-group size 16x16 from AO.cs:739-747). */
int meao_stage_render_wide(MeaoCtx *ctx, int32_t level, void *stream);
/* replaces: PushUpsampleCommands (AO.cs:750-785) with the wiring of AO.cs:528-531; lo_level 4..1.
 * lo_level == 1 writes the final AO into ao_out_dev (or the context's own result buffer if NULL).
 * Uses the main_premin variants for the levels selected in MeaoVariants.high_quality_mask. */
int meao_stage_upsample(MeaoCtx *ctx, int32_t lo_level, void *ao_out_dev, void *stream);

/* ---- buffers (debug views, AO.cs:787-820) ------------------------------------------------------ */
int meao_buffer_desc(const MeaoCtx *ctx, int32_t buffer_id, MeaoBufferDesc *out);
/* Copies buffer <id> to host in the REFERENCE layout (tightly packed rows; tiled = [16][h][w]) and
 * native storage type (f16 bits / f32 / unorm8 codes).  Synchronises the context stream.
 * The TiledDepth views are synthesised from LowDepth<k> exactly as Downsample1/2 would have
 * written them (including the padding texels, SURVEY.md P3). */
int meao_get_buffer(MeaoCtx *ctx, int32_t buffer_id, void *host_out, size_t host_bytes);
/* Test hook: overwrite an intermediate (ids 1-5, 10-21) from host data in the same format. */
int meao_set_buffer(MeaoCtx *ctx, int32_t buffer_id, const void *host_in, size_t host_bytes);
/* replaces: PushDebugBlitCommands (AO.cs:787-820) + the debug composite, Blit.shader pass 3 (:116-134): writes the
 * width x height R8 image that _result holds after the debug blit of buffer <buffer_id> (1..17, the `debug` property
 * AO.cs:60; 18..21 for the HighQuality extension) into out_r8_dev (tight rows).  Non-tiled sources: cmd.Blit(rt, _result),
 * a point-sampled stretch (texel = floor(uv * size) at the pixel centre); TiledDepth1..4: Blit.shader pass 4 "Detile"
 * (:136-156), a 4 x 4 mosaic of the 16 slices; 17: the AO texture itself.  Asynchronous on `stream`. */
int meao_debug_view(MeaoCtx *ctx, int32_t buffer_id, void *out_r8_dev, void *stream);

/* ---- CPU-side constants, exposed so they can be checked against the reference math ------------- */
/* out[0..11] gInvThicknessTable, out[12..23] gSampleWeightTable, out[24..25] gInvSliceDimension,
 * out[26] gRejectFadeoff, out[27] gIntensity            (AO.cs:678-734) */
int meao_render_constants(MeaoCtx *ctx, int32_t level, float out28[28]);
/* same layout for the non-tiled dispatch of meao_stage_render_wide (source = LowDepth<level>, AO.cs:679 applied) */
int meao_render_constants_wide(MeaoCtx *ctx, int32_t level, float out28[28]);
/* out[0..1] InvLowResolution, out[2..3] InvHighResolution, out[4] NoiseFilterStrength, out[5] StepSize,
 * out[6] kBlurTolerance, out[7] kUpsampleTolerance       (AO.cs:760-771) */
int meao_upsample_constants(MeaoCtx *ctx, int32_t lo_level, float out8[8]);
/* out[0..3] ZBufferParams (AO.cs:561-568) */
int meao_zbuffer_params(MeaoCtx *ctx, float out4[4]);

/* ---- row-band partitioning of one frame over several GPUs (new capability, SURVEY.md 8e) -------- */
/* This context computes output rows [row0, row1) of the width x height frame set by meao_resize
 * (global coordinates everywhere; image-edge semantics only at the true top/bottom).
 * row0/row1 must be multiples of 16 except row1 == height.  prev_row0 / next_row1 give the extent
 * of the bands above and below (-1 = none).  depth passed to render/stage_downsample is then the
 * BAND's rows only (row1-row0 rows), and ao_out receives the band's rows only. */
int meao_set_row_band(MeaoCtx *ctx, int32_t row0, int32_t row1, int32_t prev_row0, int32_t next_row1);
/* Border rows of LowDepth1..4 that a neighbour needs.  side: 0 = towards row 0 (up), 1 = down.
 * meao_halo_bytes: size of the packed message this context SENDS to that side (== what the
 * neighbour's unpack of the opposite side expects). */
int64_t meao_halo_bytes(MeaoCtx *ctx, int32_t side);
int64_t meao_halo_recv_bytes(MeaoCtx *ctx, int32_t side);
/* Row ranges behind those sizes: out8 = {lo1,hi1, lo2,hi2, lo3,hi3, lo4,hi4} rows of LowDepth1..4 that
 * are sent (send != 0) / received (send == 0) on that side; the packed message is those rows, level 1
 * first, each row lw[k] tightly packed f32. */
int meao_halo_rows(MeaoCtx *ctx, int32_t side, int32_t send, int32_t out8[8]);
/* out30 = for k = 0..4: rows of level k to produce [2k,2k+1]; rows of LowDepth<k> read [10+2k..];
 * rows of LowDepth<k> this band owns [20+2k..]. */
int meao_band_rows(MeaoCtx *ctx, int32_t out30[30]);
int meao_halo_pack(MeaoCtx *ctx, int32_t side, void *packed_dev, void *stream);
int meao_halo_unpack(MeaoCtx *ctx, int32_t side, const void *packed_dev, void *stream);
/* Split of meao_render around the exchange: phase A = downsample own rows; (exchange); phase B =
 * render + upsample. */
int meao_render_band_prepare(MeaoCtx *ctx, const void *depth_band_dev, int32_t depth_kind, void *stream);
int meao_render_band_finish(MeaoCtx *ctx, void *ao_band_out_dev, void *stream);

/* The same split with the halo pack / unpack fused in and each half replayed as ONE CUDA graph:
 *   phase A = prepare_depth on the band + pack of both outgoing halos (send_* may be NULL at the frame edge);
 *   phase B = unpack of both incoming halos + Render x4 + Upsample x4.
 * A band step is then: phase A, one neighbour send/recv per side (NCCL or peer copy), phase B. */
int meao_band_phase_a(MeaoCtx *ctx, const void *depth_band_dev, int32_t depth_kind, void *send_up_dev, void *send_down_dev, void *stream);
int meao_band_phase_b(MeaoCtx *ctx, const void *recv_up_dev, const void *recv_down_dev, void *ao_band_out_dev, void *stream);

/* ---- native neighbour exchange (ABI 3): the halo rows travel by PEER STORES over NVLink, inside the frame's one CUDA graph ----
 * Every band context keeps its LowDepth1..4 in full-frame global coordinates, so a band's border rows have the SAME byte offset
 * in every context's arena: the exchange kernel (csrc/band_exchange.cu) writes them straight into the neighbour's LowDepth
 * buffers through a peer mapping -- no pack, no staging, no unpack, no NCCL call -- then raises an epoch flag in the neighbour's
 * memory (st.release.sys) and waits for the neighbour's own flag (ld.acquire.sys).  A step of a connected band is ONE graph
 * launch: prepare_depth -> exchange -> Render x4 + Upsample x4 (DAG), no host code between the phases.
 *   1. meao_resize + meao_set_row_band on every band context (one per GPU; same or different processes)
 *   2. meao_band_export -> an opaque POD handle; move it to the neighbours any way the host likes (memcpy in-process;
 *      torch.distributed / MPI / a pipe between processes -- it contains a cudaIpcMemHandle_t)
 *   3. meao_band_connect(ctx, side, &neighbour_handle) for each existing neighbour (side 0 = up, 1 = down)
 *   4. per frame, on every band in lock step: meao_band_step (asynchronous on `stream`)
 * All bands must run the same number of steps.  A wait that exceeds the time-out (default 2 s, env MEAO_BAND_TIMEOUT_MS)
 * sets a sticky error instead of hanging the GPU: the remaining kernels of that step still run (on stale halo rows),
 * meao_band_status reports it and the next meao_band_step fails with MEAO_ERR_PEER.
 * meao_resize and meao_set_row_band DISCONNECT (the arena / the halo ranges change): export + connect again afterwards.
 * Scheduling contract.  The exchange kernel spins on flags its NEIGHBOUR raises, so the neighbour's kernels must be able to run
 * while it waits.  With one band per GPU that is automatic as long as every host issues the steps of its band contexts in the same
 * order (frame streams over several contexts per GPU are fine: bench.py runs 12).  When NEIGHBOURING bands share one GPU (tests,
 * single-GPU development) every band's streams need their own hardware queue: set CUDA_DEVICE_MAX_CONNECTIONS=32 before CUDA starts
 * and keep to <= 3 bands per GPU -- otherwise a band's kernels (or its first graph instantiation) can end up waiting behind the
 * spinning kernel that waits for them, which the time-out then reports as error 1 / 2 (DESIGN.md section 4). */
#define MEAO_PEER_HANDLE_BYTES 128
typedef struct { unsigned char bytes[MEAO_PEER_HANDLE_BYTES]; } MeaoPeerHandle;
int meao_band_export(MeaoCtx *ctx, MeaoPeerHandle *out);
/* peer == NULL disconnects that side.  Same process: direct pointer (+ cudaDeviceEnablePeerAccess across devices);
 * another process: cudaIpcOpenMemHandle.  Fails with MEAO_ERR_INVALID if the neighbour's frame size differs.
 * The bands' epoch counters run in lock step from 1, so a band that has already stepped can only be reconnected as a whole:
 * disconnect both of its sides (and do the same on every other band of the frame), then connect again -- the first connect of a
 * fully disconnected band restarts its epoch and clears a sticky time-out error. */
int meao_band_connect(MeaoCtx *ctx, int32_t side, const MeaoPeerHandle *peer);
int meao_band_step(MeaoCtx *ctx, const void *depth_band_dev, int32_t depth_kind, void *ao_band_out_dev, void *stream);
/* The same with HOST buffers (the band's rows only): H2D copy, the step, D2H copy, all enqueued on the context's staging slot 0 --
 * asynchronous, because the neighbours' steps must be enqueued too before anyone waits; then meao_host_wait(ctx, 0) on every band.
 * The host buffers MUST be pinned (meao_host_alloc): a pageable copy blocks the calling thread until it has completed, which it
 * cannot before the neighbour -- not yet enqueued by that same thread -- has taken part in the exchange.
 * This is what lets a single-threaded C / C# host drive all GPUs of a box (tests/c_abi/smoke.c "bands"). */
int meao_band_step_host(MeaoCtx *ctx, const void *depth_band_host, int32_t depth_kind, uint8_t *ao_band_out_host);
/* out4 = { epoch of the next exchange (1 + completed exchanges), sticky error (0 ok, 1 = time-out waiting for a neighbour's
 * ack, 2 = time-out waiting for a neighbour's rows), connected-up, connected-down }.  Synchronises nothing: reads the
 * flags with a stream-less copy, so call it after the stream has drained for a definitive answer. */
int meao_band_status(MeaoCtx *ctx, int32_t out4[4]);

/* ---- composite: the consumer end of the pipe (SURVEY.md 8f.1) ------------------------------------------- */
typedef enum {
    MEAO_FMT_RGBA8_UNORM = 0,   /* ARGB32-class LDR target, 4 bytes / pixel */
    MEAO_FMT_RGBA16_FLOAT = 1   /* ARGBHalf HDR target, 8 bytes / pixel */
} MeaoColorFormat;
/* replaces: PushCompositeCommands, frame-buffer branch (AO.cs:835-838) = Blit.shader pass 2 (:84-101),
 * "Blend Zero SrcAlpha" with src = ao.rrrr:   color.rgba *= ao.   ao_dev: width*height R8 codes (tight rows, what
 * meao_render wrote); color_dev: width*height pixels, tight rows, updated in place.  16-byte aligned pointers. */
int meao_composite_framebuffer(MeaoCtx *ctx, const void *ao_dev, void *color_dev, int32_t color_format, void *stream);
/* replaces: PushCompositeCommands, ambient-only deferred branch (AO.cs:830-834) = Blit.shader pass 1 (:66-92),
 * "Blend Zero OneMinusSrcColor, Zero OneMinusSrcAlpha" with src0 = (0,0,0,1-ao), src1 = (1-ao,1-ao,1-ao,0):
 *   gbuffer0.a *= 1-(1-ao)  (RGBA8, occlusion channel),  gbuffer3.rgb *= 1-(1-ao)  (ambient/emission target). */
int meao_composite_gbuffer(MeaoCtx *ctx, const void *ao_dev, void *gbuffer0_rgba8_dev, void *gbuffer3_dev, int32_t gbuffer3_format, void *stream);
/* replaces: PushCompositeCommands, debug branch (AO.cs:826-829) = Blit.shader pass 3 "Debug" (:116-134), no blending:
 *   color.rgba = view.rrrr   where view_r8_dev is the width*height R8 image written by meao_debug_view (or the AO texture). */
int meao_composite_debug(MeaoCtx *ctx, const void *view_r8_dev, void *color_dev, int32_t color_format, void *stream);

/* ---- command-buffer hook (Unity native-plugin style) -------------------------------------------- */
/* replaces: camera.AddCommandBuffer(..., _renderCommand) (AO.cs:412-429): a host engine issues
 * CommandBuffer.IssuePluginEvent(meao_get_render_event_func(), event_id). */
typedef void (*MeaoRenderEventFunc)(int event_id);
/* stream: the cudaStream_t the plugin event renders on (ABI 3; NULL = the CUDA legacy default stream, as before). */
int meao_bind_event(MeaoCtx *ctx, int32_t event_id, const void *depth_dev, int32_t depth_kind, void *ao_out_dev, void *stream);
void meao_render_event(int event_id);
MeaoRenderEventFunc meao_get_render_event_func(void);

/* ---- introspection ------------------------------------------------------------------------------ */
int64_t meao_launch_count(const MeaoCtx *ctx);       /* kernels launched (or replayed via graph) so far */
/* Programmatic-dependent-launch level of the captured frame graphs: -1 = nothing captured yet, 0 = plain edges, 1 = PDL on the
 * kernels whose only predecessor is the kernel before them in their stream, 2 = also where a cross-branch event joins.  The runtime
 * decides what it accepts at the first capture; env MEAO_PDL=0|1|2 caps it. */
int meao_pdl_level(const MeaoCtx *ctx);
int meao_kernels_per_frame(const MeaoCtx *ctx);      /* kernel nodes in one frame: 9 + one per bit of high_quality_mask (3 with single_scale) */
/* Algorithmic bytes of the reference data-flow (SURVEY.md 8d): stage 0 = whole frame, 1 = Downsample1,
 * 2 = Downsample2, 3 = Render x4, 4 = Upsample x4, 5 = final Upsample (L1->L0) only. */
int64_t meao_algorithmic_bytes(const MeaoCtx *ctx, int32_t stage);
/* Device time (ms) of the individual kernels of the last meao_profile_frame() call, which runs one
 * frame with a cudaEvent pair around every kernel.  names/ms arrays of length >= meao_kernels_per_frame(). */
int meao_profile_frame(MeaoCtx *ctx, const void *depth_dev, int32_t depth_kind, void *ao_out_dev,
                       float *ms_out, const char **names_out, int32_t capacity);
/* Launches per kernel inside meao_profile_frame's event pairs (default 1).  With n > 1 every kernel is launched n times back to back
 * (all of them are idempotent: out of place, inputs untouched) and the reported time is the mean -- the event pair's own overhead and
 * the launch gap are amortised, which is what a roofline figure of ONE kernel wants. */
int meao_set_profile_repeats(MeaoCtx *ctx, int32_t n);

/* Device self test: compares the guarded fast division / reciprocal the kernels use (MUFU.RCP + FMA
 * refinement, csrc/common.cuh) with the IEEE operators on n random operand pairs; *mismatches must be 0. */
int meao_selftest_div(MeaoCtx *ctx, uint64_t n, uint32_t seed, uint64_t *mismatches);

#if defined(__GNUC__)
#pragma GCC visibility pop
#endif
#ifdef __cplusplus
}
#endif
#endif /* MEAO_H */
