// emu_batch_driver.cpp -- runs a batch of frames through the HOST-compiled batched kernel sources (TEST INFRASTRUCTURE ONLY,
// see ../emu/cuda_emu.h and cuda_emu_3d.h).  It is the single-frame driver of tests/emu (included whole: the same context,
// constants, recorders and buffer read-back), driven over a batch arena the way meao_render_batch drives libmeao's.
#include "../emu/emu_driver.cpp"

namespace {

// The batch arena: `frames` frame slots (SlotLayout) and its own persistent-loop counters.  Kept until the next batch.
struct EmuBatch {
    char *base = nullptr;
    int frames = 0;
    size_t slot_bytes = 0;
    FrameBufs bufs;                     // slot 0
    uint32_t tile_ctr[8] = {0};
};
EmuBatch g_batch;

}  // namespace

extern "C" {

// `frames` frames stacked tightly in depth (16-byte aligned) -> out (frames x W x H codes), in record_frame order
void emu_run_batch(void *h, const void *depth, int in_format, int frames, uint8_t *out)
{
    Emu *e = (Emu *)h;
    free(g_batch.base);
    g_batch = EmuBatch{};
    const SlotLayout s = slot_layout(e->g);
    g_batch.base = alloc<char>(s.slot_bytes * frames);
    g_batch.frames = frames; g_batch.slot_bytes = s.slot_bytes;
    g_batch.bufs = frame_bufs(g_batch.base, s);
    const BatchRun run{frames, (long long)e->g.W * e->g.H * depth_elem_bytes(in_format), (long long)s.slot_bytes};
    const EmuArena ar{g_batch.bufs, g_batch.tile_ctr, &run};
    run_downsample(e, ar, depth, in_format);
    run_renders_upsamples(e, ar, out);
    for (uint32_t c : g_batch.tile_ctr) if (c != 0) abort();      // the last CTA of every persistent launch re-armed its counters
}

// buffer <id> (1..16, 18..21) of frame <frame> of the last batch, like emu_get_buffer
int emu_get_batch_buffer(void *h, int frame, int id, void *out)
{
    Emu *e = (Emu *)h;
    BufferView v;
    if (frame < 0 || frame >= g_batch.frames || id == MEAO_BUF_AMBIENT_OCCLUSION || !buffer_view(e->g, g_batch.bufs, nullptr, id, &v)) return -1;
    v.ptr = (char *)v.ptr + (size_t)frame * g_batch.slot_bytes;
    read_view(e, v, out);
    return 0;
}

}  // extern "C"
