// cuda_emu_3d.h -- cp.async.bulk.tensor.3d for the host emulator of tests/emu (TEST INFRASTRUCTURE ONLY, see ../emu/cuda_emu.h).
//
// Force-included (g++ -include) into every translation unit of tests/emu_batch/libmeao_emu_batch.so, the emulator build that
// also compiles the batched kernels (meao_render_batch).  A 3-D map is the emulator's 2-D CUtensorMap with the third dimension
// in its spare words: pad_[0] = number of frames (0 = a 2-D map), pad_[1] = bytes between frames; the box depth is 1.
#pragma once

#include "../emu/cuda_emu.h"

#define MEAO_EMU_TMA_3D 1

namespace meao_emu {
inline int map_frames(const CUtensorMap *m) { return (int)m->pad_[0]; }
inline size_t map_frame_bytes(const CUtensorMap *m) { return (size_t)m->pad_[1]; }
// the box of frame z, (x, y) its first element; out-of-bounds elements (any dimension) are zero-filled.  Same refusals as the
// 2-D load, plus the global-stride rule of cuTensorMapEncodeTiled (strides are multiples of 16 bytes).
inline void tma_load_3d(void *dst, const CUtensorMap *m, int x, int y, int z)
{
    if (map_frames(m) == 0) unsupported("3-D TMA load through a 2-D tensor map");
    if (((long long)x * m->elem) % 16 != 0) unsupported("TMA start coordinate not 16-byte aligned (faults on B200)");
    if (((uintptr_t)dst) % 128 != 0) unsupported("TMA shared-memory destination not 128-byte aligned (misaligned-address fault on B200)");
    if (map_frame_bytes(m) % 16 != 0) unsupported("TMA global stride not a multiple of 16 bytes");
    tma_box_loads++;
    for (int by = 0; by < m->bh; by++)
        for (int bx = 0; bx < m->bw; bx++) {
            char *d = (char *)dst + ((size_t)by * m->bw + bx) * m->elem;
            const int sx = x + bx, sy = y + by;
            if (sx >= 0 && sy >= 0 && sx < m->w && sy < m->h && z >= 0 && z < map_frames(m))
                memcpy(d, (const char *)m->base + (size_t)z * map_frame_bytes(m) + (size_t)sy * m->pitch_bytes + (size_t)sx * m->elem, m->elem);
            else memset(d, 0, m->elem);
        }
}
}  // namespace meao_emu
