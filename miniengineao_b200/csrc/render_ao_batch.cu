// render_ao_batch.cu -- the batched render kernels (meao_render_batch) and their launcher.
//
// render_ao.cu compiled again with MEAO_REN_BATCH = 1, which selects the batch pass of render_ao_kernel.inc and
// launch_render_ao_batch instead of the single-frame kernels.  A translation unit of its own, like blur_upsample_batch.cu:
// the single-frame kernels are compiled exactly as without batching, and a build of the kernel sources that leaves this file
// out (the host emulator of the single-frame path) needs no 3-D TMA.
#define MEAO_REN_BATCH 1
#include "render_ao.cu"
