// prepare_depth_batch.cu -- the batched prepare_depth kernels (meao_render_batch) and their launcher.
//
// prepare_depth.cu compiled again with MEAO_PREP_BATCH = 1, which selects the batch pass of prepare_depth_kernel.inc and
// launch_prepare_depth_batch instead of the single-frame kernels (a translation unit of its own, like blur_upsample_batch.cu).
#define MEAO_PREP_BATCH 1
#include "prepare_depth.cu"
