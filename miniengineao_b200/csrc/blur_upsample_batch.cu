// blur_upsample_batch.cu -- the batched blur + bilateral-upsample kernels (meao_render_batch) and their launcher.
//
// blur_upsample.cu compiled again with MEAO_UPS_BATCH = 1, which selects the batch pass of blur_upsample_kernel.inc and
// launch_blur_upsample_batch instead of the single-frame kernels.  A translation unit of their own on purpose: compiled next
// to the batched kernels, the single-frame kernels of blur_upsample.cu came out of the compiler with different register
// assignments; apart, their SASS is byte-identical to the build without batching.
#define MEAO_UPS_BATCH 1
#include "blur_upsample.cu"
