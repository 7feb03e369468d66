// rt_render_fast.cu — the opt-in fast copies of the bounce-stage kernels (RT_GPU_Options.fast_math).
//
// The same source as the parity path (rt_stages.cuh), compiled with FMA contraction (-fmad=true) and RT_FAST=1:
// products and sums fuse (the bounce trace's 129 FMUL + 126 FADD become FFMA), the sRGB decode, sin/cos, atan2 and asin
// come from the SFU / CUDA's f32 library instead of rt_math.h's binary64 evaluation, and the reference's f64 promotions
// are f32.  The PRIMARY trace is never taken from here: primary-hit triangle ids stay the exact kernel's
// (north star: "primary-hit triangle IDs must be bit-exact"), and so do ray generation, accumulate and the film.
// What changes is the radiance of individual samples — by rounding, and wholesale when a rounding flips a lobe pick or a
// grazing hit; bench.py --fast reports how far the 1024-spp frame moves (parity key) next to the speed-up.
#define RT_FAST 1
#include "rt_stages.cuh"
#include "rt_kernels.h"

void rt_fast_launch_trace(const StageParams &P, unsigned grid, size_t smem, cudaStream_t stream, bool wide) {
  if (wide) rt_trace_kernel_fast<false, RT_TRACE_MIN_BLOCKS_WIDE><<<grid, RT_BLOCK, smem, stream>>>(P);
  else      rt_trace_kernel_fast<false><<<grid, RT_BLOCK, smem, stream>>>(P);
}

void rt_fast_launch_miss(const StageParams &P, unsigned grid, cudaStream_t stream) {
  rt_miss_kernel_fast<<<grid, 256, 0, stream>>>(P);
}

void rt_fast_launch_shade(const StageParams &P, unsigned grid, cudaStream_t stream) {
  rt_shade_kernel_fast<<<grid, 256, 0, stream>>>(P);
}

void rt_fast_launch_sky(const StageParams &P, unsigned grid, cudaStream_t stream) {
  rt_sky_kernel_fast<<<grid, 256, 0, stream>>>(P);
}

int rt_fast_trace_setup(size_t level_bytes, int *wide_blocks_per_sm) {
  *wide_blocks_per_sm = level_store_blocks_per_sm((const void *)rt_trace_kernel_fast<false, RT_TRACE_MIN_BLOCKS_WIDE>, level_bytes);
  return level_store_blocks_per_sm((const void *)rt_trace_kernel_fast<false>, level_bytes);
}
