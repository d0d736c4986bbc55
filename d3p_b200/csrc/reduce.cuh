// CTA-wide reductions shared by the clip kernels (clip.cu) and the AutoDiagonalNormal step (autodiag.cu).
#pragma once
#include "common.cuh"

namespace d3p {

// Sum of v over the CTA (every thread receives it); smem holds >= 32 floats.  Fixed order: warp shuffles, then warp 0
// over the per-warp sums.
D3P_D float block_sum(float v, float* smem /* >= 32 floats */) {
  v = group_sum<32>(v);
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  __syncthreads();
  if (lane == 0) smem[warp] = v;
  __syncthreads();
  float t = (threadIdx.x < (blockDim.x >> 5)) ? smem[threadIdx.x] : 0.f;
  if (warp == 0) {
    t = group_sum<32>(t);
    if (lane == 0) smem[0] = t;
  }
  __syncthreads();
  return smem[0];
}

// clip factor exactly as clip_gradient: 1 / max(1, norm / C)
D3P_D float clip_factor(float norm, float C) { return 1.0f / fmaxf(1.0f, norm / C); }

}  // namespace d3p
