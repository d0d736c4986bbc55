// K6: per-example clipping of materialised [B, P] gradients and the fused clip + sum.
// Replace full_norm / clip_gradient (d3p/svi.py:68-124), DPSVI._clip_gradients (:310-325) and
// DPSVI._combine_gradients (:327-348) for arbitrary models whose per-example gradients the
// caller already holds (the path the reference's own tests drive, tests/test_dpsvi.py:146-191).
#include "common.cuh"
#include "launch.cuh"
#include "reduce.cuh"

namespace d3p {

constexpr int kClipThreads = 256;

D3P_D float row_sq_norm(const float* __restrict__ row, uint32_t P, float* smem) {
  float acc = 0.f;
  if ((reinterpret_cast<uintptr_t>(row) & 15) == 0) {
    const float4* r4 = reinterpret_cast<const float4*>(row);
    uint32_t n4 = P >> 2;
    for (uint32_t i = threadIdx.x; i < n4; i += blockDim.x) {
      float4 v = __ldg(r4 + i);
      acc = fmaf(v.x, v.x, acc); acc = fmaf(v.y, v.y, acc); acc = fmaf(v.z, v.z, acc); acc = fmaf(v.w, v.w, acc);
    }
    for (uint32_t i = (n4 << 2) + threadIdx.x; i < P; i += blockDim.x) acc = fmaf(row[i], row[i], acc);
  } else {
    for (uint32_t i = threadIdx.x; i < P; i += blockDim.x) acc = fmaf(row[i], row[i], acc);
  }
  return block_sum(acc, smem);
}

__global__ void __launch_bounds__(kClipThreads) clip_rows_kernel(float* __restrict__ g, uint32_t B, uint32_t P, float C,
                                                                 float* __restrict__ norms) {
  __shared__ float smem[32];
  for (uint32_t r = blockIdx.x; r < B; r += gridDim.x) {
    float* row = g + (size_t)r * P;
    float norm = sqrtf(row_sq_norm(row, P, smem));
    float c = clip_factor(norm, C);
    if (norms && threadIdx.x == 0) norms[r] = norm;
    for (uint32_t i = threadIdx.x; i < P; i += blockDim.x) row[i] = c * row[i];
  }
}

__global__ void __launch_bounds__(kClipThreads) row_factor_kernel(const float* __restrict__ g,
                                                                  const uint8_t* __restrict__ mask, uint32_t B,
                                                                  uint32_t P, float C, float* __restrict__ factors) {
  __shared__ float smem[32];
  for (uint32_t r = blockIdx.x; r < B; r += gridDim.x) {
    if (mask && !mask[r]) {           // uniform per CTA
      if (threadIdx.x == 0) factors[r] = 0.f;
      continue;
    }
    float norm = sqrtf(row_sq_norm(g + (size_t)r * P, P, smem));
    if (threadIdx.x == 0) factors[r] = clip_factor(norm, C);
  }
}

// partial[split][j] = sum over the split's rows of factor_i * g[i][j]; one lane per column.
__global__ void __launch_bounds__(kClipThreads) colsum_kernel(const float* __restrict__ g,
                                                              const float* __restrict__ factors, uint32_t B,
                                                              uint32_t P, uint32_t rows_per_split,
                                                              float* __restrict__ partial) {
  __shared__ float red[kClipThreads / 32][33];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const uint32_t col = blockIdx.x * 32 + lane;
  const uint32_t r0 = blockIdx.y * rows_per_split;
  const uint32_t r1 = min(B, r0 + rows_per_split);
  float acc = 0.f;
  if (col < P) {
    uint32_t r = r0 + warp;
    // 4 independent loads in flight per lane
    for (; r + 3 * (kClipThreads / 32) < r1; r += 4 * (kClipThreads / 32)) {
      float f0 = factors[r], f1 = factors[r + 8], f2 = factors[r + 16], f3 = factors[r + 24];
      float v0 = __ldg(g + (size_t)r * P + col), v1 = __ldg(g + (size_t)(r + 8) * P + col);
      float v2 = __ldg(g + (size_t)(r + 16) * P + col), v3 = __ldg(g + (size_t)(r + 24) * P + col);
      acc = fmaf(f0, v0, acc); acc = fmaf(f1, v1, acc); acc = fmaf(f2, v2, acc); acc = fmaf(f3, v3, acc);
    }
    for (; r < r1; r += kClipThreads / 32) acc = fmaf(factors[r], __ldg(g + (size_t)r * P + col), acc);
  }
  red[warp][lane] = acc;
  __syncthreads();
  if (warp == 0 && col < P) {
    float t = 0.f;
#pragma unroll
    for (int w = 0; w < kClipThreads / 32; ++w) t += red[w][lane];
    partial[(size_t)blockIdx.y * P + col] = t;
  }
}

__global__ void __launch_bounds__(kClipThreads) colsum_final_kernel(const float* __restrict__ partial, uint32_t n_splits,
                                                                    uint32_t P, const float* __restrict__ px_loss,
                                                                    const uint8_t* __restrict__ mask, uint32_t B,
                                                                    float* __restrict__ out) {
  uint32_t j = blockIdx.x * blockDim.x + threadIdx.x;
  if (j < P) {
    float t = 0.f;
    for (uint32_t s = 0; s < n_splits; ++s) t += partial[(size_t)s * P + j];
    out[j] = t;
  }
  if (blockIdx.x == 0) {
    __shared__ float smem[32];
    float l = 0.f, c = 0.f;
    for (uint32_t i = threadIdx.x; i < B; i += blockDim.x) {
      float m = (mask && !mask[i]) ? 0.f : 1.f;
      c += m;
      if (px_loss && m != 0.f) l += px_loss[i];
    }
    l = block_sum(l, smem);
    c = block_sum(c, smem);
    if (threadIdx.x == 0) { out[P] = l; out[P + 1] = c; }
  }
}

static uint32_t pick_splits(uint32_t B, uint32_t P) {
  uint32_t col_tiles = (P + 31) / 32;
  uint32_t want = ((uint32_t)sm_count() * 8 + col_tiles - 1) / col_tiles;
  uint32_t max_splits = (B + 63) / 64;
  if (want > max_splits) want = max_splits;
  if (want < 1) want = 1;
  if (want > 65535) want = 65535;
  return want;
}


// full_norm(vector_parts, ord) for ord != 2 (d3p/svi.py:68-87 -> jnp.linalg.norm of the concatenated leaves):
// inf -> max |x|, -inf -> min |x|, 0 -> number of non-zeros, p -> (sum |x|^p)^(1/p).  One CTA, fixed order.
__global__ void __launch_bounds__(1024) vector_norm_kernel(const float* __restrict__ x, size_t n, float ord, float* out) {
  __shared__ float red[32];
  const bool is_max = isinf(ord) && ord > 0, is_min = isinf(ord) && ord < 0;
  float acc = is_min ? __int_as_float(0x7f800000) : 0.f;
  for (size_t i = threadIdx.x; i < n; i += 1024) {
    const float a = fabsf(x[i]);
    if (is_max) acc = fmaxf(acc, a);
    else if (is_min) acc = fminf(acc, a);
    else if (ord == 0.f) acc += a != 0.f ? 1.f : 0.f;
    else if (ord == 1.f) acc += a;
    else acc += powf(a, ord);
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    const float v = __shfl_xor_sync(0xffffffffu, acc, o);
    acc = is_max ? fmaxf(acc, v) : is_min ? fminf(acc, v) : acc + v;
  }
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = acc;
  __syncthreads();
  if (threadIdx.x == 0) {
    float t = red[0];
#pragma unroll
    for (int w = 1; w < 32; ++w) t = is_max ? fmaxf(t, red[w]) : is_min ? fminf(t, red[w]) : t + red[w];
    if (n == 0) t = 0.f;
    *out = (is_max || is_min || ord == 0.f || ord == 1.f) ? t : powf(t, 1.0f / ord);
  }
}

}  // namespace d3p

using namespace d3p;

extern "C" {

int32_t d3p_clip_rows_f32(float* px_grads_d, uint32_t B, uint32_t P, float C, float* norms_d, void* stream) {
  if (C == 0.f) return D3P_ERR_INVALID_ARGUMENT;   // clip_gradient raises for c == 0 (d3p/svi.py:119)
  if (!px_grads_d && B && P) return D3P_ERR_INVALID_ARGUMENT;
  if (B == 0) return D3P_OK;
  unsigned grid = B < (unsigned)sm_count() * 8 ? B : (unsigned)sm_count() * 8;
  clip_rows_kernel<<<grid, kClipThreads, 0, (cudaStream_t)stream>>>(px_grads_d, B, P, C, norms_d);
  return check_launch();
}

int32_t d3p_vector_norm_f32(const float* x_d, size_t n, float ord, float* out_d, void* stream) {
  if ((!x_d && n) || !out_d || ord != ord) return D3P_ERR_INVALID_ARGUMENT;
  vector_norm_kernel<<<1, 1024, 0, (cudaStream_t)stream>>>(x_d, n, ord, out_d);
  return check_launch();
}

size_t d3p_clip_and_sum_workspace_bytes(uint32_t B, uint32_t P) {
  return align_up((size_t)B * sizeof(float), 256) + (size_t)pick_splits(B, P) * P * sizeof(float);
}

int32_t d3p_clip_and_sum_f32(const float* px_grads_d, const float* px_loss_d, const uint8_t* mask_d,
                             uint32_t B, uint32_t P, float C, float* sum_d, void* ws_d, size_t ws_bytes,
                             void* stream) {
  if (C == 0.f || !sum_d || !ws_d || (!px_grads_d && B && P)) return D3P_ERR_INVALID_ARGUMENT;
  if (ws_bytes < d3p_clip_and_sum_workspace_bytes(B, P)) return D3P_ERR_WORKSPACE;
  cudaStream_t s = (cudaStream_t)stream;
  if (B == 0 || P == 0) {
    cudaMemsetAsync(sum_d, 0, ((size_t)P + 2) * sizeof(float), s);
    if (B == 0) return check_launch();
  }
  float* factors = reinterpret_cast<float*>(ws_d);
  float* partial = reinterpret_cast<float*>(reinterpret_cast<char*>(ws_d) + align_up((size_t)B * sizeof(float), 256));
  uint32_t splits = pick_splits(B, P);
  uint32_t rows_per_split = (B + splits - 1) / splits;
  unsigned grid = B < (unsigned)sm_count() * 8 ? B : (unsigned)sm_count() * 8;
  row_factor_kernel<<<grid, kClipThreads, 0, s>>>(px_grads_d, mask_d, B, P, C, factors);
  if (P) colsum_kernel<<<dim3((P + 31) / 32, splits), kClipThreads, 0, s>>>(px_grads_d, factors, B, P, rows_per_split, partial);
  unsigned fgrid = P ? (P + kClipThreads - 1) / kClipThreads : 1;
  colsum_final_kernel<<<fgrid, kClipThreads, 0, s>>>(partial, splits, P, px_loss_d, mask_d, B, sum_d);
  return check_launch();
}

}  // extern "C"
