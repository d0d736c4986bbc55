// K11: DPSVI.evaluate (d3p/svi.py:436-449 -> numpyro SVI.evaluate): the non-private ELBO loss of a whole
// batch with ONE guide sample, for the mean-field families.  Not on the throughput path; kept on the
// device so that a training loop never copies the batch to the host.
//     loss = -( log p(theta) + (N / B) sum_i log p(x_i | theta) - log q(theta) ),  theta = loc + s * eps
// eps comes from the Threefry key the caller derives as numpyro does (split(rng_key)[1]), through the
// same seed-handler plumbing as the per-example path: (model_seed, guide_seed) = split(key); one
// split per latent site.
#include "common.cuh"
#include "launch.cuh"
#include "meanfield_common.cuh"

namespace d3p {

struct EvalArgs {
  const float* params; const float* x; size_t x_stride; const int32_t* y; const int32_t* idx;
  const uint32_t* key_d;   // *_dk: Threefry key in device memory (else nullptr)
  uint32_t B, k0, k1, d, n_main, half, loc_off, rho_off, b_loc_off, b_rho_off;
  int family, link, has_b;
  float N, inv_var, log_norm_lik;
  float* partials;   // [gridDim.x + 1]: per-CTA log-lik sums, then log p(theta) - log q(theta)
  float* loss;
};

constexpr int kEvalThreads = 256;

__global__ void __launch_bounds__(kEvalThreads) meanfield_eval_kernel(EvalArgs a) {
  extern __shared__ float th[];             // theta[n_main]
  __shared__ float red[kEvalThreads / 32];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const TfKey K = tf_key_arg(a.k0, a.k1, a.key_d);
  TfKey rng = guide_rng(K);
  const TfKey k_main = next_site(rng);
  float pq = 0.f;                           // log p(theta) - log q(theta), accumulated by every CTA, used from CTA 0
  const float kLogSqrt2Pi = 0.918938533f;
  for (uint32_t c = threadIdx.x; c < a.half; c += kEvalThreads) {
    uint32_t y0, y1;
    const uint32_t e1 = c + a.half;
    threefry2x32(k_main, c, e1 < a.n_main ? e1 : 0u, y0, y1);
#pragma unroll
    for (int h = 0; h < 2; ++h) {
      const uint32_t e = h ? e1 : c;
      if (e >= a.n_main) break;
      const float eps = bits_to_normal<false>(h ? y1 : y0);
      const float rho = a.params[a.rho_off + e];
      const float s = a.link == D3P_LINK_EXP ? expf(rho) : softplus_f(rho);
      const float t = fmaf(eps, s, a.params[a.loc_off + e]);
      th[e] = t;
      pq += (-0.5f * t * t - kLogSqrt2Pi) - (-0.5f * eps * eps - logf(2.50662827f * s));
    }
  }
  float th_b = 0.f;
  if (a.has_b) {
    const TfKey k_b = next_site(rng);
    uint32_t y0, y1;
    threefry2x32(k_b, 0u, 0u, y0, y1);
    const float eps = bits_to_normal<false>(y0);
    const float rho = a.params[a.b_rho_off];
    const float s = a.link == D3P_LINK_EXP ? expf(rho) : softplus_f(rho);
    th_b = fmaf(eps, s, a.params[a.b_loc_off]);
    if (threadIdx.x == 0) pq += (-0.5f * th_b * th_b - kLogSqrt2Pi) - (-0.5f * eps * eps - logf(2.50662827f * s));
  }
  __syncthreads();
  if (a.family == D3P_FAMILY_LOGREG && !a.has_b) th_b = th[a.d];      // joint site: intercept is element d
  float ll = 0.f;
  const uint32_t warps = gridDim.x * (kEvalThreads / 32);
  for (uint32_t r = blockIdx.x * (kEvalThreads / 32) + warp; r < a.B; r += warps) {
    const size_t row = a.idx ? (size_t)(uint32_t)a.idx[r] : (size_t)r;
    const float* xr = a.x + row * a.x_stride;
    float s = 0.f;
    if (a.family == D3P_FAMILY_LOGREG) {
      for (uint32_t j = lane; j < a.d; j += 32) s = fmaf(xr[j], th[j], s);
      s = row_loglik<D3P_FAMILY_LOGREG>(group_sum<32>(s), th_b, (float)a.y[row], a.d, a.inv_var, a.log_norm_lik);
    } else {
      for (uint32_t j = lane; j < a.d; j += 32) { const float q = xr[j] - th[j]; s = fmaf(q, q, s); }
      s = row_loglik<D3P_FAMILY_GAUSS>(group_sum<32>(s), th_b, 0.f, a.d, a.inv_var, a.log_norm_lik);
    }
    ll += s;                                  // identical on every lane
  }
  pq = group_sum<32>(pq);
  if (lane == 0) red[warp] = ll;
  __syncthreads();
  if (threadIdx.x == 0) {
    float t = 0.f;
#pragma unroll
    for (int w = 0; w < kEvalThreads / 32; ++w) t += red[w];
    a.partials[blockIdx.x] = t;
  }
  __syncthreads();
  if (blockIdx.x == 0) {
    if (lane == 0) red[warp] = pq;
    __syncthreads();
    if (threadIdx.x == 0) {
      float t = 0.f;
#pragma unroll
      for (int w = 0; w < kEvalThreads / 32; ++w) t += red[w];
      a.partials[gridDim.x] = t;
    }
  }
}

__global__ void meanfield_eval_finish_kernel(EvalArgs a, uint32_t n_ctas) {
  if (threadIdx.x != 0 || blockIdx.x != 0) return;
  float ll = 0.f;
  for (uint32_t i = 0; i < n_ctas; ++i) ll += a.partials[i];
  a.loss[0] = -(a.partials[n_ctas] + (a.N / (float)a.B) * ll);
}

}  // namespace d3p

using namespace d3p;

extern "C" size_t d3p_elbo_evaluate_workspace_bytes(void) { return ((size_t)2 * sm_count() + 1) * sizeof(float); }

extern "C" int32_t d3p_elbo_evaluate_meanfield(const d3p_meanfield_desc* desc, const float* params_d, const float* x_d,
                                               size_t x_row_stride, const int32_t* y_d, const int32_t* idx_d, uint32_t B,
                                               const uint32_t threefry_key_h[2], float* loss_d, void* ws_d,
                                               size_t ws_bytes, void* stream) {
  if (!desc || !params_d || !x_d || !threefry_key_h || !loss_d || !ws_d || B == 0) return D3P_ERR_INVALID_ARGUMENT;
  if (desc->family != D3P_FAMILY_LOGREG && desc->family != D3P_FAMILY_GAUSS) return D3P_ERR_UNSUPPORTED;
  if (desc->family == D3P_FAMILY_LOGREG && !y_d) return D3P_ERR_INVALID_ARGUMENT;
  if (ws_bytes < d3p_elbo_evaluate_workspace_bytes()) return D3P_ERR_WORKSPACE;
  MeanfieldSite site;
  if (!meanfield_site(desc, x_row_stride, site)) return D3P_ERR_INVALID_ARGUMENT;
  EvalArgs a;
  a.params = params_d; a.x = x_d; a.x_stride = x_row_stride; a.y = y_d; a.idx = idx_d; a.B = B;
  a.k0 = threefry_key_h[0]; a.k1 = threefry_key_h[1]; a.key_d = nullptr;
  a.d = desc->d; a.n_main = site.n_main; a.half = site.half;
  a.loc_off = desc->loc_off; a.rho_off = desc->rho_off; a.b_loc_off = desc->b_loc_off; a.b_rho_off = desc->b_rho_off;
  a.family = desc->family; a.link = desc->link; a.has_b = site.has_b;
  a.N = desc->num_obs_total; a.inv_var = site.inv_var; a.log_norm_lik = site.log_norm_lik;
  a.partials = static_cast<float*>(ws_d);
  a.loss = loss_d;
  const size_t smem = (size_t)(a.n_main + 1) * sizeof(float);
  if (smem > 200 * 1024) return D3P_ERR_UNSUPPORTED;
  unsigned grid = (B + 7) / 8;
  const unsigned cap = 2u * (unsigned)sm_count();
  if (grid > cap) grid = cap;
  cudaStream_t s = (cudaStream_t)stream;
  if (smem > 48 * 1024 &&
      cudaFuncSetAttribute(meanfield_eval_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess)
    return D3P_ERR_CUDA;
  meanfield_eval_kernel<<<grid, kEvalThreads, smem, s>>>(a);
  int32_t rc = check_launch();
  if (rc != D3P_OK) return rc;
  meanfield_eval_finish_kernel<<<1, 32, 0, s>>>(a, grid);
  return check_launch();
}
