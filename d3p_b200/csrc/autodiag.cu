// AutoDiagonalNormal guide over a user model: the guide draw and the per-example gradient / clip / clipped sum of
// a DP-VI step, around a model log density that the caller differentiates itself (see include/d3p_b200.h).
//
// The draw is the fused families' joint-site draw: the guide_rng / next_site key chain of common.cuh, then one
// normal per element.  The step is two passes over the caller's [rows, ld] arrays h (= dU/dtheta) and eps:
//   pass 1 (autodiag_rows_kernel): one CTA per row; norm of (gl, gs), |eps|^2 -> c_i and S * loss_i;
//   pass 2 (autodiag_colsum_kernel): column tiles x example splits; sum_i c_i (gl_i, gs_i), sum S loss_i, count.
// gl and gs are formed on the fly from (h, eps) and the per-element constants a = s' and (1/S) a / s of a small
// prologue kernel, so no [rows, 2D] array exists.  Every sum has a fixed order: results are run-to-run identical.
#include "common.cuh"
#include "launch.cuh"
#include "meanfield_common.cuh"
#include "reduce.cuh"

namespace d3p {

constexpr int kAdThreads = 256;
constexpr int kAdWarps = kAdThreads / 32;
constexpr float kLogSqrt2Pi = 0.918938533f;

struct DrawArgs {
  const float* params;
  const uint32_t* key_d;
  uint32_t k0, k1, B, pos_begin, rows, D, half, loc_off, scale_off;
  size_t ld;
  float* theta;
  float* eps;
};

// kEval: SVI.evaluate's single draw from the key itself with the exact normal transform of meanfield_eval_kernel;
// else the per-example draws with the step kernels' transform.
template <bool kEval>
__global__ void __launch_bounds__(kAdThreads) autodiag_draw_kernel(DrawArgs a) {
  const TfKey K = tf_key_arg(a.k0, a.k1, a.key_d);
  for (uint32_t r = blockIdx.x; r < a.rows; r += gridDim.x) {
    TfKey rng = guide_rng(kEval ? K : tf_example_key(K, a.B, a.pos_begin + r));   // jax.random.split(key, B)[p]
    const TfKey k_site = next_site(rng);               // the `_auto_latent` site
    float* th = a.theta + (size_t)r * a.ld;
    float* ep = a.eps + (size_t)r * a.ld;
    for (uint32_t j = threadIdx.x; j < a.half; j += kAdThreads) {
      const uint32_t e1 = j + a.half;
      uint32_t y[2];
      threefry2x32(k_site, j, e1 < a.D ? e1 : 0u, y[0], y[1]);
#pragma unroll
      for (int h = 0; h < 2; ++h) {
        const uint32_t e = h ? e1 : j;
        if (e >= a.D) break;
        const float ev = kEval ? bits_to_normal<false>(y[h]) : bits_to_normal_fast(y[h]);
        const float s = softplus_f(a.params[a.scale_off + e]);
        ep[e] = ev;
        th[e] = fmaf(ev, s, a.params[a.loc_off + e]);
      }
    }
  }
}

struct StepLayout {
  uint32_t n_partials, col_tiles, rows_per_split;
  size_t consts_off, rows_off, bytes;   // byte offsets into the workspace
};

static StepLayout step_layout(const d3p_autodiag_desc* d, uint32_t rows) {
  StepLayout L;
  const uint32_t vcols = 2u * d->latent_dim + 2u;   // loc | scale | loss | count
  L.col_tiles = (vcols + 31) / 32;
  uint32_t want = ((uint32_t)sm_count() * 8 + L.col_tiles - 1) / L.col_tiles;
  const uint32_t max_splits = (rows + 63) / 64;
  if (want > max_splits) want = max_splits;
  if (d->n_params >= 32768 && want > 64) want = 64;   // finalize_quad_kernel takes at most 64 partial rows
  if (want > 65535) want = 65535;
  if (want < 1) want = 1;
  L.n_partials = want;
  L.rows_per_split = (rows + want - 1) / want;
  L.consts_off = align_up((size_t)want * (d->n_params + 2) * sizeof(float), 256);
  L.rows_off = L.consts_off + align_up(((size_t)2 * d->latent_dim + 1) * sizeof(float), 256);
  L.bytes = L.rows_off + (size_t)3 * rows * sizeof(float);
  return L;
}

struct StepArgsAd {
  const float* params;
  const float* eps;
  const float* grad;
  size_t ld;
  const float* potential;
  const uint8_t* mask;
  const int32_t* num_valid;
  uint32_t B, pos_begin, rows, D, P, loc_off, scale_off, rows_per_split;
  float inv_S, C;
  float* consts;      // [2D + 1]: a = s' | (1/S) a / s | sum_e log s_e
  float* fac;         // [rows]: c_i (0 for skipped rows)
  float* loss;        // [rows]: S * loss_i (0 for skipped rows)
  float* cnt;         // [rows]: 1 for the rows that count, else 0
  float* px_norms;
  float* px_grads;
  float* px_loss;
  float* partials;
};

D3P_D float grad_scale(float gl, float eps, float a, float bt) { return fmaf(gl, eps * a, -bt); }

__global__ void __launch_bounds__(512) autodiag_consts_kernel(StepArgsAd a) {
  __shared__ float red[32];
  float log_s = 0.f;
  for (uint32_t e = threadIdx.x; e < a.D; e += 512) {
    float s, aa, bt, ls;
    link_terms<D3P_LINK_SOFTPLUS>(a.params[a.scale_off + e], a.inv_S, s, aa, bt, ls);
    a.consts[e] = aa;
    a.consts[a.D + e] = bt;
    log_s += ls;
  }
  log_s = block_sum(log_s, red);
  if (threadIdx.x == 0) a.consts[2 * a.D] = log_s;
}

__global__ void __launch_bounds__(kAdThreads) autodiag_rows_kernel(StepArgsAd a) {
  __shared__ float red[32];
  const uint32_t nv = a.num_valid ? (uint32_t)max(*a.num_valid, 0) : 0xffffffffu;
  const float* __restrict__ A = a.consts;
  const float* __restrict__ BT = a.consts + a.D;
  for (uint32_t r = blockIdx.x; r < a.rows; r += gridDim.x) {
    const uint32_t p = a.pos_begin + r;
    if (p >= nv || (a.mask && !a.mask[p])) {          // uniform per CTA; the row's inputs are not read
      if (threadIdx.x == 0) { a.fac[r] = 0.f; a.loss[r] = 0.f; a.cnt[r] = 0.f; }
      continue;
    }
    const float* __restrict__ h = a.grad + (size_t)r * a.ld;
    const float* __restrict__ ep = a.eps + (size_t)r * a.ld;
    float* pg = a.px_grads ? a.px_grads + (size_t)p * a.P : nullptr;
    float nrm = 0.f, e2 = 0.f;
    for (uint32_t e = threadIdx.x; e < a.D; e += kAdThreads) {
      const float ev = __ldg(ep + e);
      const float gl = __ldg(h + e) * a.inv_S;
      const float gs = grad_scale(gl, ev, A[e], BT[e]);
      nrm = fmaf(gl, gl, fmaf(gs, gs, nrm));
      e2 = fmaf(ev, ev, e2);
      if (pg) { pg[a.loc_off + e] = gl; pg[a.scale_off + e] = gs; }
    }
    nrm = block_sum(nrm, red);
    e2 = block_sum(e2, red);
    if (threadIdx.x == 0) {
      const float norm = sqrtf(nrm);
      // S * loss_i = U_i - log q(theta_i) with log q = -|eps|^2 / 2 - sum log s - D log sqrt(2 pi)
      const float l = a.potential[r] - 0.5f * e2 - a.consts[2 * a.D] - (float)a.D * kLogSqrt2Pi;
      a.fac[r] = clip_factor(norm, a.C);
      a.loss[r] = l;
      a.cnt[r] = 1.f;
      if (a.px_norms) a.px_norms[p] = norm;
      if (a.px_loss) a.px_loss[p] = l;
    }
  }
}

// partials[split][col]: virtual column j < D is auto_loc[j], D <= j < 2D auto_scale[j - D], 2D the loss, 2D + 1 the
// count; one lane per column, the CTA's warps take every kAdWarps-th row of the split and are summed in warp order.
__global__ void __launch_bounds__(kAdThreads) autodiag_colsum_kernel(StepArgsAd a) {
  __shared__ float red[kAdWarps][33];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const uint32_t j = blockIdx.x * 32 + lane;
  const uint32_t r0 = blockIdx.y * a.rows_per_split;
  const uint32_t r1 = min(a.rows, r0 + a.rows_per_split);
  const uint32_t D = a.D;
  float acc = 0.f;
  if (j < 2 * D) {
    const bool is_scale = j >= D;
    const uint32_t e = is_scale ? j - D : j;
    const float ae = is_scale ? a.consts[e] : 0.f, bte = is_scale ? a.consts[D + e] : 0.f;
#pragma unroll 4
    for (uint32_t r = r0 + warp; r < r1; r += kAdWarps) {
      if (a.cnt[r] == 0.f) continue;                  // warp-uniform: padding rows may hold NaN
      const float gl = __ldg(a.grad + (size_t)r * a.ld + e) * a.inv_S;
      const float g = is_scale ? grad_scale(gl, __ldg(a.eps + (size_t)r * a.ld + e), ae, bte) : gl;
      acc = fmaf(a.fac[r], g, acc);
    }
  } else if (j < 2 * D + 2) {
    const float* v = j == 2 * D ? a.loss : a.cnt;     // 0 on the rows that do not count
    for (uint32_t r = r0 + warp; r < r1; r += kAdWarps) acc += v[r];
  }
  red[warp][lane] = acc;
  __syncthreads();
  if (warp == 0 && j < 2 * D + 2) {
    float t = 0.f;
#pragma unroll
    for (int w = 0; w < kAdWarps; ++w) t += red[w][lane];
    const uint32_t col = j < D ? a.loc_off + j : j < 2 * D ? a.scale_off + (j - D) : a.P + (j - 2 * D);
    a.partials[(size_t)blockIdx.y * (a.P + 2) + col] = t;
  }
}

static bool desc_ok(const d3p_autodiag_desc* d) {
  if (!d || d->latent_dim == 0) return false;
  const uint64_t D = d->latent_dim;
  if ((uint64_t)d->loc_off + D > d->n_params || (uint64_t)d->scale_off + D > d->n_params) return false;
  const uint64_t lo = d->loc_off, so = d->scale_off;
  return lo + D <= so || so + D <= lo;             // the two leaves do not overlap
}

static int32_t draw_impl(const d3p_autodiag_desc* desc, const float* params_d, const uint32_t* key_h,
                         const uint32_t* key_d, uint32_t B, uint32_t pos_begin, uint32_t pos_end, float* theta_d,
                         float* eps_d, size_t ld, void* stream) {
  if (!desc_ok(desc) || !params_d || (!key_h && !key_d) || ld < desc->latent_dim) return D3P_ERR_INVALID_ARGUMENT;
  if (B != 0 && (pos_begin > pos_end || pos_end > B)) return D3P_ERR_INVALID_ARGUMENT;
  DrawArgs a;
  a.params = params_d; a.key_d = key_d;
  a.k0 = key_h ? key_h[0] : 0u; a.k1 = key_h ? key_h[1] : 0u;
  a.B = B; a.pos_begin = B ? pos_begin : 0u; a.rows = B ? pos_end - pos_begin : 1u;
  a.D = desc->latent_dim; a.half = (a.D + 1) / 2; a.loc_off = desc->loc_off; a.scale_off = desc->scale_off;
  a.ld = ld; a.theta = theta_d; a.eps = eps_d;
  if (a.rows == 0) return D3P_OK;
  if (!theta_d || !eps_d) return D3P_ERR_INVALID_ARGUMENT;
  const unsigned cap = 16u * (unsigned)sm_count();
  const unsigned grid = a.rows < cap ? a.rows : cap;
  cudaStream_t s = (cudaStream_t)stream;
  if (B == 0) autodiag_draw_kernel<true><<<grid, kAdThreads, 0, s>>>(a);
  else autodiag_draw_kernel<false><<<grid, kAdThreads, 0, s>>>(a);
  return check_launch();
}

}  // namespace d3p

using namespace d3p;

extern "C" {

int32_t d3p_autodiag_draw_f32(const d3p_autodiag_desc* desc, const float* params_d, const uint32_t threefry_key_h[2],
                              uint32_t B, uint32_t pos_begin, uint32_t pos_end, float* theta_d, float* eps_d,
                              size_t ld, void* stream) {
  if (!threefry_key_h) return D3P_ERR_INVALID_ARGUMENT;
  return draw_impl(desc, params_d, threefry_key_h, nullptr, B, pos_begin, pos_end, theta_d, eps_d, ld, stream);
}

int32_t d3p_autodiag_draw_f32_dk(const d3p_autodiag_desc* desc, const float* params_d, const uint32_t* threefry_key_d,
                                 uint32_t B, uint32_t pos_begin, uint32_t pos_end, float* theta_d, float* eps_d,
                                 size_t ld, void* stream) {
  if (!threefry_key_d) return D3P_ERR_INVALID_ARGUMENT;
  return draw_impl(desc, params_d, nullptr, threefry_key_d, B, pos_begin, pos_end, theta_d, eps_d, ld, stream);
}

size_t d3p_autodiag_workspace_bytes(const d3p_autodiag_desc* desc, uint32_t rows, uint32_t* n_partials_out) {
  if (!desc_ok(desc)) return 0;
  const StepLayout L = step_layout(desc, rows);
  if (n_partials_out) *n_partials_out = L.n_partials;
  return L.bytes;
}

int32_t d3p_dpsvi_step_autodiag(const d3p_autodiag_desc* desc, const float* params_d, const float* eps_d,
                                const float* grad_d, size_t ld, const float* potential_d, const uint8_t* mask_d,
                                const int32_t* num_valid_d, uint32_t B, uint32_t pos_begin, uint32_t pos_end,
                                float obs_scale, float C, float* px_norms_d, float* px_grads_d, float* px_loss_d,
                                void* ws_d, size_t ws_bytes, void* stream) {
  if (!desc_ok(desc) || !params_d || !ws_d || ld < desc->latent_dim) return D3P_ERR_INVALID_ARGUMENT;
  if (C == 0.f || obs_scale == 0.f || B == 0 || pos_begin > pos_end || pos_end > B) return D3P_ERR_INVALID_ARGUMENT;
  const uint32_t rows = pos_end - pos_begin;
  if (rows && (!eps_d || !grad_d || !potential_d)) return D3P_ERR_INVALID_ARGUMENT;
  const StepLayout L = step_layout(desc, rows);
  if (ws_bytes < L.bytes) return D3P_ERR_WORKSPACE;
  char* ws = static_cast<char*>(ws_d);
  StepArgsAd a;
  a.params = params_d; a.eps = eps_d; a.grad = grad_d; a.ld = ld; a.potential = potential_d; a.mask = mask_d;
  a.num_valid = num_valid_d; a.B = B; a.pos_begin = pos_begin; a.rows = rows; a.D = desc->latent_dim;
  a.P = desc->n_params; a.loc_off = desc->loc_off; a.scale_off = desc->scale_off; a.rows_per_split = L.rows_per_split;
  a.inv_S = 1.0f / obs_scale; a.C = C;
  a.consts = reinterpret_cast<float*>(ws + L.consts_off);
  a.fac = reinterpret_cast<float*>(ws + L.rows_off);
  a.loss = a.fac + rows;
  a.cnt = a.loss + rows;
  a.px_norms = px_norms_d; a.px_grads = px_grads_d; a.px_loss = px_loss_d;
  a.partials = reinterpret_cast<float*>(ws);
  cudaStream_t s = (cudaStream_t)stream;
  if (2ull * desc->latent_dim < desc->n_params &&       // parameters outside the two leaves get zero partials
      cudaMemsetAsync(a.partials, 0, (size_t)L.n_partials * (a.P + 2) * sizeof(float), s) != cudaSuccess)
    return D3P_ERR_CUDA;
  autodiag_consts_kernel<<<1, 512, 0, s>>>(a);
  if (rows) {
    const unsigned cap = 16u * (unsigned)sm_count();
    autodiag_rows_kernel<<<rows < cap ? rows : cap, kAdThreads, 0, s>>>(a);
  }
  autodiag_colsum_kernel<<<dim3(L.col_tiles, L.n_partials), kAdThreads, 0, s>>>(a);
  return check_launch();
}

}  // extern "C"
