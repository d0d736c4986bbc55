// K5a/K5b (+K10): fused per-example gradient, L2 norm, clip and clipped sum for mean-field
// Normal guides.  Replaces DPSVI._compute_per_example_gradients, _clip_gradients and the sum
// half of _combine_gradients (d3p/svi.py:238-348) for
//   LOGREG: examples/logistic_regression.py:49-86  (and its AutoDiagonalNormal variant)
//   GAUSS : examples/simple_gaussian_posterior.py:50-83
// No [B, P] per-example gradient tensor exists: a group of G lanes owns one example at a time,
// draws the example's guide noise with Threefry in registers (jax.random.split per example,
// d3p/svi.py:289-290, + numpyro seed/Normal.sample plumbing), forms the closed-form gradient
// (SURVEY.md App. A), reduces the norm with shuffles and accumulates c_i * g_i in registers
// across all examples the lane processes.  CTA partial sums are written in a fixed order.
//
// Element e of the (main) latent site: x_e = X[row, e] for e < d, and 1.0 for the intercept when
// it is part of a joint `_auto_latent` site (e == d).  With theta_e = loc_e + eps_e * s_e:
//   gl_e = d loss / d loc_e = theta_e / S + h_e,   h_e = (N/S) * d(-loglik)/d theta_e
//   gs_e = d loss / d rho_e = gl_e * eps_e * s'_e - (1/S) * s'_e / s_e
#include <type_traits>

#include "common.cuh"
#include "launch.cuh"
#include "meanfield_common.cuh"

namespace d3p {

template <int FAMILY, int LINK, int G, int NQ>
__global__ void __launch_bounds__(kStepThreads, 1) meanfield_step_kernel(StepArgs a) {
  constexpr int SUB = 32 / G;                 // examples in flight per warp
  constexpr int TILE = G < 8 ? G : 8;         // examples per group between key-derivation rounds
  constexpr int NS = 2 * NQ;                  // latent elements owned by a lane
  constexpr int NALLOC = 2 * G * NQ;          // padded element count
  static_assert(NS <= 64, "the slot validity mask has 64 bits");
  extern __shared__ float smem[];
  float* s_loc = smem;
  float* s_scl = s_loc + NALLOC;
  float* s_a = s_scl + NALLOC;                // softplus only: s'
  float* s_sa = s_a + (LINK == D3P_LINK_EXP ? 0 : NALLOC);    // softplus only: s / s'
  float* s_bt = s_sa + (LINK == D3P_LINK_EXP ? 0 : NALLOC);   // softplus only: (1/S) s'/s
  float* s_acc = s_bt + (LINK == D3P_LINK_EXP ? 0 : NALLOC);  // [P + 2] CTA partial sums
  __shared__ float s_red[kStepWarps];

  asm volatile("griddepcontrol.launch_dependents;");   // see meanfield_step_vec.cu: the finalize kernel may be placed early
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int glane = lane & (G - 1), sg = lane / G;
  const unsigned gm = group_mask<G>(lane);

  // ---- prologue: constrained guide parameters into shared memory ----------------------------
  float log_s_part = 0.f;
  for (int e = threadIdx.x; e < NALLOC; e += kStepThreads) {
    float loc = 0.f, s = 0.f, aa = 0.f, bt = 0.f, ls = 0.f;
    if ((uint32_t)e < a.n_main) {
      loc = a.params[a.loc_off + e];
      link_terms<LINK>(a.params[a.rho_off + e], a.inv_S, s, aa, bt, ls);
    }
    s_loc[e] = loc; s_scl[e] = s;
    if (LINK != D3P_LINK_EXP) { s_a[e] = aa; s_sa[e] = (aa != 0.f) ? s / aa : 0.f; s_bt[e] = bt; }
    log_s_part += ls;
  }
  float b_loc = 0.f, b_s = 0.f, b_a = 0.f, b_bt = 0.f;
  if (a.has_b) {
    float ls;
    b_loc = a.params[a.b_loc_off];
    link_terms<LINK>(a.params[a.b_rho_off], a.inv_S, b_s, b_a, b_bt, ls);
    if (threadIdx.x == 0) log_s_part += ls;
  }
  log_s_part = gsum<32>(log_s_part, 0xffffffffu);
  if (lane == 0) s_red[warp] = log_s_part;
  for (uint32_t j = threadIdx.x; j < a.P + 2; j += kStepThreads) s_acc[j] = 0.f;
  __syncthreads();
  float sum_log_s = 0.f;
#pragma unroll
  for (int w = 0; w < kStepWarps; ++w) sum_log_s += s_red[w];
  const InterceptGuide b{b_loc, b_s, b_a, b_bt};

  // validity of the lane's slots
  using mask_t = typename std::conditional<(NS > 32), uint64_t, uint32_t>::type;
  mask_t vmask = 0;          // one bit per slot (NS <= 64)
#pragma unroll
  for (int k = 0; k < NQ; ++k) {
    uint32_t q = glane + G * k;
    if (q < a.half) {
      vmask |= (mask_t)1 << (2 * k);
      if (q + a.half < a.n_main) vmask |= (mask_t)1 << (2 * k + 1);
    }
  }

  float acc_loc[NS], acc_rho[NS];
#pragma unroll
  for (int s = 0; s < NS; ++s) { acc_loc[s] = 0.f; acc_rho[s] = 0.f; }
  float acc_bloc = 0.f, acc_brho = 0.f, acc_loss = 0.f, acc_cnt = 0.f;

  const TfKey K = tf_key_arg(a.k0, a.k1, a.key_d);
  const uint32_t npos = a.pos_end - a.pos_begin;
  const uint32_t nv = a.num_valid ? (uint32_t)max(*a.num_valid, 0) : 0xffffffffu;
  const uint32_t total_warps = gridDim.x * kStepWarps;

  for (uint32_t wt = blockIdx.x * kStepWarps + warp; (uint64_t)wt * (SUB * TILE) < npos; wt += total_warps) {
    const uint32_t base = a.pos_begin + (wt * SUB + sg) * TILE;
    // ---- per-example keys: lane t of the group derives example base + t -----------------------
    const uint32_t my_p = base + glane;
    bool my_valid = (glane < TILE) && (my_p < a.pos_end) && (my_p < nv) && (!a.mask || a.mask[my_p]);
    uint32_t my_k0 = 0, my_k1 = 0, my_row = 0;
    float my_eb = 0.f, my_y = 0.f;
    if (my_valid) {
      TfKey rng = guide_rng(tf_example_key(K, a.B, my_p));   // jax.random.split(key, B)[p]
      const TfKey k_main = next_site(rng);
      my_k0 = k_main.k0; my_k1 = k_main.k1;
      if (a.has_b) {
        const TfKey k_b = next_site(rng);                // second latent site (intercept)
        uint32_t y0, y1;
        threefry2x32(k_b, 0u, 0u, y0, y1);               // random_bits(k, 32, ()) -> counts [0, pad 0]
        my_eb = bits_to_normal_fast(y0);
      }
      my_row = a.idx ? (uint32_t)a.idx[my_p] : my_p;
      if (FAMILY == D3P_FAMILY_LOGREG) my_y = (float)a.y[my_row];
    }
#pragma unroll 1
    for (int t = 0; t < TILE; ++t) {
      const bool valid = __shfl_sync(gm, (int)my_valid, t, G) != 0;
      if (!valid) continue;                              // group-uniform
      const uint32_t kw0 = __shfl_sync(gm, my_k0, t, G), kw1 = __shfl_sync(gm, my_k1, t, G);
      const uint32_t row = __shfl_sync(gm, my_row, t, G);
      const float eb = __shfl_sync(gm, my_eb, t, G);
      const float yv = __shfl_sync(gm, my_y, t, G);
      const float* __restrict__ xr = a.x + (size_t)row * a.x_stride;

      float xv[NS], ev[NS];
#pragma unroll
      for (int k = 0; k < NQ; ++k) {
        const uint32_t e0 = glane + G * k, e1 = e0 + a.half;
        xv[2 * k] = ((vmask >> (2 * k)) & (mask_t)1) ? (e0 < a.d ? __ldg(xr + e0) : 1.0f) : 0.f;
        xv[2 * k + 1] = ((vmask >> (2 * k + 1)) & (mask_t)1) ? (e1 < a.d ? __ldg(xr + e1) : 1.0f) : 0.f;
      }
      const TfKey km(kw0, kw1);
#pragma unroll
      for (int k = 0; k < NQ; ++k) {
        const uint32_t e0 = glane + G * k, e1 = e0 + a.half;
        ev[2 * k] = 0.f; ev[2 * k + 1] = 0.f;
        if ((vmask >> (2 * k)) & (mask_t)1) {
          uint32_t y0, y1;
          threefry2x32(km, e0, (e1 < a.n_main) ? e1 : 0u, y0, y1);
          ev[2 * k] = bits_to_normal_fast(y0);
          if ((vmask >> (2 * k + 1)) & (mask_t)1) ev[2 * k + 1] = bits_to_normal_fast(y1);
        }
      }
      // ---- pass 1: theta, sums -----------------------------------------------------------------
      float zdot = 0.f, s_th2 = 0.f, s_e2 = 0.f, s_res2 = 0.f;
#pragma unroll
      for (int s = 0; s < NS; ++s) {
        const int e = glane + G * (s >> 1) + ((s & 1) ? (int)a.half : 0);
        const bool ok = (vmask >> s) & (mask_t)1;
        const int es = ok ? e : 0;
        const float th = fmaf(ev[s], s_scl[es], s_loc[es]);
        s_e2 = fmaf(ev[s], ev[s], s_e2);
        if (ok) {
          s_th2 = fmaf(th, th, s_th2);
          if (FAMILY == D3P_FAMILY_LOGREG) zdot = fmaf(xv[s], th, zdot);
          else { float r = xv[s] - th; s_res2 = fmaf(r, r, s_res2); }
        }
        ev[s] = ev[s] * (LINK == D3P_LINK_EXP ? s_scl[es] : s_a[es]);   // u = eps * s'
      }
      if (FAMILY == D3P_FAMILY_LOGREG) zdot = gsum<G>(zdot, gm);
      else s_res2 = gsum<G>(s_res2, gm);
      s_th2 = gsum<G>(s_th2, gm);
      s_e2 = gsum<G>(s_e2, gm);

      float th_b, Lr;
      const float loss_i = example_loss<FAMILY>(a, b, eb, yv, FAMILY == D3P_FAMILY_LOGREG ? zdot : s_res2, s_th2, s_e2,
                                                sum_log_s, a.n_main, th_b, Lr);

      // ---- pass 2: gradient wrt loc (kept in xv), norm -----------------------------------------
      float nrm = 0.f;
#pragma unroll
      for (int s = 0; s < NS; ++s) {
        const int e = glane + G * (s >> 1) + ((s & 1) ? (int)a.half : 0);
        const bool ok = (vmask >> s) & (mask_t)1;
        const int es = ok ? e : 0;
        const float th = (LINK == D3P_LINK_EXP) ? (s_loc[es] + ev[s]) : fmaf(ev[s], s_sa[es], s_loc[es]);
        float h;
        if (FAMILY == D3P_FAMILY_LOGREG) h = Lr * xv[s];
        else h = a.L * a.inv_var * (th - xv[s]);
        const float gl = fmaf(th, a.inv_S, h);
        const float gs = fmaf(gl, ev[s], -(LINK == D3P_LINK_EXP ? a.inv_S : s_bt[es]));
        xv[s] = ok ? gl : 0.f;
        if (ok) {
          nrm = fmaf(gl, gl, fmaf(gs, gs, nrm));
          if (a.px_grads) {
            float* pg = a.px_grads + (size_t)(base + t) * a.P;
            pg[a.loc_off + e] = gl;
            pg[a.rho_off + e] = gs;
          }
        }
      }
      float glb, gsb;
      nrm = intercept_grad(a, b, th_b, eb, Lr, gsum<G>(nrm, gm), glb, gsb);
      const float norm = sqrtf(nrm);
      const float c = 1.0f / fmaxf(1.0f, norm / a.C);      // clip_gradient, d3p/svi.py:121-122

      // ---- pass 3: accumulate the clipped gradient ---------------------------------------------
#pragma unroll
      for (int s = 0; s < NS; ++s) {
        const int e = glane + G * (s >> 1) + ((s & 1) ? (int)a.half : 0);
        const bool ok = (vmask >> s) & (mask_t)1;
        const float bt = (LINK == D3P_LINK_EXP) ? a.inv_S : s_bt[ok ? e : 0];
        const float gs = fmaf(xv[s], ev[s], -bt);
        acc_loc[s] = fmaf(c, xv[s], acc_loc[s]);
        if (ok) acc_rho[s] = fmaf(c, gs, acc_rho[s]);
      }
      if (glane == 0) {
        acc_bloc = fmaf(c, glb, acc_bloc);
        acc_brho = fmaf(c, gsb, acc_brho);
        acc_loss += loss_i;
        acc_cnt += 1.0f;
        if (a.px_norms) a.px_norms[base + t] = norm;
        if (a.px_loss) a.px_loss[base + t] = loss_i;
        if (a.px_grads && a.has_b) {
          float* pg = a.px_grads + (size_t)(base + t) * a.P;
          pg[a.b_loc_off] = glb;
          pg[a.b_rho_off] = gsb;
        }
      }
    }
  }

  // ---- epilogue: groups -> warp -> CTA, fixed order ---------------------------------------------
#pragma unroll
  for (int s = 0; s < NS; ++s) {
#pragma unroll
    for (int o = G; o < 32; o <<= 1) {
      acc_loc[s] += __shfl_xor_sync(0xffffffffu, acc_loc[s], o);
      acc_rho[s] += __shfl_xor_sync(0xffffffffu, acc_rho[s], o);
    }
  }
  acc_bloc = gsum<32>(acc_bloc, 0xffffffffu);
  acc_brho = gsum<32>(acc_brho, 0xffffffffu);
  acc_loss = gsum<32>(acc_loss, 0xffffffffu);
  acc_cnt = gsum<32>(acc_cnt, 0xffffffffu);
  for (int w = 0; w < kStepWarps; ++w) {
    if (warp == w) {
      if (sg == 0) {
#pragma unroll
        for (int s = 0; s < NS; ++s) {
          const uint32_t e = glane + G * (s >> 1) + ((s & 1) ? a.half : 0u);
          if ((vmask >> s) & (mask_t)1) {
            s_acc[a.loc_off + e] += acc_loc[s];
            s_acc[a.rho_off + e] += acc_rho[s];
          }
        }
      }
      if (lane == 0) {
        if (a.has_b) { s_acc[a.b_loc_off] += acc_bloc; s_acc[a.b_rho_off] += acc_brho; }
        s_acc[a.P] += acc_loss;
        s_acc[a.P + 1] += acc_cnt;
      }
    }
    __syncthreads();
  }
  float* out = a.partials + (size_t)blockIdx.x * (a.P + 2);
  for (uint32_t j = threadIdx.x; j < a.P + 2; j += kStepThreads) out[j] = s_acc[j];
}

int32_t launch_meanfield_vec(int family, int link, const StepArgs& a, unsigned grid, cudaStream_t s);

struct Shape { int G, NQ; };

static bool pick_shape(uint32_t half, Shape& sh) {
  // {32, 32}: latent sites of 1025 .. 2048 elements (e.g. the joint AutoDiagonalNormal site of a d = 1024 logistic
  // regression): 64 elements per lane do not fit the register file, the accumulators live in local memory - a
  // correct, slower path for shapes outside the tuned ones
  static const Shape table[] = {{1, 4}, {2, 4}, {4, 4}, {8, 4}, {16, 4}, {32, 4}, {32, 8}, {32, 16}, {32, 32}};
  for (const Shape& s : table)
    if ((uint32_t)(s.G * s.NQ) >= half) { sh = s; return true; }
  return false;
}

static size_t step_smem_bytes(const d3p_meanfield_desc* d, const Shape& sh) {
  size_t nalloc = 2 * (size_t)sh.G * sh.NQ;
  size_t arrays = d->link == D3P_LINK_EXP ? 2 : 5;
  return (arrays * nalloc + d->n_params + 2) * sizeof(float);
}

static uint32_t main_site_len(const d3p_meanfield_desc* d) {
  return d->d + ((d->family == D3P_FAMILY_LOGREG && d->joint_site) ? 1u : 0u);
}

static bool desc_ok(const d3p_meanfield_desc* d) {
  if (!d) return false;
  if (d->family != D3P_FAMILY_LOGREG && d->family != D3P_FAMILY_GAUSS) return false;
  if (d->link != D3P_LINK_EXP && d->link != D3P_LINK_SOFTPLUS) return false;
  if (d->d == 0) return false;
  uint32_t nm = main_site_len(d);
  if ((uint64_t)d->loc_off + nm > d->n_params || (uint64_t)d->rho_off + nm > d->n_params) return false;
  if (d->family == D3P_FAMILY_LOGREG && !d->joint_site &&
      (d->b_loc_off >= d->n_params || d->b_rho_off >= d->n_params)) return false;
  return true;
}

bool meanfield_site(const d3p_meanfield_desc* d, size_t x_row_stride, MeanfieldSite& site) {
  if (!desc_ok(d) || x_row_stride < d->d) return false;
  if (d->family == D3P_FAMILY_GAUSS && !(d->lik_scale > 0.f)) return false;
  site.n_main = main_site_len(d);
  site.half = (site.n_main + 1) / 2;
  site.has_b = (d->family == D3P_FAMILY_LOGREG && !d->joint_site) ? 1 : 0;
  site.inv_var = 0.f; site.log_norm_lik = 0.f;
  if (d->family == D3P_FAMILY_GAUSS) {
    site.inv_var = 1.0f / (d->lik_scale * d->lik_scale);
    site.log_norm_lik = logf(2.50662827463f * d->lik_scale);   // log(sqrt(2 pi) * scale)
  }
  return true;
}

template <int FAMILY, int LINK, int G, int NQ>
static int32_t launch_one(const StepArgs& a, size_t smem, unsigned grid, cudaStream_t s) {
  auto kern = meanfield_step_kernel<FAMILY, LINK, G, NQ>;
  if (smem > 48 * 1024 &&
      cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess)
    return D3P_ERR_CUDA;
  kern<<<grid, kStepThreads, smem, s>>>(a);
  return check_launch();
}

template <int FAMILY, int LINK>
static int32_t launch_shape(const Shape& sh, const StepArgs& a, size_t smem, unsigned grid, cudaStream_t s) {
#define D3P_CASE(g, nq) if (sh.G == g && sh.NQ == nq) return launch_one<FAMILY, LINK, g, nq>(a, smem, grid, s);
  D3P_CASE(1, 4) D3P_CASE(2, 4) D3P_CASE(4, 4) D3P_CASE(8, 4) D3P_CASE(16, 4) D3P_CASE(32, 4) D3P_CASE(32, 8)
  D3P_CASE(32, 16) D3P_CASE(32, 32)
#undef D3P_CASE
  return D3P_ERR_UNSUPPORTED;
}

}  // namespace d3p

using namespace d3p;

extern "C" {

size_t d3p_meanfield_workspace_bytes(const d3p_meanfield_desc* desc, uint32_t* n_partials_out) {
  if (!desc_ok(desc)) return 0;
  uint32_t n_partials = 2u * (uint32_t)sm_count();   // two resident CTAs per SM on the fast path
  if (n_partials_out) *n_partials_out = n_partials;
  return (size_t)n_partials * (desc->n_params + 2) * sizeof(float);
}

}  // extern "C"

int32_t d3p::step_meanfield_impl(const d3p_meanfield_desc* desc, const float* params_d, const float* x_d,
                                 size_t x_row_stride, const int32_t* y_d, const int32_t* idx_d,
                                 const uint8_t* mask_d, const int32_t* num_valid_d, uint32_t B,
                                 uint32_t pos_begin, uint32_t pos_end, const uint32_t* threefry_key_h,
                                 const uint32_t* threefry_key_d, float obs_scale, float C, float* px_norms_d,
                                 float* px_grads_d, float* px_loss_d, void* ws_d, size_t ws_bytes, void* stream) {
  MeanfieldSite site;
  if (!meanfield_site(desc, x_row_stride, site) || !params_d || !x_d || (!threefry_key_h && !threefry_key_d) || !ws_d)
    return D3P_ERR_INVALID_ARGUMENT;
  if (desc->family == D3P_FAMILY_LOGREG && !y_d) return D3P_ERR_INVALID_ARGUMENT;
  if (C == 0.f || obs_scale == 0.f || B == 0 || pos_begin > pos_end || pos_end > B) return D3P_ERR_INVALID_ARGUMENT;
  uint32_t n_partials = 0;
  size_t need = d3p_meanfield_workspace_bytes(desc, &n_partials);
  if (ws_bytes < need) return D3P_ERR_WORKSPACE;
  StepArgs a;
  a.params = params_d; a.x = x_d; a.x_stride = x_row_stride; a.y = y_d; a.idx = idx_d; a.mask = mask_d;
  a.num_valid = num_valid_d; a.B = B; a.pos_begin = pos_begin; a.pos_end = pos_end;
  a.k0 = threefry_key_h ? threefry_key_h[0] : 0u; a.k1 = threefry_key_h ? threefry_key_h[1] : 0u;
  a.key_d = threefry_key_d;
  a.inv_S = 1.0f / obs_scale; a.L = desc->num_obs_total / obs_scale; a.C = C; a.N = desc->num_obs_total;
  a.inv_var = site.inv_var; a.log_norm_lik = site.log_norm_lik;
  a.d = desc->d; a.n_main = site.n_main; a.half = site.half; a.P = desc->n_params;
  a.loc_off = desc->loc_off; a.rho_off = desc->rho_off; a.b_loc_off = desc->b_loc_off; a.b_rho_off = desc->b_rho_off;
  a.has_b = site.has_b;
  a.px_norms = px_norms_d; a.px_grads = px_grads_d; a.px_loss = px_loss_d; a.partials = reinterpret_cast<float*>(ws_d);
  {
    int32_t rc = launch_meanfield_vec(desc->family, desc->link, a, n_partials, (cudaStream_t)stream);
    if (rc != D3P_ERR_UNSUPPORTED) return rc;
  }
  Shape sh;
  if (!pick_shape(a.half, sh)) return D3P_ERR_UNSUPPORTED;
  size_t smem = step_smem_bytes(desc, sh);
  if (smem > 200 * 1024) return D3P_ERR_UNSUPPORTED;
  cudaStream_t s = (cudaStream_t)stream;
  if (desc->family == D3P_FAMILY_LOGREG) {
    if (desc->link == D3P_LINK_EXP) return launch_shape<D3P_FAMILY_LOGREG, D3P_LINK_EXP>(sh, a, smem, n_partials, s);
    return launch_shape<D3P_FAMILY_LOGREG, D3P_LINK_SOFTPLUS>(sh, a, smem, n_partials, s);
  }
  if (desc->link == D3P_LINK_EXP) return launch_shape<D3P_FAMILY_GAUSS, D3P_LINK_EXP>(sh, a, smem, n_partials, s);
  return launch_shape<D3P_FAMILY_GAUSS, D3P_LINK_SOFTPLUS>(sh, a, smem, n_partials, s);
}

extern "C" {

int32_t d3p_dpsvi_step_meanfield(const d3p_meanfield_desc* desc, const float* params_d, const float* x_d,
                                 size_t x_row_stride, const int32_t* y_d, const int32_t* idx_d,
                                 const uint8_t* mask_d, const int32_t* num_valid_d, uint32_t B,
                                 uint32_t pos_begin, uint32_t pos_end, const uint32_t threefry_key_h[2],
                                 float obs_scale, float C, float* px_norms_d, float* px_grads_d, float* px_loss_d,
                                 void* ws_d, size_t ws_bytes, void* stream) {
  if (!threefry_key_h) return D3P_ERR_INVALID_ARGUMENT;
  return step_meanfield_impl(desc, params_d, x_d, x_row_stride, y_d, idx_d, mask_d, num_valid_d, B, pos_begin, pos_end,
                             threefry_key_h, nullptr, obs_scale, C, px_norms_d, px_grads_d, px_loss_d, ws_d, ws_bytes, stream);
}

// Device-key form: the Threefry key (convert_to_jax_rng_key of the step's ChaCha key, d3p_dpsvi_keys_dk) is read from
// device memory by the kernel, so a jitted caller never brings a key to the host.
int32_t d3p_dpsvi_step_meanfield_dk(const d3p_meanfield_desc* desc, const float* params_d, const float* x_d,
                                    size_t x_row_stride, const int32_t* y_d, const int32_t* idx_d,
                                    const uint8_t* mask_d, const int32_t* num_valid_d, uint32_t B,
                                    uint32_t pos_begin, uint32_t pos_end, const uint32_t* threefry_key_d,
                                    float obs_scale, float C, float* px_norms_d, float* px_grads_d, float* px_loss_d,
                                    void* ws_d, size_t ws_bytes, void* stream) {
  if (!threefry_key_d) return D3P_ERR_INVALID_ARGUMENT;
  return step_meanfield_impl(desc, params_d, x_d, x_row_stride, y_d, idx_d, mask_d, num_valid_d, B, pos_begin, pos_end,
                             nullptr, threefry_key_d, obs_scale, C, px_norms_d, px_grads_d, px_loss_d, ws_d, ws_bytes, stream);
}

}  // extern "C"
