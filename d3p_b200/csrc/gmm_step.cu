// K5c: fused DP-SVI step for the Gaussian-mixture model of examples/gaussian_mixture_model.py:51-85
// with the d3p.gmm.GaussianMixture likelihood (d3p/gmm.py:71-86): per-example gradient, norm, clip and
// clipped sum (d3p/svi.py:238-348) without a [B, P] tensor.
//
// Every example draws its own guide sample (d3p/svi.py:283-290):
//   pis  ~ Dirichlet(exp(alpha_log))      jax.random.dirichlet = softmax(loggamma(alpha)), K Marsaglia-Tsang
//                                         draws + the implicit-reparametrisation derivative of each
//   mus  ~ Normal(mus_loc, 1)   [K, d]    K d Threefry normals
//   sigs ~ InverseGamma(1, 1)   [K, d]    K d Marsaglia-Tsang gamma(1) draws with per-element keys
// i.e. ~10 Threefry-2x32-20 calls per data float x K: the kernel is ALU-bound by construction (SURVEY
// 8(d)); HBM traffic is one 4 d byte row per example.
//
// One CTA works on one example at a time (persistent grid):
//   A1  sigs: lane-level work queue over the rejection sampler (a lane that accepts moves on to its next
//       element immediately, so rejected draws do not idle the other 31 lanes)            -> smem S
//   A2  mus noise, (x - mu) / sig^2, component log-density terms                          -> smem T, PM, A (= S)
//   B   Dirichlet sample + implicit gradients (threads k < K), row sums, logsumexp, responsibilities,
//       gradient wrt alpha_log
//   C   gradient wrt mus_loc, squared norm, clip factor, accumulation into the CTA's partial row
// Every (k, j) is owned by one thread, so the partial row is accumulated without atomics and the
// result is run-to-run deterministic.
#include "common.cuh"
#include "jrandom.cuh"
#include "launch.cuh"

namespace d3p {

constexpr int kGmmThreads = 256;
constexpr int kGmmMaxK = 256;

struct GmmArgs {
  const float* params; const float* x; size_t x_stride; const int32_t* idx; const uint8_t* mask;
  const int32_t* num_valid;
  uint32_t B, pos_begin, pos_end, k0, k1;
  const uint32_t* key_d;      // *_dk entry point: Threefry key in device memory (else nullptr)
  uint32_t K, d, P, alpha_off, mus_off;
  float N, inv_S, C;
  float* px_norms; float* px_grads; float* px_loss; float* partials;
};

D3P_D float digamma_f32(float x) {      // x > 0
  float r = 0.f;
  while (x < 6.0f) { r -= 1.0f / x; x += 1.0f; }
  const float i = 1.0f / x, i2 = i * i;
  // ln x - 1/(2x) - 1/(12x^2) + 1/(120x^4) - 1/(252x^6) + 1/(240x^8)
  return r + logf(x) - 0.5f * i - i2 * (1.0f / 12.0f - i2 * (1.0f / 120.0f - i2 * (1.0f / 252.0f - i2 * (1.0f / 240.0f))));
}

// lax.random_gamma_grad(a, x) as lowered by XLA (RandomGammaGrad, xla/client/lib/math.cc): d sample / d alpha
D3P_D float gamma_grad_f32(float a, float x) {
  const float eps = 1.1920929e-07f;
  if (x == 0.f) return 0.f;
  const bool use_igammac = (x > 1.0f) && (x > a);
  if (!use_igammac) {       // IgammaSeries<SAMPLE_DERIVATIVE>
    float r = a, c = 1.0f, ans = 1.0f, dc_da = 0.f, dans_da = 0.f;
    for (int it = 0; it < 2000; ++it) {
      r += 1.0f;
      dc_da = dc_da * (x / r) + (-1.0f * c * x) / (r * r);
      dans_da = dans_da + dc_da;
      c = c * (x / r);
      ans = ans + c;
      if (!(fabsf(dc_da / dans_da) > eps)) break;
    }
    const float dlogax_da = logf(x) - digamma_f32(a + 1.0f);
    return -(dans_da + ans * dlogax_da) * x / a;
  }
  // IgammacContinuedFraction<SAMPLE_DERIVATIVE>, negated
  float y = 1.0f - a, z = x + y + 1.0f, cc = 0.f;
  float pkm2 = 1.0f, qkm2 = x, pkm1 = x + 1.0f, qkm1 = z * x;
  float ans = pkm1 / qkm1;
  float dpkm2 = 0.f, dqkm2 = 0.f, dpkm1 = 0.f, dqkm1 = -x;
  float dans = (dpkm1 - ans * dqkm1) / qkm1;
  for (int it = 0; it < 2000; ++it) {
    cc += 1.0f; y += 1.0f; z += 2.0f;
    const float yc = y * cc;
    const float pk = pkm1 * z - pkm2 * yc;
    const float qk = qkm1 * z - qkm2 * yc;
    const bool nz = qk != 0.f;
    if (nz) ans = pk / qk;
    const float dpk = dpkm1 * z - pkm1 - dpkm2 * yc + pkm2 * cc;
    const float dqk = dqkm1 * z - qkm1 - dqkm2 * yc + qkm2 * cc;
    const float dans_new = nz ? (dpk - ans * dqk) / qk : dans;
    const float grad_cond = nz ? fabsf(dans_new - dans) : 1.0f;
    dans = dans_new;
    pkm2 = pkm1; pkm1 = pk; qkm2 = qkm1; qkm1 = qk;
    dpkm2 = dpkm1; dqkm2 = dqkm1; dpkm1 = dpk; dqkm1 = dqk;
    if (fabsf(pk) > 1.0f / eps) {
      pkm2 *= eps; pkm1 *= eps; qkm2 *= eps; qkm1 *= eps;
      dpkm2 *= eps; dqkm2 *= eps; dpkm1 *= eps; dqkm1 *= eps;
    }
    if (!(grad_cond > eps)) break;
  }
  const float dlogax_da = logf(x) - digamma_f32(a);
  return (dans + ans * dlogax_da) * x;      // = -(-(dans + ans * dlogax_da) * x)
}

template <int NW>
D3P_D float block_sum(float v, float* red, int lane, int warp) {   // fixed order; all threads get the total
  v = group_sum<32>(v);
  __syncthreads();
  if (lane == 0) red[warp] = v;
  __syncthreads();
  float s = 0.f;
#pragma unroll
  for (int w = 0; w < NW; ++w) s += red[w];
  return s;
}

template <int NW>
D3P_D float block_max(float v, float* red, int lane, int warp) {   // all threads get the maximum
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
  __syncthreads();
  if (lane == 0) red[warp] = v;
  __syncthreads();
  float s = red[0];
#pragma unroll
  for (int w = 1; w < NW; ++w) s = fmaxf(s, red[w]);
  return s;
}

__global__ void __launch_bounds__(kGmmThreads, 2) gmm_step_kernel(GmmArgs a) {
  extern __shared__ float smem[];
  constexpr int NW = kGmmThreads / 32;
  const uint32_t K = a.K, d = a.d, n = a.K * a.d;
  float* S = smem;              // [n]  sig, then the component log-density term
  float* T = S + n;             // [n]  (x - mu) / sig^2
  float* PM = T + n;            // [n]  mu / 100
  float* xs = PM + n;           // [d]
  float* alpha_s = xs + d;      // [K]  exp(alpha_log)
  float* cst = alpha_s + K;     // [K]  digamma(sum alpha) - digamma(alpha_k)
  float* comp = cst + K;        // [K]
  float* lpi = comp + K;        // [K]  log pi (clipped)
  float* wv = lpi + K;          // [K]  clip weight * pi / pi_clipped
  float* dlg = wv + K;          // [K]  d log g_k / d alpha_k
  float* pi_s = dlg + K;        // [K]  pi (unclipped)
  float* ga = pi_s + K;         // [K]  gradient wrt alpha_log (unscaled by c)
  float* red = ga + K;          // [NW + 4]
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;

  float* part = a.partials + (size_t)blockIdx.x * (a.P + 2);
  for (uint32_t j = tid; j < a.P + 2; j += kGmmThreads) part[j] = 0.f;
  // per-step constants of the guide's Dirichlet
  float asum_part = 0.f, lgam_part = 0.f;
  for (uint32_t k = tid; k < K; k += kGmmThreads) {
    const float al = expf(a.params[a.alpha_off + k]);
    alpha_s[k] = al;
    asum_part += al;
    lgam_part += lgammaf(al);
  }
  const float alpha_sum = block_sum<NW>(asum_part, red, lane, warp);
  const float lgam_sum = block_sum<NW>(lgam_part, red, lane, warp);
  const float dig_sum = digamma_f32(alpha_sum);
  for (uint32_t k = tid; k < K; k += kGmmThreads) cst[k] = dig_sum - digamma_f32(alpha_s[k]);
  const float log_norm_q_pis = lgammaf(alpha_sum) - lgam_sum;       // + lgamma(sum) - sum lgamma
  const float lgamma_K = lgammaf((float)K);
  __syncthreads();

  const TfKey Kk = tf_key_arg(a.k0, a.k1, a.key_d);
  const uint32_t nv = a.num_valid ? (uint32_t)max(*a.num_valid, 0) : 0xffffffffu;
  const uint32_t half = (n + 1) / 2;
  const float kLogSqrt2Pi = 0.918938533f, kLog10Sqrt2Pi = 3.22152363f;
  float acc_loss = 0.f, acc_cnt = 0.f;

  for (uint32_t p = a.pos_begin + blockIdx.x; p < a.pos_end; p += gridDim.x) {
    const bool valid = (p < nv) && (!a.mask || a.mask[p]);     // CTA-uniform
    if (!valid) continue;
    const uint32_t row = a.idx ? (uint32_t)a.idx[p] : p;
    for (uint32_t j = tid; j < d; j += kGmmThreads) xs[j] = a.x[(size_t)row * a.x_stride + j];
    // per-example keys: key_p -> (_, guide_seed) -> site keys of pis, mus, sigs (one split each)
    TfKey rng = guide_rng(tf_example_key(Kk, a.B, p));
    const TfKey k_pis = next_site(rng), k_mus = next_site(rng), k_sigs = next_site(rng);

    // ---- A1: sigs[m] = 1 / gamma(split(k_sigs, n)[m], 1); lane-level work queue ---------------------------
    {
      const float dd = 1.0f - 1.0f / 3.0f, cc = (1.0f / 3.0f) / sqrtf(dd);
      uint32_t m = tid;
      TfKey key;
      bool have = m < n;
      if (have) {
        TfKey ek(tf_split_word(k_sigs, n, 2u * m), tf_split_word(k_sigs, n, 2u * m + 1u)), sub;
        tf_split2(ek, key, sub);            // u_boost (from `sub`) is unused for alpha >= 1
      }
      while (__any_sync(0xffffffffu, have)) {
        if (have) {
          float X, V, U;
          mt_propose(key, cc, X, V, U);
          if (!mt_reject(X, V, U, dd)) {
            S[m] = 1.0f / (dd * V);         // InverseGamma = PowerTransform(-1) of the Gamma draw
            m += kGmmThreads;
            have = m < n;
            if (have) {
              TfKey ek(tf_split_word(k_sigs, n, 2u * m), tf_split_word(k_sigs, n, 2u * m + 1u)), sub;
              tf_split2(ek, key, sub);
            }
          }
        }
      }
    }
    __syncthreads();

    // ---- A2: mus, per-element terms; Threefry call c yields the noise of elements c and c + half ----------
    float s_mu2 = 0.f, s_e2 = 0.f;
    for (uint32_t c = tid; c < half; c += kGmmThreads) {
      uint32_t y0, y1;
      const uint32_t m1 = c + half;
      threefry2x32(k_mus, c, m1 < n ? m1 : 0u, y0, y1);
#pragma unroll
      for (int h = 0; h < 2; ++h) {
        const uint32_t m = h ? m1 : c;
        if (m >= n) break;
        const float eps = bits_to_normal_fast(h ? y1 : y0);       // value-only use: MUFU.LG2 form (<= 2e-7 relative)
        const uint32_t j = m % d;
        const float mu = a.params[a.mus_off + m] + eps;
        const float sg = S[m];
        const float zs = (xs[j] - mu) / sg;
        S[m] = -0.5f * zs * zs - logf(2.50662827f * sg);      // Normal.log_prob: -log(sqrt(2 pi) * scale)
        T[m] = (xs[j] - mu) / (sg * sg);
        PM[m] = mu * 0.01f;                                   // -d log N(mu; 0, 10) / d mu
        s_mu2 = fmaf(mu, mu, s_mu2);
        s_e2 = fmaf(eps, eps, s_e2);
      }
    }
    // ---- B (part 1): Dirichlet draw and implicit gradients, one thread per component ----------------------
    for (uint32_t k = tid; k < K; k += kGmmThreads) {
      TfKey ek(tf_split_word(k_pis, K, 2u * k), tf_split_word(k_pis, K, 2u * k + 1u));
      const float lg = loggamma_one(ek, alpha_s[k]);
      float g = expf(lg);
      if (g == 0.f) g = 1.17549435e-38f;
      comp[k] = lg;                                   // staged: log g_k
      dlg[k] = gamma_grad_f32(alpha_s[k], g) / g;
    }
    const float sum_mu2 = block_sum<NW>(s_mu2, red, lane, warp);
    const float sum_e2 = block_sum<NW>(s_e2, red, lane, warp);
    // softmax over log g: K <= 256 = one component per thread, fixed-order block reductions (the former
    // thread-serial loops over K on all 256 threads were 11 % of the kernel's instructions)
    const float lg_own = tid < K ? comp[tid] : -3.4e38f;
    const float mx = block_max<NW>(lg_own, red, lane, warp);
    const float den = block_sum<NW>(tid < K ? expf(lg_own - mx) : 0.f, red, lane, warp);
    __syncthreads();
    for (uint32_t k = tid; k < K; k += kGmmThreads) {
      const float pi = expf(comp[k] - mx) / den;
      const float tiny = 1.17549435e-38f, omax = 0.99999988079071044921875f;
      const float pc = fminf(fmaxf(pi, tiny), omax);
      const float w = (pi > tiny ? 1.0f : (pi == tiny ? 0.5f : 0.f)) * (pi < omax ? 1.0f : (pi == omax ? 0.5f : 0.f));
      pi_s[k] = pi;
      lpi[k] = logf(pc);
      wv[k] = w * pi / pc;
    }
    __syncthreads();
    // row sums: comp_k = sum_j A[k, j] + log pi_k  (warp per row, fixed shuffle order)
    for (uint32_t k = warp; k < K; k += NW) {
      float s = 0.f;
      for (uint32_t j = lane; j < d; j += 32) s += S[k * d + j];
      s = group_sum<32>(s);
      if (lane == 0) comp[k] = s + lpi[k];
    }
    __syncthreads();
    const float c_own = tid < K ? comp[tid] : -3.4e38f;
    const float cmx = block_max<NW>(c_own, red, lane, warp);
    const float e_own = tid < K ? expf(c_own - cmx) : 0.f;
    const float cden = block_sum<NW>(e_own, red, lane, warp);
    const float loglik = cmx + logf(cden);
    // D_m = (alpha_m - 1) - N r_m ; sumDw = sum_m D_m w'_m ; log q(pis) = sum (alpha - 1) log pi + norm
    float dw_own = 0.f, lq_own = 0.f;
    if (tid < K) {
      const float r = e_own / cden;
      const float D = (alpha_s[tid] - 1.0f) - a.N * r;
      dw_own = D * wv[tid];
      lq_own = (alpha_s[tid] - 1.0f) * lpi[tid];
    }
    const float sumDw = block_sum<NW>(dw_own, red, lane, warp);
    const float lq_pis = block_sum<NW>(lq_own, red, lane, warp) + log_norm_q_pis;
    __syncthreads();
    float nrm_part = 0.f;
    for (uint32_t k = tid; k < K; k += kGmmThreads) {
      const float r = expf(comp[k] - cmx) / cden;
      const float D = (alpha_s[k] - 1.0f) - a.N * r;
      const float dL_dalpha = lpi[k] + cst[k] + dlg[k] * (D * wv[k] - pi_s[k] * sumDw);
      const float g = a.inv_S * alpha_s[k] * dL_dalpha;
      ga[k] = g;
      nrm_part = fmaf(g, g, nrm_part);
      comp[k] = r;                                    // staged: responsibility
    }
    __syncthreads();
    // ---- C: gradient wrt mus_loc, norm, clip, accumulate --------------------------------------------------
    for (uint32_t m = tid; m < n; m += kGmmThreads) {
      // L = -elbo: dL/dmu = mu / 100 - N r_k (x - mu) / sig^2 ; g = dL / obs_scale
      const float g = a.inv_S * (PM[m] - a.N * comp[m / d] * T[m]);
      T[m] = g;
      nrm_part = fmaf(g, g, nrm_part);
    }
    const float nrm2 = block_sum<NW>(nrm_part, red, lane, warp);
    const float norm = sqrtf(nrm2);
    const float cfac = 1.0f / fmaxf(1.0f, norm / a.C);
    for (uint32_t m = tid; m < n; m += kGmmThreads) {
      part[a.mus_off + m] = fmaf(cfac, T[m], part[a.mus_off + m]);
      if (a.px_grads) a.px_grads[(size_t)p * a.P + a.mus_off + m] = T[m];
    }
    for (uint32_t k = tid; k < K; k += kGmmThreads) {
      part[a.alpha_off + k] = fmaf(cfac, ga[k], part[a.alpha_off + k]);
      if (a.px_grads) a.px_grads[(size_t)p * a.P + a.alpha_off + k] = ga[k];
    }
    if (tid == 0) {
      // -elbo = -[log p(pis) + log p(mus) + N loglik - log q(pis) - log q(mus)]
      const float log_p_mus = -0.5f * sum_mu2 * 0.01f - (float)n * kLog10Sqrt2Pi;
      const float log_q_mus = -0.5f * sum_e2 - (float)n * kLogSqrt2Pi;
      const float loss = -(lgamma_K + log_p_mus + a.N * loglik - lq_pis - log_q_mus);
      const float loss_s = loss;                                  // obs_scale * (1 / obs_scale) * (-elbo)
      acc_loss += loss_s;
      acc_cnt += 1.0f;
      if (a.px_norms) a.px_norms[p] = norm;
      if (a.px_loss) a.px_loss[p] = loss_s;
    }
    __syncthreads();
  }
  if (tid == 0) { part[a.P] = acc_loss; part[a.P + 1] = acc_cnt; }
}

// ---- DPSVI.evaluate for the mixture (d3p/svi.py:436-449 -> numpyro SVI.evaluate -> Trace_ELBO.loss on the whole batch) --
// ONE guide draw (pis, mus, sigs) from numpyro's rng_key_eval, then the log-likelihood of every example of the batch under
// it, plate scale N / B:   loss = -[log p(pis) + log p(mus) + (N / B) sum_i log p(x_i | pis, mus, sigs) - log q(pis) - log q(mus)].
struct GmmEvalArgs {
  const float* params; const float* x; size_t x_stride; const int32_t* idx;
  uint32_t B, k0, k1;
  uint32_t K, d, alpha_off, mus_off;
  float N;
  float* aT;        // [d][K]  -1 / (2 sig^2)
  float* muT;       // [d][K]
  float* ck;        // [K]     sum_j -log(sqrt(2 pi) sig_kj) + log pi_k
  float* terms;     // [1]     log p(pis) + log p(mus) - log q(pis) - log q(mus)
  float* partial;   // [grid]  per-CTA sums of log p(x_i | ...)
  float* loss;
};

// one CTA: the guide draw, with the same device samplers (and the same key plumbing) as the step kernel
__global__ void __launch_bounds__(kGmmThreads) gmm_eval_draw_kernel(GmmEvalArgs a) {
  extern __shared__ float smem[];
  constexpr int NW = kGmmThreads / 32;
  const uint32_t K = a.K, d = a.d, n = a.K * a.d;
  float* S = smem;              // [n] sig, then -log(sqrt(2 pi) sig)
  float* alpha_s = S + n;       // [K]
  float* comp = alpha_s + K;    // [K] log g, then row sums
  float* lpi = comp + K;        // [K]
  float* red = lpi + K;         // [NW + 4]
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  float asum_part = 0.f, lgam_part = 0.f;
  for (uint32_t k = tid; k < K; k += kGmmThreads) {
    const float al = expf(a.params[a.alpha_off + k]);
    alpha_s[k] = al;
    asum_part += al;
    lgam_part += lgammaf(al);
  }
  const float alpha_sum = block_sum<NW>(asum_part, red, lane, warp);
  const float lgam_sum = block_sum<NW>(lgam_part, red, lane, warp);
  const float log_norm_q_pis = lgammaf(alpha_sum) - lgam_sum;
  __syncthreads();
  TfKey rng = guide_rng(TfKey(a.k0, a.k1));
  const TfKey k_pis = next_site(rng), k_mus = next_site(rng), k_sigs = next_site(rng);
  {   // sigs[m] = 1 / gamma(split(k_sigs, n)[m], 1): lane-level work queue (see gmm_step_kernel A1)
    const float dd = 1.0f - 1.0f / 3.0f, cc = (1.0f / 3.0f) / sqrtf(dd);
    uint32_t m = tid;
    TfKey key;
    bool have = m < n;
    if (have) {
      TfKey ek(tf_split_word(k_sigs, n, 2u * m), tf_split_word(k_sigs, n, 2u * m + 1u)), sub;
      tf_split2(ek, key, sub);
    }
    while (__any_sync(0xffffffffu, have)) {
      if (have) {
        float X, V, U;
        mt_propose(key, cc, X, V, U);
        if (!mt_reject(X, V, U, dd)) {
          S[m] = 1.0f / (dd * V);
          m += kGmmThreads;
          have = m < n;
          if (have) {
            TfKey ek(tf_split_word(k_sigs, n, 2u * m), tf_split_word(k_sigs, n, 2u * m + 1u)), sub;
            tf_split2(ek, key, sub);
          }
        }
      }
    }
  }
  __syncthreads();
  const uint32_t half = (n + 1) / 2;
  float s_mu2 = 0.f, s_e2 = 0.f;
  for (uint32_t c = tid; c < half; c += kGmmThreads) {
    uint32_t y0, y1;
    const uint32_t m1 = c + half;
    threefry2x32(k_mus, c, m1 < n ? m1 : 0u, y0, y1);
#pragma unroll
    for (int h = 0; h < 2; ++h) {
      const uint32_t m = h ? m1 : c;
      if (m >= n) break;
      const float eps = bits_to_normal_fast(h ? y1 : y0);
      const uint32_t k = m / d, j = m % d;
      const float mu = a.params[a.mus_off + m] + eps;
      const float sg = S[m];
      a.muT[(size_t)j * K + k] = mu;
      a.aT[(size_t)j * K + k] = -0.5f / (sg * sg);
      S[m] = -logf(2.50662827f * sg);
      s_mu2 = fmaf(mu, mu, s_mu2);
      s_e2 = fmaf(eps, eps, s_e2);
    }
  }
  for (uint32_t k = tid; k < K; k += kGmmThreads) {
    TfKey ek(tf_split_word(k_pis, K, 2u * k), tf_split_word(k_pis, K, 2u * k + 1u));
    comp[k] = loggamma_one(ek, alpha_s[k]);
  }
  const float sum_mu2 = block_sum<NW>(s_mu2, red, lane, warp);
  const float sum_e2 = block_sum<NW>(s_e2, red, lane, warp);
  const float lg_own = tid < K ? comp[tid] : -3.4e38f;
  const float mx = block_max<NW>(lg_own, red, lane, warp);
  const float den = block_sum<NW>(tid < K ? expf(lg_own - mx) : 0.f, red, lane, warp);
  __syncthreads();
  float lq_own = 0.f;
  for (uint32_t k = tid; k < K; k += kGmmThreads) {
    const float pi = expf(comp[k] - mx) / den;
    const float pc = fminf(fmaxf(pi, 1.17549435e-38f), 0.99999988079071044921875f);
    lpi[k] = logf(pc);
    lq_own += (alpha_s[k] - 1.0f) * lpi[k];
  }
  const float lq_pis = block_sum<NW>(lq_own, red, lane, warp) + log_norm_q_pis;
  __syncthreads();
  for (uint32_t k = warp; k < K; k += NW) {
    float s = 0.f;
    for (uint32_t j = lane; j < d; j += 32) s += S[k * d + j];
    s = group_sum<32>(s);
    if (lane == 0) a.ck[k] = s + lpi[k];
  }
  if (tid == 0) {
    const float kLogSqrt2Pi = 0.918938533f, kLog10Sqrt2Pi = 3.22152363f;
    const float log_p_mus = -0.5f * sum_mu2 * 0.01f - (float)n * kLog10Sqrt2Pi;
    const float log_q_mus = -0.5f * sum_e2 - (float)n * kLogSqrt2Pi;
    a.terms[0] = lgammaf((float)K) + log_p_mus - lq_pis - log_q_mus;
  }
}

// warp per example, lanes over the components: comp_k = ck_k + sum_j aT[j][k] (x_j - muT[j][k])^2, logsumexp over k
constexpr int kGmmEvalMaxKPerLane = kGmmMaxK / 32;
__global__ void __launch_bounds__(kGmmThreads) gmm_eval_loglik_kernel(GmmEvalArgs a) {
  extern __shared__ float smem[];
  constexpr int NW = kGmmThreads / 32;
  const uint32_t K = a.K, d = a.d, n = a.K * a.d;
  float* aT = smem;             // [d][K]
  float* muT = aT + n;          // [d][K]
  float* ck = muT + n;          // [K]
  float* xs = ck + K;           // [NW][d]
  __shared__ float wsum[NW];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  for (uint32_t i = tid; i < n; i += kGmmThreads) { aT[i] = a.aT[i]; muT[i] = a.muT[i]; }
  for (uint32_t k = tid; k < K; k += kGmmThreads) ck[k] = a.ck[k];
  __syncthreads();
  float* x_w = xs + (size_t)warp * d;
  float acc_ll = 0.f;
  for (uint32_t p = blockIdx.x * NW + warp; p < a.B; p += gridDim.x * NW) {
    const uint32_t row = a.idx ? (uint32_t)a.idx[p] : p;
    __syncwarp();
    for (uint32_t j = lane; j < d; j += 32) x_w[j] = a.x[(size_t)row * a.x_stride + j];
    __syncwarp();
    float acc[kGmmEvalMaxKPerLane];
#pragma unroll
    for (int t = 0; t < kGmmEvalMaxKPerLane; ++t) acc[t] = 0.f;
    for (uint32_t j = 0; j < d; ++j) {
      const float xj = x_w[j];
#pragma unroll
      for (int t = 0; t < kGmmEvalMaxKPerLane; ++t) {
        const uint32_t k = lane + 32u * t;
        if (k < K) { const float df = xj - muT[j * K + k]; acc[t] = fmaf(aT[j * K + k] * df, df, acc[t]); }
      }
    }
    float mx = -3.4e38f;
#pragma unroll
    for (int t = 0; t < kGmmEvalMaxKPerLane; ++t) {
      const uint32_t k = lane + 32u * t;
      acc[t] = k < K ? acc[t] + ck[k] : -3.4e38f;
      mx = fmaxf(mx, acc[t]);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
    float se = 0.f;
#pragma unroll
    for (int t = 0; t < kGmmEvalMaxKPerLane; ++t) se += (lane + 32u * t < K) ? expf(acc[t] - mx) : 0.f;
    se = group_sum<32>(se);
    acc_ll += mx + logf(se);
  }
  if (lane == 0) wsum[warp] = acc_ll;
  __syncthreads();
  if (tid == 0) {
    float s = 0.f;
#pragma unroll
    for (int w = 0; w < NW; ++w) s += wsum[w];
    a.partial[blockIdx.x] = s;
  }
}

__global__ void gmm_eval_finish_kernel(GmmEvalArgs a, uint32_t n_partial) {
  if (threadIdx.x != 0 || blockIdx.x != 0) return;
  float s = 0.f;
  for (uint32_t i = 0; i < n_partial; ++i) s += a.partial[i];
  *a.loss = -(a.terms[0] + (a.N / (float)a.B) * s);
}

static size_t gmm_smem_bytes(uint32_t K, uint32_t d) {
  return ((size_t)3 * K * d + d + 9 * (size_t)K + kGmmThreads / 32 + 4) * sizeof(float);
}

static bool gmm_supported(const d3p_gmm_desc* g) {
  return g && g->K >= 1 && g->K <= (uint32_t)kGmmMaxK && g->d >= 1 && gmm_smem_bytes(g->K, g->d) <= 110 * 1024;
}

}  // namespace d3p

using namespace d3p;

extern "C" size_t d3p_gmm_workspace_bytes(const d3p_gmm_desc* desc, uint32_t* n_partials_out) {
  if (!gmm_supported(desc)) return 0;
  const uint32_t n_part = 2u * (uint32_t)sm_count();
  if (n_partials_out) *n_partials_out = n_part;
  return (size_t)n_part * (desc->n_params + 2) * sizeof(float);
}

int32_t d3p::step_gmm_impl(const d3p_gmm_desc* desc, const float* params_d, const float* x_d, size_t x_row_stride,
                           const int32_t* idx_d, const uint8_t* mask_d, const int32_t* num_valid_d, uint32_t B,
                           uint32_t pos_begin, uint32_t pos_end, const uint32_t* threefry_key_h,
                           const uint32_t* threefry_key_d, float obs_scale, float C, float* px_norms_d,
                           float* px_grads_d, float* px_loss_d, void* ws_d, size_t ws_bytes, void* stream) {
  if (!desc || !params_d || !x_d || (!threefry_key_h && !threefry_key_d) || !ws_d) return D3P_ERR_INVALID_ARGUMENT;
  if (!gmm_supported(desc)) return D3P_ERR_UNSUPPORTED;
  if (pos_end > B || pos_begin > pos_end || !(C > 0.f) || !(obs_scale != 0.f)) return D3P_ERR_INVALID_ARGUMENT;
  const uint32_t n_part = 2u * (uint32_t)sm_count();
  if (ws_bytes < (size_t)n_part * (desc->n_params + 2) * sizeof(float)) return D3P_ERR_WORKSPACE;
  GmmArgs a;
  a.params = params_d; a.x = x_d; a.x_stride = x_row_stride; a.idx = idx_d; a.mask = mask_d; a.num_valid = num_valid_d;
  a.B = B; a.pos_begin = pos_begin; a.pos_end = pos_end; a.k0 = threefry_key_h ? threefry_key_h[0] : 0u;
  a.k1 = threefry_key_h ? threefry_key_h[1] : 0u; a.key_d = threefry_key_d;
  a.K = desc->K; a.d = desc->d; a.P = desc->n_params; a.alpha_off = desc->alpha_off; a.mus_off = desc->mus_off;
  a.N = desc->num_obs_total; a.inv_S = 1.0f / obs_scale; a.C = C;
  a.px_norms = px_norms_d; a.px_grads = px_grads_d; a.px_loss = px_loss_d; a.partials = static_cast<float*>(ws_d);
  const size_t smem = gmm_smem_bytes(a.K, a.d);
  if (smem > 48 * 1024 &&
      cudaFuncSetAttribute(gmm_step_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess)
    return D3P_ERR_CUDA;
  gmm_step_kernel<<<n_part, kGmmThreads, smem, (cudaStream_t)stream>>>(a);
  return check_launch();
}

extern "C" int32_t d3p_dpsvi_step_gmm(const d3p_gmm_desc* desc, const float* params_d, const float* x_d,
                                      size_t x_row_stride, const int32_t* idx_d, const uint8_t* mask_d,
                                      const int32_t* num_valid_d, uint32_t B, uint32_t pos_begin, uint32_t pos_end,
                                      const uint32_t threefry_key_h[2], float obs_scale, float C, float* px_norms_d,
                                      float* px_grads_d, float* px_loss_d, void* ws_d, size_t ws_bytes, void* stream) {
  if (!threefry_key_h) return D3P_ERR_INVALID_ARGUMENT;
  return step_gmm_impl(desc, params_d, x_d, x_row_stride, idx_d, mask_d, num_valid_d, B, pos_begin, pos_end, threefry_key_h,
                       nullptr, obs_scale, C, px_norms_d, px_grads_d, px_loss_d, ws_d, ws_bytes, stream);
}

extern "C" int32_t d3p_dpsvi_step_gmm_dk(const d3p_gmm_desc* desc, const float* params_d, const float* x_d,
                                         size_t x_row_stride, const int32_t* idx_d, const uint8_t* mask_d,
                                         const int32_t* num_valid_d, uint32_t B, uint32_t pos_begin, uint32_t pos_end,
                                         const uint32_t* threefry_key_d, float obs_scale, float C, float* px_norms_d,
                                         float* px_grads_d, float* px_loss_d, void* ws_d, size_t ws_bytes, void* stream) {
  if (!threefry_key_d) return D3P_ERR_INVALID_ARGUMENT;
  return step_gmm_impl(desc, params_d, x_d, x_row_stride, idx_d, mask_d, num_valid_d, B, pos_begin, pos_end, nullptr,
                       threefry_key_d, obs_scale, C, px_norms_d, px_grads_d, px_loss_d, ws_d, ws_bytes, stream);
}

extern "C" size_t d3p_elbo_evaluate_gmm_workspace_bytes(const d3p_gmm_desc* desc) {
  if (!gmm_supported(desc)) return 0;
  return ((size_t)2 * desc->K * desc->d + desc->K + 4 + 2 * (size_t)sm_count()) * sizeof(float);
}

// DPSVI.evaluate for the mixture: threefry_key_h = numpyro's rng_key_eval (d3p/svi.py:447 + SVI.evaluate's split).
extern "C" int32_t d3p_elbo_evaluate_gmm(const d3p_gmm_desc* desc, const float* params_d, const float* x_d,
                                         size_t x_row_stride, const int32_t* idx_d, uint32_t B,
                                         const uint32_t threefry_key_h[2], float* loss_d, void* ws_d, size_t ws_bytes,
                                         void* stream) {
  if (!desc || !params_d || !x_d || !threefry_key_h || !loss_d || !ws_d || B == 0) return D3P_ERR_INVALID_ARGUMENT;
  if (!gmm_supported(desc)) return D3P_ERR_UNSUPPORTED;
  if (ws_bytes < d3p_elbo_evaluate_gmm_workspace_bytes(desc)) return D3P_ERR_WORKSPACE;
  const uint32_t K = desc->K, d = desc->d, n = K * d;
  GmmEvalArgs a;
  a.params = params_d; a.x = x_d; a.x_stride = x_row_stride; a.idx = idx_d; a.B = B;
  a.k0 = threefry_key_h[0]; a.k1 = threefry_key_h[1];
  a.K = K; a.d = d; a.alpha_off = desc->alpha_off; a.mus_off = desc->mus_off; a.N = desc->num_obs_total;
  float* w = static_cast<float*>(ws_d);
  a.aT = w; a.muT = w + n; a.ck = w + 2 * (size_t)n; a.terms = a.ck + K; a.partial = a.terms + 4; a.loss = loss_d;
  cudaStream_t s = (cudaStream_t)stream;
  const size_t smem1 = ((size_t)n + 3 * K + kGmmThreads / 32 + 4) * sizeof(float);
  const size_t smem2 = ((size_t)2 * n + K + (size_t)(kGmmThreads / 32) * d) * sizeof(float);
  if (smem2 > 200 * 1024) return D3P_ERR_UNSUPPORTED;
  if (smem1 > 48 * 1024 &&
      cudaFuncSetAttribute(gmm_eval_draw_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem1) != cudaSuccess)
    return D3P_ERR_CUDA;
  if (smem2 > 48 * 1024 &&
      cudaFuncSetAttribute(gmm_eval_loglik_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem2) != cudaSuccess)
    return D3P_ERR_CUDA;
  gmm_eval_draw_kernel<<<1, kGmmThreads, smem1, s>>>(a);
  unsigned grid = (B + kGmmThreads / 32 - 1) / (kGmmThreads / 32);
  const unsigned cap = 2u * (unsigned)sm_count();
  if (grid > cap) grid = cap;
  gmm_eval_loglik_kernel<<<grid, kGmmThreads, smem2, s>>>(a);
  gmm_eval_finish_kernel<<<1, 32, 0, s>>>(a, grid);
  return check_launch();
}
