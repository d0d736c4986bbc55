// Definitions shared by the generic and the vectorised fused mean-field step kernels.
#pragma once
#include "common.cuh"

namespace d3p {

constexpr int kStepThreads = 256;
constexpr int kStepWarps = kStepThreads / 32;

struct StepArgs {
  const float* params;
  const float* x;
  size_t x_stride;
  const int32_t* y;
  const int32_t* idx;
  const uint8_t* mask;
  const int32_t* num_valid;
  uint32_t B, pos_begin, pos_end;
  uint32_t k0, k1;
  const uint32_t* key_d;      // *_dk entry points: the Threefry key lives in device memory (else nullptr)
  float inv_S, L, C, N;
  float inv_var, log_norm_lik;
  uint32_t d, n_main, half, P, loc_off, rho_off, b_loc_off, b_rho_off;
  int has_b;
  float* px_norms;
  float* px_grads;
  float* px_loss;
  float* partials;
};

template <int LINK>
D3P_D void link_terms(float rho, float inv_S, float& s, float& a, float& bt, float& log_s) {
  if (LINK == D3P_LINK_EXP) {
    s = expf(rho); a = s; bt = inv_S; log_s = rho;
  } else {
    s = softplus_f(rho); a = sigmoid_f(rho); bt = inv_S * a / s; log_s = logf(s);
  }
}

template <int G>
D3P_D unsigned group_mask(int lane) {
  return G == 32 ? 0xffffffffu : (((1u << G) - 1u) << (lane & ~(G - 1)));
}

template <int G>
D3P_D float gsum(float v, unsigned m) {
#pragma unroll
  for (int o = G / 2; o > 0; o >>= 1) v += __shfl_xor_sync(m, v, o);
  return v;
}

struct InterceptGuide { float loc, s, a, bt; };   // the separate intercept site: loc, s, s', (1/S) s'/s (link_terms)

// log p(x_i | theta) of one example.  Bernoulli-logit (numpyro BernoulliLogits.log_prob): r = x . theta of the main
// site, th_b the intercept; Gaussian: r = sum (x - theta)^2 over the n elements of the row.
template <int FAMILY>
D3P_D float row_loglik(float r, float th_b, float y, uint32_t n, float inv_var, float log_norm_lik) {
  if (FAMILY == D3P_FAMILY_LOGREG) {
    const float z = r + th_b;
    return -(fmaxf(z, 0.f) + log1pf(expf(-fabsf(z))) - z * y);
  }
  return -0.5f * r * inv_var - (float)n * log_norm_lik;
}

// Per-example ELBO terms of the step kernels from the group-reduced sums (r as in row_loglik, |theta|^2, |eps|^2
// of the main site over its n elements): the intercept's draw th_b = loc + eb s joins the sums, then
//   S * loss_i = -(log p(theta) - log q(theta)) - N * loglik     (the sqrt(2 pi) terms cancel; returned)
//   Lr = L (sigmoid(z) - y)                                       (logreg; 0 for the Gaussian family)
template <int FAMILY>
D3P_D float example_loss(const StepArgs& a, const InterceptGuide& b, float eb, float y, float r, float s_th2,
                         float s_e2, float sum_log_s, uint32_t n, float& th_b, float& Lr) {
  th_b = 0.f; Lr = 0.f;
  if (a.has_b) { th_b = fmaf(eb, b.s, b.loc); s_th2 = fmaf(th_b, th_b, s_th2); s_e2 = fmaf(eb, eb, s_e2); }
  const float loglik = row_loglik<FAMILY>(r, th_b, y, n, a.inv_var, a.log_norm_lik);
  if (FAMILY == D3P_FAMILY_LOGREG) Lr = a.L * (sigmoid_f(r + th_b) - y);
  return 0.5f * s_th2 - 0.5f * s_e2 - sum_log_s - a.N * loglik;
}

// The intercept's gradient (glb wrt its loc, gsb wrt its rho; 0 without one); returns nrm plus their squares.
D3P_D float intercept_grad(const StepArgs& a, const InterceptGuide& b, float th_b, float eb, float Lr, float nrm,
                           float& glb, float& gsb) {
  glb = 0.f; gsb = 0.f;
  if (a.has_b) {
    glb = fmaf(th_b, a.inv_S, Lr);
    gsb = fmaf(glb, eb * b.a, -b.bt);
    nrm = fmaf(glb, glb, fmaf(gsb, gsb, nrm));
  }
  return nrm;
}

}  // namespace d3p
