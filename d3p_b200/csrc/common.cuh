// Shared device/host helpers for the d3p_b200 hot path (sm_100a).
// ChaCha20 (RFC 8439) block function, Threefry-2x32-20, the jax.random bits->float->normal
// transform (d3p/random/__init__.py:76-81) and small warp utilities.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/d3p_b200.h"

#define D3P_HD __host__ __device__ __forceinline__
#define D3P_D __device__ __forceinline__

namespace d3p {

struct ChaChaState { uint32_t w[16]; };

D3P_HD uint32_t rotl32(uint32_t x, int n) {
#ifdef __CUDA_ARCH__
  return __funnelshift_l(x, x, n);
#else
  return (x << n) | (x >> (32 - n));
#endif
}

#define D3P_QR(a, b, c, d)            \
  a += b; d ^= a; d = rotl32(d, 16);  \
  c += d; b ^= c; b = rotl32(b, 12);  \
  a += b; d ^= a; d = rotl32(d, 8);   \
  c += d; b ^= c; b = rotl32(b, 7);

// RFC 8439 section 2.3: 10 double rounds + feed-forward. `counter` replaces word 12.
D3P_HD void chacha20_block(const uint32_t (&in)[16], uint32_t counter, uint32_t (&out)[16]) {
  uint32_t x0 = in[0], x1 = in[1], x2 = in[2], x3 = in[3], x4 = in[4], x5 = in[5], x6 = in[6],
           x7 = in[7], x8 = in[8], x9 = in[9], x10 = in[10], x11 = in[11], x12 = counter,
           x13 = in[13], x14 = in[14], x15 = in[15];
#pragma unroll
  for (int i = 0; i < 10; ++i) {
    D3P_QR(x0, x4, x8, x12) D3P_QR(x1, x5, x9, x13) D3P_QR(x2, x6, x10, x14) D3P_QR(x3, x7, x11, x15)
    D3P_QR(x0, x5, x10, x15) D3P_QR(x1, x6, x11, x12) D3P_QR(x2, x7, x8, x13) D3P_QR(x3, x4, x9, x14)
  }
  out[0] = x0 + in[0]; out[1] = x1 + in[1]; out[2] = x2 + in[2]; out[3] = x3 + in[3];
  out[4] = x4 + in[4]; out[5] = x5 + in[5]; out[6] = x6 + in[6]; out[7] = x7 + in[7];
  out[8] = x8 + in[8]; out[9] = x9 + in[9]; out[10] = x10 + in[10]; out[11] = x11 + in[11];
  out[12] = x12 + counter; out[13] = x13 + in[13]; out[14] = x14 + in[14]; out[15] = x15 + in[15];
}

// ---- ChaCha key derivation: the ONE swappable rule behind rng_suite.split / fold_in ---------------------------
// (d3p/random/__init__.py:28-30 -> jax-chacha-prng >= 1, < 2, which is not in the reference tree: PARITY UNPINNED.
// tests/golden/make_reference_golden.py dumps the real package's outputs where it is installed and
// tests/test_reference_golden.py then holds this rule — and oracle/chacha.py:derive_key, its mirror — to them.)
//   child key  = words 0..7 of the ChaCha20 block of the parent state with counter := data and nonce word 2 ^= tag
//   child      = {constants, child key, counter 0, nonce of the parent}
// split(S, n)[i] = derive(S, i, SPLIT) and fold_in(S, d) = derive(S, d, FOLD_IN) use DIFFERENT tags, so a key that is
// both split and folded (DPSVI splits its state key 3 ways, the batchifiers fold the step index into theirs) never
// reuses a stream; neither tag can collide with a keystream block of S itself (those have nonce word 2 unchanged).
enum : uint32_t { D3P_DERIVE_SPLIT = 0x80000000u, D3P_DERIVE_FOLD_IN = 0x40000000u };

D3P_HD void chacha_derive_key(const uint32_t (&in)[16], uint32_t data, uint32_t domain_tag, uint32_t (&out)[16]) {
  uint32_t tmp[16], blk[16];
#pragma unroll
  for (int i = 0; i < 16; ++i) tmp[i] = in[i];
  tmp[15] ^= domain_tag;
  chacha20_block(tmp, data, blk);
  out[0] = 0x61707865u; out[1] = 0x3320646Eu; out[2] = 0x79622D32u; out[3] = 0x6B206574u;
#pragma unroll
  for (int i = 0; i < 8; ++i) out[4 + i] = blk[i];
  out[12] = 0;
  out[13] = in[13]; out[14] = in[14]; out[15] = in[15];
}

// A ChaCha state handed to a kernel either BY VALUE (the host-key entry points: the 16 words travel in the kernel
// parameters) or BY DEVICE POINTER (the *_dk entry points: the key was produced on the device, e.g. by a split /
// fold_in inside a jitted loop body, and no host ever sees it).  d == nullptr selects the by-value words.
struct ChaChaArg {
  ChaChaState v;
  const uint32_t* d;
};
__device__ __forceinline__ void load_chacha(const ChaChaArg& a, ChaChaState& st) {
  if (a.d) {
#pragma unroll
    for (int i = 0; i < 16; ++i) st.w[i] = __ldg(a.d + i);
  } else {
    st = a.v;
  }
}
inline ChaChaArg chacha_arg(const uint32_t* host_words, const uint32_t* dev_words) {
  ChaChaArg a;
  for (int i = 0; i < 16; ++i) a.v.w[i] = host_words ? host_words[i] : 0u;
  a.d = dev_words;
  return a;
}

// Threefry-2x32, 20 rounds (Random123), as used by jax.random (d3p/svi.py:290).
struct TfKey {
  uint32_t k0, k1, k2;
  D3P_HD TfKey() : k0(0), k1(0), k2(0) {}
  D3P_HD TfKey(uint32_t a, uint32_t b) : k0(a), k1(b), k2(a ^ b ^ 0x1BD11BDAu) {}
};

#define D3P_TF_ROUND(r) x0 += x1; x1 = rotl32(x1, r); x1 ^= x0;

D3P_HD void threefry2x32(const TfKey& k, uint32_t c0, uint32_t c1, uint32_t& y0, uint32_t& y1) {
  uint32_t x0 = c0 + k.k0, x1 = c1 + k.k1;
  D3P_TF_ROUND(13) D3P_TF_ROUND(15) D3P_TF_ROUND(26) D3P_TF_ROUND(6)
  x0 += k.k1; x1 += k.k2 + 1u;
  D3P_TF_ROUND(17) D3P_TF_ROUND(29) D3P_TF_ROUND(16) D3P_TF_ROUND(24)
  x0 += k.k2; x1 += k.k0 + 2u;
  D3P_TF_ROUND(13) D3P_TF_ROUND(15) D3P_TF_ROUND(26) D3P_TF_ROUND(6)
  x0 += k.k0; x1 += k.k1 + 3u;
  D3P_TF_ROUND(17) D3P_TF_ROUND(29) D3P_TF_ROUND(16) D3P_TF_ROUND(24)
  x0 += k.k1; x1 += k.k2 + 4u;
  D3P_TF_ROUND(13) D3P_TF_ROUND(15) D3P_TF_ROUND(26) D3P_TF_ROUND(6)
  x0 += k.k2; x1 += k.k0 + 5u;
  y0 = x0; y1 = x1;
}

// The step kernels take the Threefry key as two words by value, or - the *_dk entry points - from device memory.
__device__ __forceinline__ TfKey tf_key_arg(uint32_t k0, uint32_t k1, const uint32_t* dev) {
  return dev ? TfKey(__ldg(dev), __ldg(dev + 1)) : TfKey(k0, k1);
}

// jax.random.split(key, 2): counts iota(4) -> calls (0,2),(1,3); child0=(a.y0,b.y0), child1=(a.y1,b.y1)
D3P_HD void tf_split2(const TfKey& k, TfKey& child0, TfKey& child1) {
  uint32_t a0, a1, b0, b1;
  threefry2x32(k, 0u, 2u, a0, a1);
  threefry2x32(k, 1u, 3u, b0, b1);
  child0 = TfKey(a0, b0);
  child1 = TfKey(a1, b1);
}

// word m of jax.random.split(K, B) flattened ([B,2] row-major): counts iota(2B) halves.
D3P_HD uint32_t tf_split_word(const TfKey& K, uint32_t B, uint32_t m) {
  uint32_t y0, y1;
  const bool first = m < B;                  // one call either way: counts (j, j + B), j = m mod B
  const uint32_t j = first ? m : m - B;
  threefry2x32(K, j, j + B, y0, y1);
  return first ? y0 : y1;
}

D3P_HD TfKey tf_example_key(const TfKey& K, uint32_t B, uint32_t p) {
  return TfKey(tf_split_word(K, B, 2u * p), tf_split_word(K, B, 2u * p + 1u));
}

// numpyro's seed-handler plumbing under Trace_ELBO: (model_seed, guide_seed) = split(kp); the guide's handler then
// takes one split per latent site, in the order the guide samples them:
//   rng = guide_rng(kp); k_site0 = next_site(rng); k_site1 = next_site(rng); ...
D3P_HD TfKey guide_rng(const TfKey& kp) {
  TfKey model_seed, guide_seed;
  tf_split2(kp, model_seed, guide_seed);
  return guide_seed;
}

// (rng, site) = split(rng); returns site
D3P_HD TfKey next_site(TfKey& rng) {
  TfKey next, site;
  tf_split2(rng, next, site);
  rng = next;
  return site;
}

// ---- bits -> uniform -> normal (jax.random._uniform / _normal_real) -------------------------
D3P_HD float bits_to_unit_float(uint32_t bits) {
#ifdef __CUDA_ARCH__
  return __uint_as_float((bits >> 9) | 0x3F800000u) - 1.0f;
#else
  union { uint32_t u; float f; } v; v.u = (bits >> 9) | 0x3F800000u; return v.f - 1.0f;
#endif
}

// Giles' single-precision erfinv polynomial as lowered by XLA for f32 (lax.erf_inv).
// kFast: w = -log(1 - x*x) through MUFU.LG2 (abs error ~4e-7 in w, <2e-7 relative in the
// result, see DESIGN.md); otherwise log1pf as XLA does.
template <bool kFast>
D3P_D float erfinv_f32(float x) {
  float w;
  // XLA lowers erf_inv's w = -log1p(x * -x) with the PRODUCT ROUNDED to float32 first: in the tails (|x| -> 1) that
  // rounding moves w by up to 2e-4 and the result by ~1e-5 relative, so it is part of the reference's arithmetic
  // and is kept (a fused 1 - x*x is more accurate and therefore different)
  if (kFast) w = -__logf(__fadd_rn(1.0f, __fmul_rn(-x, x)));
  else w = -log1pf(__fmul_rn(-x, x));
  float p;
  if (w < 5.0f) {
    w = w - 2.5f;
    p = 2.81022636e-08f;
    p = fmaf(p, w, 3.43273939e-07f);
    p = fmaf(p, w, -3.5233877e-06f);
    p = fmaf(p, w, -4.39150654e-06f);
    p = fmaf(p, w, 0.00021858087f);
    p = fmaf(p, w, -0.00125372503f);
    p = fmaf(p, w, -0.00417768164f);
    p = fmaf(p, w, 0.246640727f);
    p = fmaf(p, w, 1.50140941f);
  } else {
    w = (kFast ? __fsqrt_rn(w) : sqrtf(w)) - 3.0f;
    p = -0.000200214257f;
    p = fmaf(p, w, 0.000100950558f);
    p = fmaf(p, w, 0.00134934322f);
    p = fmaf(p, w, -0.00367342844f);
    p = fmaf(p, w, 0.00573950773f);
    p = fmaf(p, w, -0.0076224613f);
    p = fmaf(p, w, 0.00943887047f);
    p = fmaf(p, w, 1.00167406f);
    p = fmaf(p, w, 2.83297682f);
  }
  return (fabsf(x) == 1.0f) ? x * __int_as_float(0x7F800000) : p * x;
}

#define D3P_NORMAL_LO (-0.99999994f)   // nextafter(-1, 0) in float32
#define D3P_SQRT2 1.41421354f          // float32(sqrt(2))

template <bool kFast>
D3P_D float bits_to_normal(uint32_t bits) {
  float f = bits_to_unit_float(bits);
  // (hi - lo) rounds to exactly 2.0f in float32, so f*(hi-lo)+lo == fma(f, 2, lo) exactly
  float u = fmaxf(D3P_NORMAL_LO, fmaf(f, 2.0f, D3P_NORMAL_LO));
  return D3P_SQRT2 * erfinv_f32<kFast>(u);
}

// ---- fast path for the in-kernel guide noise (Threefry normals) --------------------------------
// Same function as bits_to_normal, restructured for throughput:
//   * u = fma(f, 2, lo) already satisfies u >= lo and |u| < 1, so the max() and the |x| == 1 test
//     of the reference transform are no-ops and are dropped (bit-identical);
//   * w - 2.5 = fma(lg2(1 - rn(u*u)), -ln2, -2.5) through MUFU.LG2 (absolute error ~4e-7 in w); u*u is rounded to
//     float32 before the subtraction like XLA's log1p(x * -x) (see erfinv_f32);
//   * sqrt(2) is folded into the polynomial coefficients (<= 1 ulp difference);
//   * the |u| > 0.9966 tail (0.34 % of the variates) is not evaluated here: the caller checks
//     `needs_tail` for a whole group of variates with one warp-uniform branch and patches them
//     with normal_tail(), which keeps the common path branch-free (ILP across variates).
struct FastNormal { float value; float w; };

D3P_D float unit_to_u(uint32_t bits) {
  return fmaf(bits_to_unit_float(bits), 2.0f, D3P_NORMAL_LO);
}

// 1 - u*u lies in [2^-23, 1]: never denormal, so the .ftz forms are bit-identical to the plain ones
// and compile to a single MUFU (the non-ftz __log2f adds a denormal guard: FSETP + 2 predicated ops).
D3P_D float lg2_ftz(float x) { float r; asm("lg2.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x)); return r; }
D3P_D float sqrt_ftz(float x) { float r; asm("sqrt.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x)); return r; }

D3P_D float normal_central(float u, float& w_out) {
  const float l2 = lg2_ftz(__fadd_rn(1.0f, __fmul_rn(-u, u)));   // product rounded first, as XLA's log1p(x * -x)
  w_out = l2;                                            // w = -ln2 * l2 ; tail iff w >= 5
  const float w = fmaf(l2, -0.693147182f, -2.5f);
  float p = 2.81022636e-08f * D3P_SQRT2;
  p = fmaf(p, w, 3.43273939e-07f * D3P_SQRT2);
  p = fmaf(p, w, -3.5233877e-06f * D3P_SQRT2);
  p = fmaf(p, w, -4.39150654e-06f * D3P_SQRT2);
  p = fmaf(p, w, 0.00021858087f * D3P_SQRT2);
  p = fmaf(p, w, -0.00125372503f * D3P_SQRT2);
  p = fmaf(p, w, -0.00417768164f * D3P_SQRT2);
  p = fmaf(p, w, 0.246640727f * D3P_SQRT2);
  p = fmaf(p, w, 1.50140941f * D3P_SQRT2);
  return p * u;
}

// lg2(1 - u^2) <= -5 / ln2  <=>  w >= 5
#define D3P_TAIL_L2 (-7.21347523f)

D3P_D float normal_tail(float u, float l2) {
  const float w = sqrt_ftz(l2 * -0.693147182f) - 3.0f;   // MUFU.SQRT: <= 2 ulp in w, tail variates only
  float p = -0.000200214257f * D3P_SQRT2;
  p = fmaf(p, w, 0.000100950558f * D3P_SQRT2);
  p = fmaf(p, w, 0.00134934322f * D3P_SQRT2);
  p = fmaf(p, w, -0.00367342844f * D3P_SQRT2);
  p = fmaf(p, w, 0.00573950773f * D3P_SQRT2);
  p = fmaf(p, w, -0.0076224613f * D3P_SQRT2);
  p = fmaf(p, w, 0.00943887047f * D3P_SQRT2);
  p = fmaf(p, w, 1.00167406f * D3P_SQRT2);
  p = fmaf(p, w, 2.83297682f * D3P_SQRT2);
  return p * u;
}

// scalar convenience form (per-variate branch): used by the generic kernel
D3P_D float bits_to_normal_fast(uint32_t bits) {
  const float u = unit_to_u(bits);
  float l2;
  float r = normal_central(u, l2);
  if (l2 <= D3P_TAIL_L2) r = normal_tail(u, l2);
  return r;
}

D3P_D float bits_to_uniform(uint32_t bits, float lo, float hi) {
  float f = bits_to_unit_float(bits);
  return fmaxf(lo, __fadd_rn(__fmul_rn(f, hi - lo), lo));
}

// ---- warp helpers ---------------------------------------------------------------------------
template <int W>
D3P_D float group_sum(float v) {
#pragma unroll
  for (int o = W / 2; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

D3P_D float softplus_f(float x) { return fmaxf(x, 0.f) + log1pf(expf(-fabsf(x))); }
D3P_D float sigmoid_f(float x) { return 1.0f / (1.0f + expf(-x)); }

}  // namespace d3p
