// K7: fused DP-SVI step for the VAE of examples/vae.py:65-153 — per-example gradient, ghost norm,
// clip and clipped sum (d3p/svi.py:238-348) without ever materialising the [B, P] per-example
// gradients (10.7 GB at B = 4096, P = 652 824).
//
// A dense layer's per-example gradient is the outer product a_i (x) delta_i (+ delta_i for the bias):
//     ||g_i||^2 = sum_layers (||a_i||^2 + 1) ||delta_i||^2          (ghost norm)
//     sum_i c_i g_i = A^T diag(c) Delta                               (clipped sum)
// Pipeline (one stream, no host sync; GEMMs = 3xTF32 tcgen05 kernels of tc_gemm_kernel.cuh):
//   split W1, W5 -> hi/lo | prep X (gather, hi/lo, ||x||^2, ones column)
//   G1  pre1 = X W1          epilogue: + b1, softplus -> H1 hi/lo, ||h1||^2
//   S1  heads z_loc, log z_std (K = H, N = 2Z), eps (Threefry), z, KL part, pre4 = z W4, H2 hi/lo
//   G5  logits = H2 W5       epilogue: + b5, sigmoid, Bernoulli loss, delta5 hi/lo, ||delta5||^2
//   G5b dh2 = delta5 W5^T    epilogue: * softplus'(pre4) -> delta4, ||delta4||^2
//   S2  delta_z, delta2/3, delta1, ghost norm, c_i; writes c*delta1 hi/lo, c*delta4, c*[delta2|delta3],
//       [c*h2 | c] hi/lo
//   GW1 [X | 1]^T (c delta1)        -> dW1, db1  (split over the batch, partial rows)
//   GW5 delta5^T [c h2 | c]         -> dW5^T, db5
//   GW23 [H1 | 1]^T (c [delta2|delta3]) -> dW2, dW3, db2, db3;  GW4 (c delta4)^T [z | 1] -> dW4^T, db4
//   loss / count columns of the partial rows
// The partial rows [S, P + 2] are reduced in a fixed order by d3p_perturb_finalize_f32.
#include <cstdlib>
#include <mutex>

#include "common.cuh"
#include "launch.cuh"
#include "tc_gemm_kernel.cuh"

namespace d3p {

constexpr int kVaeBN = 224;            // N tile of the GEMMs with N = D (784 -> 4 tiles x 32 M tiles = 128 CTAs)
constexpr int kVaeBNH = 128;           // N tile of the forward/backward GEMMs with N = H: 400 -> 4 tiles = 128 CTAs
                                       // (224 gave 2 tiles = 64 CTAs on 148 SMs: measured 36 / 58 us for G1 / G5b)
constexpr int kMidWarps = 16;
constexpr int kMidE = 2;               // examples per warp iteration in the SIMT "middle" kernels (the kernels are
                                       // latency-bound: 16 warps x 2 examples hide more than 8 x 4 did)
constexpr float kF32Tiny = 1.17549435e-38f;
constexpr float kF32OneMinusEps = 0.99999988079071044921875f;   // 1 - 2^-23

// ---- epilogues ---------------------------------------------------------------------------------------
struct EpiFwd1 {   // H1 = softplus(acc + b1)
  struct Args { const float* bias; float* h_hi; float* h_lo; size_t ld; float* rowsq; uint32_t rows_ld; };
  struct RowState { float sq; };
  __device__ static void begin(const Args&, const tc::GemmShape&, uint32_t, uint32_t, uint32_t, RowState& rs) { rs.sq = 0.f; }
  __device__ static void tile(const Args& a, const tc::GemmShape& g, uint32_t row, uint32_t col0, uint32_t,
                              const uint32_t (&v)[32], RowState& rs, float*) {
    // direct 16-byte stores (one row per lane): this epilogue is bound by the softplus arithmetic, not by its stores —
    // the transposed, fully coalesced form of EpiFwd5 / EpiBwd5 measured slower here (8.5 vs 6.9 us)
    if (row >= g.M) return;
#pragma unroll
    for (int j = 0; j < 32; j += 4) {
      if (col0 + j < g.N) {                       // N is a multiple of 4; a guard, not a break: the loop must unroll
        float h[4], hi[4], lo[4];
#pragma unroll
        for (int t = 0; t < 4; ++t) {
          h[t] = softplus_f(__uint_as_float(v[j + t]) + __ldg(a.bias + col0 + j + t));
          hi[t] = tc::tf32_hi(h[t]);
          lo[t] = h[t] - hi[t];
          rs.sq = fmaf(h[t], h[t], rs.sq);
        }
        *reinterpret_cast<float4*>(a.h_hi + (size_t)row * a.ld + col0 + j) = make_float4(hi[0], hi[1], hi[2], hi[3]);
        *reinterpret_cast<float4*>(a.h_lo + (size_t)row * a.ld + col0 + j) = make_float4(lo[0], lo[1], lo[2], lo[3]);
      }
    }
  }
  __device__ static void end(const Args& a, const tc::GemmShape& g, uint32_t row, uint32_t n_tile, uint32_t, RowState& rs) {
    if (row < g.M) a.rowsq[(size_t)n_tile * a.rows_ld + row] = rs.sq;
  }
};

struct EpiFwd5 {   // p = sigmoid(acc + b5); Bernoulli(probs) log-lik (numpyro clamp_probs); delta5 = p - x
  struct Args {
    const float* bias; const float* x_hi; size_t ldx;          // x_hi holds x unmasked
    float* d_hi; float* d_lo; size_t ld; float* rowsq; float* rowloss; uint32_t rows_ld;
  };
  struct RowState { float sq, loss; };
  __device__ static void begin(const Args&, const tc::GemmShape&, uint32_t, uint32_t, uint32_t, RowState& rs) {
    rs.sq = 0.f; rs.loss = 0.f;
  }
  __device__ static void tile(const Args& a, const tc::GemmShape& g, uint32_t row, uint32_t col0, uint32_t,
                              const uint32_t (&v)[32], RowState& rs, float* scratch) {
    const uint32_t row0 = row - (threadIdx.x & 31);
    const uint32_t nr = g.M > row0 ? g.M - row0 : 0, nc = g.N > col0 ? g.N - col0 : 0;
    // x (held unmasked in x_hi) and delta5 move as full 128-byte row segments through the warp's scratch
    float xs[32], d[32];
    tc::warp_load_rows(scratch, a.x_hi + (size_t)row0 * a.ldx + col0, a.ldx, nr, nc, xs);
#pragma unroll
    for (int j = 0; j < 32; ++j) {
      const bool ok = row < g.M && col0 + j < g.N;
      const float logit = __uint_as_float(v[j]) + __ldg(a.bias + min(col0 + j, g.N - 1));
      const float p = __fdividef(1.0f, 1.0f + __expf(-logit));     // MUFU.EX2 / MUFU.RCP: <= 1e-6 relative
      // numpyro clamps the probabilities (jnp.clip = minimum(maximum(p, tiny), 1 - eps): gradient 1 inside, 1/2 at a
      // bound, 0 outside)
      const float wclip = (p > kF32Tiny ? 1.0f : (p == kF32Tiny ? 0.5f : 0.f)) *
                          (p < kF32OneMinusEps ? 1.0f : (p == kF32OneMinusEps ? 0.5f : 0.f));
      const float pc = fminf(fmaxf(p, kF32Tiny), kF32OneMinusEps);
      // log1p(-pc) = log(1 - pc): 1 - pc is exact for pc >= 1/2 (Sterbenz) and within 6e-8 below; MUFU.LG2 logs
      const float l = xs[j] * __logf(pc) + (1.0f - xs[j]) * __logf(1.0f - pc);
      const float dj = ok ? wclip * (p - xs[j]) : 0.f;
      rs.loss -= ok ? l : 0.f;
      rs.sq = fmaf(dj, dj, rs.sq);
      d[j] = dj;                          // unmasked: kind::tf32 truncates, and dW5's GEMM splits delta5 itself
    }
    tc::warp_store_rows(scratch, a.d_hi + (size_t)row0 * a.ld + col0, a.ld, nr, nc, d);
#pragma unroll
    for (int j = 0; j < 32; ++j) d[j] = d[j] - tc::tf32_hi(d[j]);
    tc::warp_store_rows(scratch, a.d_lo + (size_t)row0 * a.ld + col0, a.ld, nr, nc, d);
  }
  __device__ static void end(const Args& a, const tc::GemmShape& g, uint32_t row, uint32_t n_tile, uint32_t, RowState& rs) {
    if (row < g.M) {
      a.rowsq[(size_t)n_tile * a.rows_ld + row] = rs.sq;
      a.rowloss[(size_t)n_tile * a.rows_ld + row] = rs.loss;
    }
  }
};

struct EpiBwd5 {   // delta4 = acc * softplus'(pre4) = acc * (1 - exp(-h2))
  struct Args { const float* h_hi; const float* h_lo; size_t ld; float* d4; float* rowsq; uint32_t rows_ld; };
  struct RowState { float sq; };
  __device__ static void begin(const Args&, const tc::GemmShape&, uint32_t, uint32_t, uint32_t, RowState& rs) { rs.sq = 0.f; }
  __device__ static void tile(const Args& a, const tc::GemmShape& g, uint32_t row, uint32_t col0, uint32_t,
                              const uint32_t (&v)[32], RowState& rs, float* scratch) {
    const uint32_t row0 = row - (threadIdx.x & 31);
    const uint32_t nr = g.M > row0 ? g.M - row0 : 0, nc = g.N > col0 ? g.N - col0 : 0;
    float hs[32], d[32];                                  // h2 (unmasked) in, delta4 out: coalesced through the scratch
    tc::warp_load_rows(scratch, a.h_hi + (size_t)row0 * a.ld + col0, a.ld, nr, nc, hs);
#pragma unroll
    for (int j = 0; j < 32; ++j) {
      const bool ok = row < g.M && col0 + j < g.N;
      d[j] = ok ? __uint_as_float(v[j]) * (-expm1f(-hs[j])) : 0.f;
      rs.sq = fmaf(d[j], d[j], rs.sq);
    }
    tc::warp_store_rows(scratch, a.d4 + (size_t)row0 * a.ld + col0, a.ld, nr, nc, d);
  }
  __device__ static void end(const Args& a, const tc::GemmShape& g, uint32_t row, uint32_t n_tile, uint32_t, RowState& rs) {
    if (row < g.M) a.rowsq[(size_t)n_tile * a.rows_ld + row] = rs.sq;
  }
};

struct EpiGrad {   // clipped-sum tile -> partial row `split`: weight block(s) + the bias row / column
  struct Args {
    float* partials; size_t row_stride;   // P + 2
    uint32_t w_off, b_off;                // offsets of the weight matrix and of the bias in the flat vector
    uint32_t w_ld;                        // row stride of the weight matrix
    uint32_t main;                        // !transpose: rows < main are weights, row == main is the bias
    int transpose;                        //  transpose: cols < main are weights (stored [col, row]), col == main the bias
    uint32_t split_col;                   // !transpose only: cols >= split_col belong to a second matrix / bias
    uint32_t w_off2, b_off2;              //   (both matrices have w_ld columns)
  };
  struct RowState {};
  __device__ static void begin(const Args&, const tc::GemmShape&, uint32_t, uint32_t, uint32_t, RowState&) {}
  __device__ static void end(const Args&, const tc::GemmShape&, uint32_t, uint32_t, uint32_t, RowState&) {}
  __device__ static void tile(const Args& a, const tc::GemmShape& g, uint32_t row, uint32_t col0, uint32_t split,
                              const uint32_t (&v)[32], RowState&, float* scratch) {
    float* out = a.partials + (size_t)split * a.row_stride;
    if (!a.transpose) {
      const uint32_t sc = a.split_col ? a.split_col : 0xffffffffu;
      // weight rows of a full chunk (the common case): the warp's 32 rows are w_ld floats apart in the flat vector, so
      // the chunk goes out as 128-byte row segments through the scratch (16-byte pieces, or 8-byte ones when this
      // split's partial row sits 8 bytes off); warp-uniform conditions only
      const uint32_t row0 = row - (threadIdx.x & 31);
      if (col0 + 32 <= g.N && col0 + 32 <= sc && row0 + 32 <= a.main && row0 + 32 <= g.M && (a.w_ld & 1) == 0) {
        float* base = out + a.w_off + (size_t)row0 * a.w_ld + col0;
        const uintptr_t mis = reinterpret_cast<uintptr_t>(base) & 15;
        float f[32];
#pragma unroll
        for (int j = 0; j < 32; ++j) f[j] = __uint_as_float(v[j]);
        if (mis == 0 && (a.w_ld & 3) == 0) { tc::warp_store_rows(scratch, base, a.w_ld, 32, 32, f); return; }
        if ((mis & 7) == 0) { tc::warp_store_rows8(scratch, base, a.w_ld, 32, 32, f); return; }
      }
      if (row >= g.M) return;
      float* p1 = row < a.main ? out + a.w_off + (size_t)row * a.w_ld : out + a.b_off;
      float* p2 = row < a.main ? out + a.w_off2 + (size_t)row * a.w_ld : out + a.b_off2;
#pragma unroll
      for (int j = 0; j < 32; ++j) {
        const uint32_t col = col0 + j;
        if (col < g.N) {
          if (col < sc) p1[col] = __uint_as_float(v[j]);
          else p2[col - sc] = __uint_as_float(v[j]);
        }
      }
    } else {
      if (row >= g.M) return;
#pragma unroll
      for (int j = 0; j < 32; ++j) {
        const uint32_t col = col0 + j;
        if (col < a.main) out[a.w_off + (size_t)col * a.w_ld + row] = __uint_as_float(v[j]);
        else if (col == a.main) out[a.b_off + row] = __uint_as_float(v[j]);
      }
    }
  }
};

// ---- SIMT kernels ------------------------------------------------------------------------------------
struct VaeArgs {
  uint32_t D, H, Z, B, Bl, pos_begin;
  size_t ldx, ldh, ldz, ld23;         // D + 4, H + 4, roundup(Z + 1, 4), roundup(2 Z, 4)
  const float* params;
  uint32_t off_w4, off_b4, off_w5, off_b5, off_w1, off_b1, off_w2, off_b2, off_w3, off_b3, P;
  const float* x; size_t x_stride; const int32_t* idx; const uint8_t* mask; const int32_t* num_valid;
  uint32_t k0, k1;
  const uint32_t* key_d;              // *_dk entry point: Threefry key in device memory (else nullptr)
  int eval_mode;                      // DPSVI.evaluate: the key is numpyro's rng_key_eval, z [B, Z] is ONE draw (see vae_eval_eps)
  float site_scale, inv_S, C;
  uint32_t ns_h, ns_d;                // row-reduction slots over H and over D (N tiles x epilogue parts)
  uint32_t S;                         // partial rows
  // workspace
  float *x_hi, *x_lo; int* x_lo_flag;
  float *h1_hi, *h1_lo, *h2_hi, *h2_lo, *ch2_hi, *ch2_lo, *d5_hi, *d5_lo, *d4, *cd4_hi, *cd4_lo, *cd1_hi, *cd1_lo;
  float *z_hi, *z_lo, *u, *cd23_hi, *cd23_lo;
  float *sq_x, *sq_h1, *sq_h2, *sq_z, *sq_d5, *loss_rec, *sq_d4, *loss_kl, *lossv, *cnt;
  float* partials;
  float* px_norms; float* px_loss;
  // fragment-ordered hi/lo copies of the thin weight matrices (vae_prep_mid_kernel) for the warp-MMA mid kernels
  float4 *wf23, *wf4, *wf4t, *wf23t;
};

// X rows -> [X | 1 | 0 0 0] hi / lo (row stride D + 4), ||x||^2, "some lo != 0" flag.  One warp per row, 16-byte
// accesses when the rows are 16-byte aligned (kVec), several independent loads in flight per lane.
template <bool kVec>
__global__ void vae_prep_x_kernel(VaeArgs a) {
  const int lane = threadIdx.x & 31;
  const uint32_t warps = (blockDim.x >> 5) * gridDim.x;
  bool any_lo = false;
  for (uint32_t r = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5); r < a.Bl; r += warps) {
    const uint32_t p = a.pos_begin + r;
    // masked-out positions are never dereferenced (the sharded Poisson sampler leaves their index slots unwritten):
    // they become all-zero rows, which the clip factor 0 removes from every sum anyway
    const bool valid = (!a.num_valid || p < (uint32_t)max(*a.num_valid, 0)) && (!a.mask || a.mask[p]);
    const size_t src = valid ? (size_t)(a.idx ? (uint32_t)a.idx[p] : p) * a.x_stride : 0;
    float sq = 0.f;
    if (kVec) {
      const float4* __restrict__ xs = reinterpret_cast<const float4*>(a.x + src);
      float4* __restrict__ oh = reinterpret_cast<float4*>(a.x_hi + (size_t)r * a.ldx);
      float4* __restrict__ ol = reinterpret_cast<float4*>(a.x_lo + (size_t)r * a.ldx);
      const uint32_t n4 = a.D / 4;
#pragma unroll 4
      for (uint32_t j = lane; j <= n4; j += 32) {
        const float4 v = j < n4 ? (valid ? __ldg(xs + j) : make_float4(0.f, 0.f, 0.f, 0.f)) : make_float4(1.0f, 0.f, 0.f, 0.f);
        const float4 hi = make_float4(tc::tf32_hi(v.x), tc::tf32_hi(v.y), tc::tf32_hi(v.z), tc::tf32_hi(v.w));
        const float4 lo = make_float4(v.x - hi.x, v.y - hi.y, v.z - hi.z, v.w - hi.w);
        oh[j] = v;               // unmasked: kind::tf32 truncates the operand itself, and EpiFwd5 reads x from here
        ol[j] = lo;
        if (j < n4) sq = fmaf(v.x, v.x, fmaf(v.y, v.y, fmaf(v.z, v.z, fmaf(v.w, v.w, sq))));
        any_lo |= (lo.x != 0.f) | (lo.y != 0.f) | (lo.z != 0.f) | (lo.w != 0.f);
      }
    } else {
      for (uint32_t j = lane; j < a.D + 4; j += 32) {
        float v = j < a.D ? (valid ? a.x[src + j] : 0.f) : (j == a.D ? 1.0f : 0.0f);
        const float hi = tc::tf32_hi(v), lo = v - hi;
        a.x_hi[(size_t)r * a.ldx + j] = v;       // unmasked, see the vector path
        a.x_lo[(size_t)r * a.ldx + j] = lo;
        if (j < a.D) sq = fmaf(v, v, sq);
        any_lo |= (lo != 0.f);
      }
    }
    sq = group_sum<32>(sq);
    if (lane == 0) a.sq_x[r] = sq;
  }
  if (__any_sync(0xffffffffu, any_lo) && lane == 0) atomicOr(a.x_lo_flag, 1);
}

// DPSVI.evaluate (d3p/svi.py:436-449 -> numpyro SVI.evaluate -> Trace_ELBO.loss on the whole batch): one guide trace,
// so z ~ Normal(z_loc, z_std).to_event(1) of shape [B, Z] is drawn with ONE key: rng_key_eval -> (_, guide_seed) ->
// (rng, k_plate) -> (_, k_z); eps = jax.random.normal(k_z, (B, Z)), i.e. element e = p Z + j of B Z variates in the
// legacy Threefry layout (call c yields elements c and c + half).
D3P_D float vae_eval_eps(const TfKey& K_eval, uint32_t B, uint32_t Z, uint32_t p, uint32_t j) {
  TfKey model_seed, guide_seed, rng, k_plate, rng2, k_z;
  tf_split2(K_eval, model_seed, guide_seed);
  tf_split2(guide_seed, rng, k_plate);
  tf_split2(rng, rng2, k_z);
  const uint32_t n = B * Z, half = (n + 1) / 2, e = p * Z + j;
  uint32_t y0, y1;
  if (e < half) {
    threefry2x32(k_z, e, e + half < n ? e + half : 0u, y0, y1);
    return bits_to_normal<false>(y0);
  }
  threefry2x32(k_z, e - half, e, y0, y1);
  return bits_to_normal<false>(y1);
}

// S1: encoder heads, guide sample, KL part of the loss, decoder hidden layer.  The three thin weight
// matrices are staged in shared memory once per CTA; each warp walks groups of kMidE examples.
__global__ void __launch_bounds__(kMidWarps * 32) vae_mid_fwd_kernel(VaeArgs a) {
  extern __shared__ float smem[];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const uint32_t H = a.H, Z = a.Z, Z2 = 2 * a.Z;
  float* w23s = smem;                                   // [H][2Z]: row k = (W2[k, :], W3[k, :])
  float* w4s = w23s + (size_t)H * Z2;                   // [Z][H]
  float* b23s = w4s + (size_t)Z * H;                    // [2Z]
  float* b4s = b23s + 64;                               // [H]
  float* wsm = b4s + H + (size_t)warp * kMidE * (H + 3 * 64);
  float* h1s = wsm;                                     // [E][H]
  float* zs = h1s + kMidE * H;                          // [E][64]  (z_loc | log z_std)
  float* es = zs + kMidE * 64;                          // [E][64]  eps
  float* zz = es + kMidE * 64;                          // [E][64]  z
  for (uint32_t i0 = threadIdx.x; i0 < H * Z; i0 += 4 * blockDim.x) {     // 12 independent loads in flight
    float v2[4], v3[4], v4[4];
#pragma unroll
    for (int t = 0; t < 4; ++t) {
      const uint32_t i = i0 + t * blockDim.x;
      const bool ok = i < H * Z;
      v2[t] = ok ? __ldg(a.params + a.off_w2 + i) : 0.f;
      v3[t] = ok ? __ldg(a.params + a.off_w3 + i) : 0.f;
      v4[t] = ok ? __ldg(a.params + a.off_w4 + i) : 0.f;
    }
#pragma unroll
    for (int t = 0; t < 4; ++t) {
      const uint32_t i = i0 + t * blockDim.x;
      if (i >= H * Z) break;
      const uint32_t k = i / Z, j = i - k * Z;
      w23s[k * Z2 + j] = v2[t];
      w23s[k * Z2 + Z + j] = v3[t];
      w4s[i] = v4[t];
    }
  }
  for (uint32_t i = threadIdx.x; i < Z; i += blockDim.x) { b23s[i] = a.params[a.off_b2 + i]; b23s[Z + i] = a.params[a.off_b3 + i]; }
  for (uint32_t i = threadIdx.x; i < H; i += blockDim.x) b4s[i] = a.params[a.off_b4 + i];
  __syncthreads();
  const TfKey K = tf_key_arg(a.k0, a.k1, a.key_d);
  const uint32_t half = (Z + 1) / 2;
  const uint32_t groups = (a.Bl + kMidE - 1) / kMidE;
  for (uint32_t gidx = blockIdx.x * kMidWarps + warp; gidx < groups; gidx += gridDim.x * kMidWarps) {
    const uint32_t r0 = gidx * kMidE;
#pragma unroll
    for (int e = 0; e < kMidE; ++e) {
      const uint32_t r = r0 + e;
      {
        const float* __restrict__ ph = a.h1_hi + (size_t)r * a.ldh;
        const float* __restrict__ pl = a.h1_lo + (size_t)r * a.ldh;
        for (uint32_t k0 = 0; k0 < H; k0 += 128) {          // 8 independent loads in flight per lane
          float vh[4], vl[4];
#pragma unroll
          for (int t = 0; t < 4; ++t) {
            const uint32_t k = k0 + 32 * t + lane;
            const bool ok = r < a.Bl && k < H;
            vh[t] = ok ? __ldg(ph + k) : 0.f;
            vl[t] = ok ? __ldg(pl + k) : 0.f;
          }
#pragma unroll
          for (int t = 0; t < 4; ++t) {
            const uint32_t k = k0 + 32 * t + lane;
            if (k < H) h1s[e * H + k] = vh[t] + vl[t];
          }
        }
      }
      // guide noise: key_p -> (_, guide_seed) -> (rng, k_plate) -> (_, k_z); eps = normal(k_z, (Z,))
      if (r < a.Bl && a.eval_mode) {
        for (uint32_t j = lane; j < Z; j += 32) es[e * 64 + j] = vae_eval_eps(K, a.B, Z, a.pos_begin + r, j);
      } else if (r < a.Bl) {
        TfKey kp = tf_example_key(K, a.B, a.pos_begin + r);
        TfKey model_seed, guide_seed, rng, k_plate, rng2, k_z;
        tf_split2(kp, model_seed, guide_seed);
        tf_split2(guide_seed, rng, k_plate);
        tf_split2(rng, rng2, k_z);
        for (uint32_t j = lane; j < half; j += 32) {
          uint32_t y0, y1;
          const uint32_t c1 = (j + half < Z) ? j + half : 0u;
          threefry2x32(k_z, j, c1, y0, y1);
          es[e * 64 + j] = bits_to_normal<false>(y0);
          if (j + half < Z) es[e * 64 + j + half] = bits_to_normal<false>(y1);
        }
      }
      if (r < a.Bl) {
        if (lane < 4) {     // ones column of [H1 | 1] (bias row of the dW2 / dW3 clipped-sum GEMM)
          a.h1_hi[(size_t)r * a.ldh + H + lane] = lane == 0 ? 1.0f : 0.f;
          a.h1_lo[(size_t)r * a.ldh + H + lane] = 0.f;
        }
      }
    }
    __syncwarp();
    // heads: output j < Z is z_loc_j (W2), Z <= j < 2Z is log z_std (W3); lane owns j = lane, lane + 32
    float acc[kMidE][2];
    const uint32_t j0 = lane, j1 = lane + 32;
    const bool v0 = j0 < Z2, v1 = j1 < Z2;
    const uint32_t jj0 = v0 ? j0 : 0, jj1 = v1 ? j1 : 0;
#pragma unroll
    for (int e = 0; e < kMidE; ++e) { acc[e][0] = 0.f; acc[e][1] = 0.f; }
#pragma unroll 4
    for (uint32_t k = 0; k < H; ++k) {
      const float w0 = w23s[k * Z2 + jj0];
      const float w1 = w23s[k * Z2 + jj1];
#pragma unroll
      for (int e = 0; e < kMidE; ++e) {
        const float h = h1s[e * H + k];
        acc[e][0] = fmaf(h, w0, acc[e][0]);
        acc[e][1] = fmaf(h, w1, acc[e][1]);
      }
    }
#pragma unroll
    for (int e = 0; e < kMidE; ++e) {
      if (v0) zs[e * 64 + j0] = acc[e][0] + b23s[j0];
      if (v1) zs[e * 64 + j1] = acc[e][1] + b23s[j1];
    }
    __syncwarp();
#pragma unroll
    for (int e = 0; e < kMidE; ++e) {
      const uint32_t r = r0 + e;
      float kl = 0.f, sqz = 0.f;
      for (uint32_t j = lane; j < Z; j += 32) {
        const float zl = zs[e * 64 + j], sr = zs[e * 64 + Z + j], eps = es[e * 64 + j];
        const float u = expf(sr) * eps;
        const float z = zl + u;
        zz[e * 64 + j] = z;
        if (r < a.Bl) {
          const float hi = tc::tf32_hi(z);
          a.z_hi[(size_t)r * a.ldz + j] = hi;
          a.z_lo[(size_t)r * a.ldz + j] = z - hi;
          a.u[(size_t)r * Z + j] = u;
        }
        kl += 0.5f * z * z - 0.5f * eps * eps - sr;       // -log N(z;0,1) + log N(z; z_loc, z_std), constants cancel
        sqz = fmaf(z, z, sqz);
      }
      if (r < a.Bl)
        for (uint32_t j = Z + lane; j < a.ldz; j += 32) {   // ones column of [z | 1] (db4 of the dW4 GEMM) + padding
          a.z_hi[(size_t)r * a.ldz + j] = j == Z ? 1.0f : 0.f;
          a.z_lo[(size_t)r * a.ldz + j] = 0.f;
        }
      kl = group_sum<32>(kl);
      sqz = group_sum<32>(sqz);
      if (lane == 0 && r < a.Bl) { a.loss_kl[r] = kl; a.sq_z[r] = sqz; }
    }
    __syncwarp();
    // decoder hidden layer: h2 = softplus(z W4 + b4)
    float sq2[kMidE];
#pragma unroll
    for (int e = 0; e < kMidE; ++e) sq2[e] = 0.f;
    for (uint32_t h = lane; h < H; h += 32) {
      float s[kMidE];
      const float b = b4s[h];
#pragma unroll
      for (int e = 0; e < kMidE; ++e) s[e] = b;
#pragma unroll 4
      for (uint32_t j = 0; j < Z; ++j) {
        const float w = w4s[j * H + h];
#pragma unroll
        for (int e = 0; e < kMidE; ++e) s[e] = fmaf(zz[e * 64 + j], w, s[e]);
      }
#pragma unroll
      for (int e = 0; e < kMidE; ++e) {
        const uint32_t r = r0 + e;
        const float h2 = softplus_f(s[e]);
        sq2[e] = fmaf(h2, h2, sq2[e]);
        if (r < a.Bl) {
          const float hi = tc::tf32_hi(h2);
          a.h2_hi[(size_t)r * H + h] = h2;          // unmasked (kind::tf32 truncates; consumers read h2 from here)
          a.h2_lo[(size_t)r * H + h] = h2 - hi;
        }
      }
    }
#pragma unroll
    for (int e = 0; e < kMidE; ++e) {
      const float s = group_sum<32>(sq2[e]);
      if (lane == 0 && r0 + e < a.Bl) a.sq_h2[r0 + e] = s;
    }
    __syncwarp();
  }
}

// S2: back-propagation through the z layer and the encoder heads, ghost norm, clip factor, scaled
// operands of the clipped-sum GEMMs.  W4, W2^T, W3^T staged in shared memory.
__global__ void __launch_bounds__(kMidWarps * 32) vae_mid_bwd_kernel(VaeArgs a) {
  extern __shared__ float smem[];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const uint32_t H = a.H, Z = a.Z;
  float* w4s = smem;                                    // [Z][H]
  float* w2t = w4s + (size_t)Z * H;                     // [Z][H] = W2^T
  float* w3t = w2t + (size_t)Z * H;                     // [Z][H] = W3^T
  float* wsm = w3t + (size_t)Z * H + (size_t)warp * kMidE * (H + 128);
  float* d4s = wsm;                                     // [E][H]
  float* d23 = d4s + kMidE * H;                         // [E][128]: delta2 at [0,64), delta3 at [64,128)
  for (uint32_t i0 = threadIdx.x; i0 < H * Z; i0 += 4 * blockDim.x) {     // 12 independent loads in flight
    float v2[4], v3[4], v4[4];
#pragma unroll
    for (int t = 0; t < 4; ++t) {
      const uint32_t i = i0 + t * blockDim.x;
      const bool ok = i < H * Z;
      v2[t] = ok ? __ldg(a.params + a.off_w2 + i) : 0.f;
      v3[t] = ok ? __ldg(a.params + a.off_w3 + i) : 0.f;
      v4[t] = ok ? __ldg(a.params + a.off_w4 + i) : 0.f;
    }
#pragma unroll
    for (int t = 0; t < 4; ++t) {
      const uint32_t i = i0 + t * blockDim.x;
      if (i >= H * Z) break;
      const uint32_t h = i / Z, j = i - h * Z;
      w4s[i] = v4[t];
      w2t[j * H + h] = v2[t];
      w3t[j * H + h] = v3[t];
    }
  }
  __syncthreads();
  const uint32_t nv = a.num_valid ? (uint32_t)max(*a.num_valid, 0) : 0xffffffffu;
  const float ratio = a.site_scale * a.inv_S;                   // (1 / obs_scale) * site scale
  const uint32_t groups = (a.Bl + kMidE - 1) / kMidE;
  for (uint32_t gidx = blockIdx.x * kMidWarps + warp; gidx < groups; gidx += gridDim.x * kMidWarps) {
    const uint32_t r0 = gidx * kMidE;
#pragma unroll
    for (int e = 0; e < kMidE; ++e) {
      const uint32_t r = r0 + e;
      for (uint32_t h0 = 0; h0 < H; h0 += 128) {
        float v[4];
#pragma unroll
        for (int t = 0; t < 4; ++t) {
          const uint32_t h = h0 + 32 * t + lane;
          v[t] = (r < a.Bl && h < H) ? __ldg(a.d4 + (size_t)r * H + h) : 0.f;
        }
#pragma unroll
        for (int t = 0; t < 4; ++t) {
          const uint32_t h = h0 + 32 * t + lane;
          if (h < H) d4s[e * H + h] = v[t];
        }
      }
    }
    __syncwarp();
    // delta_z_j = z_j + sum_h delta4_h W4[j, h]; lane j keeps z_j and u_j of every example of the group
    float sq23[kMidE], zreg[kMidE], ureg[kMidE];
#pragma unroll
    for (int e = 0; e < kMidE; ++e) {
      const uint32_t r = r0 + e;
      const bool ok = r < a.Bl && (uint32_t)lane < Z;
      sq23[e] = 0.f;
      zreg[e] = ok ? a.z_hi[(size_t)r * a.ldz + lane] + a.z_lo[(size_t)r * a.ldz + lane] : 0.f;
      ureg[e] = ok ? a.u[(size_t)r * Z + lane] : 0.f;
    }
    for (uint32_t j = 0; j < Z; ++j) {
      float part[kMidE];
#pragma unroll
      for (int e = 0; e < kMidE; ++e) part[e] = 0.f;
#pragma unroll 4
      for (uint32_t h = lane; h < H; h += 32) {
        const float w = w4s[j * H + h];
#pragma unroll
        for (int e = 0; e < kMidE; ++e) part[e] = fmaf(d4s[e * H + h], w, part[e]);
      }
#pragma unroll
      for (int e = 0; e < kMidE; ++e) {
        const float s = group_sum<32>(part[e]);
        if ((uint32_t)lane == j) {
          const float dz = s + zreg[e];
          const float d3 = fmaf(dz, ureg[e], -1.0f);
          d23[e * 128 + j] = dz;
          d23[e * 128 + 64 + j] = d3;
          sq23[e] = fmaf(dz, dz, d3 * d3);
        }
      }
    }
    __syncwarp();
    // delta_h1 = delta2 W2^T + delta3 W3^T ; delta1 = delta_h1 * softplus'(pre1); raw delta1 parked in cd1_hi
    float sq1[kMidE];
#pragma unroll
    for (int e = 0; e < kMidE; ++e) sq1[e] = 0.f;
    for (uint32_t h = lane; h < H; h += 32) {
      float s[kMidE];
#pragma unroll
      for (int e = 0; e < kMidE; ++e) s[e] = 0.f;
#pragma unroll 4
      for (uint32_t j = 0; j < Z; ++j) {
        const float w2 = w2t[j * H + h], w3 = w3t[j * H + h];
#pragma unroll
        for (int e = 0; e < kMidE; ++e) s[e] = fmaf(d23[e * 128 + j], w2, fmaf(d23[e * 128 + 64 + j], w3, s[e]));
      }
      float h1v[kMidE];
#pragma unroll
      for (int e = 0; e < kMidE; ++e) {
        const uint32_t r = r0 + e;
        h1v[e] = r < a.Bl ? __ldg(a.h1_hi + (size_t)r * a.ldh + h) + __ldg(a.h1_lo + (size_t)r * a.ldh + h) : 0.f;
      }
#pragma unroll
      for (int e = 0; e < kMidE; ++e) {
        const uint32_t r = r0 + e;
        if (r < a.Bl) {
          const float d1 = s[e] * (-expm1f(-h1v[e]));
          a.cd1_hi[(size_t)r * H + h] = d1;
          sq1[e] = fmaf(d1, d1, sq1[e]);
        }
      }
    }
    __syncwarp();
#pragma unroll
    for (int e = 0; e < kMidE; ++e) {
      const uint32_t r = r0 + e;
      if (r >= a.Bl) continue;                     // warp-uniform
      const float s1 = group_sum<32>(sq1[e]);
      const float s23 = group_sum<32>(sq23[e]);
      // row-reduction slots of the GEMM epilogues: lane t reads slot t, fixed shuffle-tree order
      float sq_h1 = 0.f, sq_d4 = 0.f, sq_d5 = 0.f, lrec = 0.f;
      for (uint32_t t = lane; t < a.ns_h; t += 32) { sq_h1 += a.sq_h1[(size_t)t * a.Bl + r]; sq_d4 += a.sq_d4[(size_t)t * a.Bl + r]; }
      for (uint32_t t = lane; t < a.ns_d; t += 32) { sq_d5 += a.sq_d5[(size_t)t * a.Bl + r]; lrec += a.loss_rec[(size_t)t * a.Bl + r]; }
      sq_h1 = group_sum<32>(sq_h1); sq_d4 = group_sum<32>(sq_d4);
      sq_d5 = group_sum<32>(sq_d5); lrec = group_sum<32>(lrec);
      const float n2 = (a.sq_h2[r] + 1.0f) * sq_d5 + (a.sq_z[r] + 1.0f) * sq_d4 + (sq_h1 + 1.0f) * s23 +
                       (a.sq_x[r] + 1.0f) * s1;
      const float norm = fabsf(ratio) * sqrtf(n2);
      const uint32_t p = a.pos_begin + r;
      const bool valid = (p < nv) && (!a.mask || a.mask[p]);
      const float c = valid ? 1.0f / fmaxf(1.0f, norm / a.C) : 0.f;
      const float cc = c * ratio;
      const float loss_s = valid ? a.site_scale * (a.loss_kl[r] + lrec) : 0.f;   // = obs_scale * loss_i
      if (lane == 0) {
        a.lossv[r] = loss_s;
        a.cnt[r] = valid ? 1.0f : 0.f;
        if (a.px_norms) a.px_norms[p] = valid ? norm : 0.f;
        if (a.px_loss) a.px_loss[p] = loss_s;
      }
      for (uint32_t h0 = 0; h0 < H; h0 += 128) {             // batched loads: 12 in flight per lane
        float d1v[4], h2h[4], h2l[4];
#pragma unroll
        for (int t = 0; t < 4; ++t) {
          const uint32_t h = h0 + 32 * t + lane;
          const bool ok = h < H;
          d1v[t] = ok ? a.cd1_hi[(size_t)r * H + h] : 0.f;
          h2h[t] = ok ? __ldg(a.h2_hi + (size_t)r * H + h) : 0.f;      // h2, unmasked
          h2l[t] = 0.f;
        }
#pragma unroll
        for (int t = 0; t < 4; ++t) {
          const uint32_t h = h0 + 32 * t + lane;
          if (h >= H) continue;
          const float v1 = cc * d1v[t];
          a.cd1_hi[(size_t)r * H + h] = v1;          // unmasked: split by the dW1 GEMM itself (tc_gemm_kernel.cuh)
          a.cd1_lo[(size_t)r * H + h] = v1 - tc::tf32_hi(v1);
          const float v4 = cc * d4s[e * H + h];
          const float hi4 = tc::tf32_hi(v4);
          a.cd4_hi[(size_t)r * H + h] = hi4;
          a.cd4_lo[(size_t)r * H + h] = v4 - hi4;
          const float v2 = cc * (h2h[t] + h2l[t]);
          a.ch2_hi[(size_t)r * a.ldh + h] = v2;      // unmasked, as above (dW5 GEMM)
          a.ch2_lo[(size_t)r * a.ldh + h] = v2 - tc::tf32_hi(v2);
        }
      }
      if (lane < 4) {
        const float v = lane == 0 ? cc : 0.f;
        a.ch2_hi[(size_t)r * a.ldh + H + lane] = v;
        a.ch2_lo[(size_t)r * a.ldh + H + lane] = v - tc::tf32_hi(v);
      }
      for (uint32_t j = lane; j < a.ld23; j += 32) {
        const float v = j < 2 * Z ? cc * (j < Z ? d23[e * 128 + j] : d23[e * 128 + 64 + j - Z]) : 0.f;
        const float hi = tc::tf32_hi(v);
        a.cd23_hi[(size_t)r * a.ld23 + j] = hi;
        a.cd23_lo[(size_t)r * a.ld23 + j] = v - hi;
      }
    }
    __syncwarp();
  }
}


// ---- thin layers on warp-level tensor-core MMA ------------------------------------------------------------
// The encoder heads (K = H, N = 2Z), the decoder hidden layer (K = Z, N = H) and their transposes in the backward
// pass are far too thin for a 128-row tcgen05 tile (N = 40, K = 20) and were SIMT loops that re-read the weights
// from shared memory per warp (47 + 55 us of the 0.40 ms step).  Here a CTA of 4 warps owns 16 examples = one
// mma.sync m16n8k8 row block; products are 3xTF32 (a_hi b_hi + a_lo b_hi + a_hi b_lo, fp32 accumulate) like the
// tcgen05 GEMMs.  B operands come from global memory in fragment order (one LDG.128 per lane per 8x8 block:
// {hi(b0), hi(b1), lo(b0), lo(b1)}), written once per step by vae_prep_mid_kernel.  The reduction index is
// permuted so that a lane's two k slots (t, t + 4) are adjacent columns (2t, 2t + 1) in memory: A rows are read
// as 8-byte pairs.  Shapes: H % 8 == 0, Z % 4 == 0, Z <= 32; other shapes keep the SIMT kernels above.
constexpr int kMmaRows = 16;
constexpr int kMmaWarps = 8;              // the kernels are latency-bound (16 rows per CTA): 8 warps split K / N
constexpr int kMmaThreads = kMmaWarps * 32;
constexpr int kMmaTpe = kMmaThreads / kMmaRows;   // threads per example in the element-wise phases

template <int W>
D3P_D float sum_warps(const float (*p)[kMmaRows], int e) {        // fixed order
  float v = p[0][e];
#pragma unroll
  for (int w = 1; w < W; ++w) v += p[w][e];
  return v;
}

D3P_D void mma_tf32(float (&d)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1) {
  asm volatile("mma.sync.aligned.m16n8k8.row.col.f32.tf32.tf32.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
               : "+f"(d[0]), "+f"(d[1]), "+f"(d[2]), "+f"(d[3])
               : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}
// d += a b with a = ah + al, b = (b.x, b.y) + (b.z, b.w); small terms first
D3P_D void mma3(float (&d)[4], const uint32_t (&ah)[4], const uint32_t (&al)[4], const float4& b) {
  mma_tf32(d, al, __float_as_uint(b.x), __float_as_uint(b.y));
  mma_tf32(d, ah, __float_as_uint(b.z), __float_as_uint(b.w));
  mma_tf32(d, ah, __float_as_uint(b.x), __float_as_uint(b.y));
}
// A fragment of rows (g, g + 8) at permuted columns (k0 + 2t, k0 + 2t + 1) from two row pointers
D3P_D void load_a_pair(const float* row_g, const float* row_g8, uint32_t k, uint32_t (&a)[4]) {
  const float2 v0 = *reinterpret_cast<const float2*>(row_g + k), v1 = *reinterpret_cast<const float2*>(row_g8 + k);
  a[0] = __float_as_uint(v0.x); a[1] = __float_as_uint(v1.x); a[2] = __float_as_uint(v0.y); a[3] = __float_as_uint(v1.y);
}
D3P_D void split_a(const float2 v0, const float2 v1, uint32_t (&ah)[4], uint32_t (&al)[4]) {
  const float h0 = tc::tf32_hi(v0.x), h1 = tc::tf32_hi(v1.x), h2 = tc::tf32_hi(v0.y), h3 = tc::tf32_hi(v1.y);
  ah[0] = __float_as_uint(h0); ah[1] = __float_as_uint(h1); ah[2] = __float_as_uint(h2); ah[3] = __float_as_uint(h3);
  al[0] = __float_as_uint(v0.x - h0); al[1] = __float_as_uint(v1.x - h1);
  al[2] = __float_as_uint(v0.y - h2); al[3] = __float_as_uint(v1.y - h3);
}

struct MidFragDims {
  uint32_t ks23, nt23, ks4, nt4, ks4t, nt4t, ks23t, nt23t;
  __host__ __device__ MidFragDims(uint32_t H, uint32_t Z)
      : ks23(H / 8), nt23(2 * Z / 8), ks4((Z + 7) / 8), nt4(H / 8), ks4t(H / 8), nt4t((Z + 7) / 8), ks23t(2 * Z / 8),
        nt23t(H / 8) {}
  __host__ __device__ size_t n23() const { return (size_t)ks23 * nt23 * 32; }
  __host__ __device__ size_t n4() const { return (size_t)ks4 * nt4 * 32; }
  __host__ __device__ size_t n4t() const { return (size_t)ks4t * nt4t * 32; }
  __host__ __device__ size_t n23t() const { return (size_t)ks23t * nt23t * 32; }
};

// One thread per float4: entry (ks, nt, lane) of matrix m holds rows k = 8 ks + 2t, k + 1 of column n = 8 nt + g.
__global__ void vae_prep_mid_kernel(VaeArgs a) {
  const uint32_t H = a.H, Z = a.Z;
  const MidFragDims fd(H, Z);
  const size_t n0 = fd.n23(), n1 = n0 + fd.n4(), n2 = n1 + fd.n4t(), n3 = n2 + fd.n23t();
  const float* __restrict__ W2 = a.params + a.off_w2;
  const float* __restrict__ W3 = a.params + a.off_w3;
  const float* __restrict__ W4 = a.params + a.off_w4;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n3; i += (size_t)gridDim.x * blockDim.x) {
    int m; size_t loc; uint32_t nt_count;
    if (i < n0) { m = 0; loc = i; nt_count = fd.nt23; }
    else if (i < n1) { m = 1; loc = i - n0; nt_count = fd.nt4; }
    else if (i < n2) { m = 2; loc = i - n1; nt_count = fd.nt4t; }
    else { m = 3; loc = i - n2; nt_count = fd.nt23t; }
    const uint32_t lane = (uint32_t)(loc & 31), blk = (uint32_t)(loc >> 5);
    const uint32_t ks = blk / nt_count, nt = blk - ks * nt_count;
    const uint32_t k = 8 * ks + 2 * (lane & 3), n = 8 * nt + (lane >> 2);
    float v[2];
#pragma unroll
    for (int q = 0; q < 2; ++q) {
      const uint32_t kk = k + q;
      float x;
      if (m == 0) x = n < Z ? W2[(size_t)kk * Z + n] : W3[(size_t)kk * Z + n - Z];            // [h][j]
      else if (m == 1) x = kk < Z ? W4[(size_t)kk * H + n] : 0.f;                                // [j][h]
      else if (m == 2) x = n < Z ? W4[(size_t)n * H + kk] : 0.f;                                 // [h][j] = W4[j][h]
      else x = kk < Z ? W2[(size_t)n * Z + kk] : W3[(size_t)n * Z + kk - Z];                     // [j'][h]
      v[q] = x;
    }
    const float h0 = tc::tf32_hi(v[0]), h1 = tc::tf32_hi(v[1]);
    const float4 out = make_float4(h0, h1, v[0] - h0, v[1] - h1);
    float4* dst = m == 0 ? a.wf23 : m == 1 ? a.wf4 : m == 2 ? a.wf4t : a.wf23t;
    dst[loc] = out;
  }
}

// S1 on MMA: encoder heads, guide sample, KL part of the loss, decoder hidden layer for 16 examples per CTA.
__global__ void __launch_bounds__(kMmaThreads) vae_mid_fwd_mma_kernel(VaeArgs a) {
  __shared__ float s_eps[kMmaRows][32];
  __shared__ float s_red[kMmaWarps][kMmaRows][66];            // per-warp partial head sums (K split over the warps)
  __shared__ __align__(8) float s_z[2][kMmaRows][32]; // z hi / lo, zero-padded in k
  __shared__ float s_sq[kMmaWarps][kMmaRows];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, g = lane >> 2, t = lane & 3;
  const uint32_t H = a.H, Z = a.Z;
  const MidFragDims fd(H, Z);
  const uint32_t r0 = blockIdx.x * kMmaRows;
  const uint32_t e8 = threadIdx.x / kMmaTpe, j8 = threadIdx.x % kMmaTpe;     // phase 0 / 2 mapping: kMmaTpe threads per example
  // ---- phase 0: guide noise: key_p -> (_, guide_seed) -> (rng, k_plate) -> (_, k_z); eps = normal(k_z, (Z,)) ----
  for (uint32_t j = j8; j < 32; j += kMmaTpe) { s_z[0][e8][j] = 0.f; s_z[1][e8][j] = 0.f; }
  if (r0 + e8 < a.Bl && a.eval_mode) {
    const TfKey K = tf_key_arg(a.k0, a.k1, a.key_d);
    for (uint32_t j = j8; j < Z; j += kMmaTpe) s_eps[e8][j] = vae_eval_eps(K, a.B, Z, a.pos_begin + r0 + e8, j);
  } else if (r0 + e8 < a.Bl) {
    const TfKey K = tf_key_arg(a.k0, a.k1, a.key_d);
    TfKey kp = tf_example_key(K, a.B, a.pos_begin + r0 + e8);
    TfKey model_seed, guide_seed, rng, k_plate, rng2, k_z;
    tf_split2(kp, model_seed, guide_seed);
    tf_split2(guide_seed, rng, k_plate);
    tf_split2(rng, rng2, k_z);
    const uint32_t half = (Z + 1) / 2;
    for (uint32_t j = j8; j < half; j += kMmaTpe) {
      uint32_t y0, y1;
      const uint32_t c1 = (j + half < Z) ? j + half : 0u;
      threefry2x32(k_z, j, c1, y0, y1);
      s_eps[e8][j] = bits_to_normal<false>(y0);
      if (j + half < Z) s_eps[e8][j + half] = bits_to_normal<false>(y1);
    }
  }
  // ---- phase 1: heads, [16, H] x [H, 2Z]; warp w takes k-steps w, w + 4, ... -----------------------------------
  const uint32_t rg = min(r0 + g, a.Bl - 1), rg8 = min(r0 + g + 8, a.Bl - 1);      // clamped rows (results unused)
  {
    float acc[8][4];
#pragma unroll
    for (int nt = 0; nt < 8; ++nt) { acc[nt][0] = acc[nt][1] = acc[nt][2] = acc[nt][3] = 0.f; }
    const float* ph0 = a.h1_hi + (size_t)rg * a.ldh;
    const float* ph1 = a.h1_hi + (size_t)rg8 * a.ldh;
    const float* pl0 = a.h1_lo + (size_t)rg * a.ldh;
    const float* pl1 = a.h1_lo + (size_t)rg8 * a.ldh;
#pragma unroll 4
    for (uint32_t ks = warp; ks < fd.ks23; ks += kMmaWarps) {
      uint32_t ah[4], al[4];
      load_a_pair(ph0, ph1, 8 * ks + 2 * t, ah);
      load_a_pair(pl0, pl1, 8 * ks + 2 * t, al);
      const float4* bf = a.wf23 + (size_t)ks * fd.nt23 * 32 + lane;
#pragma unroll
      for (int nt = 0; nt < 8; ++nt)
        if ((uint32_t)nt < fd.nt23) mma3(acc[nt], ah, al, __ldg(bf + nt * 32));
    }
#pragma unroll
    for (int nt = 0; nt < 8; ++nt)
      if ((uint32_t)nt < fd.nt23) {
        s_red[warp][g][8 * nt + 2 * t] = acc[nt][0]; s_red[warp][g][8 * nt + 2 * t + 1] = acc[nt][1];
        s_red[warp][g + 8][8 * nt + 2 * t] = acc[nt][2]; s_red[warp][g + 8][8 * nt + 2 * t + 1] = acc[nt][3];
      }
  }
  __syncthreads();
  // ---- phase 2: z = z_loc + exp(log z_std) eps, KL part, operands of the dW4 GEMM ---------------------------
  {
    const uint32_t r = r0 + e8;
    const bool live = r < a.Bl;
    float kl = 0.f, sqz = 0.f;
    for (uint32_t j = j8; j < Z; j += kMmaTpe) {
      float zl = s_red[0][e8][j], sr = s_red[0][e8][Z + j];
#pragma unroll
      for (int w = 1; w < kMmaWarps; ++w) { zl += s_red[w][e8][j]; sr += s_red[w][e8][Z + j]; }
      zl += a.params[a.off_b2 + j];
      sr += a.params[a.off_b3 + j];
      const float eps = live ? s_eps[e8][j] : 0.f;
      const float u = expf(sr) * eps;
      const float z = zl + u;
      const float hi = tc::tf32_hi(z);
      s_z[0][e8][j] = hi; s_z[1][e8][j] = z - hi;
      if (live) {
        a.z_hi[(size_t)r * a.ldz + j] = hi;
        a.z_lo[(size_t)r * a.ldz + j] = z - hi;
        a.u[(size_t)r * Z + j] = u;
      }
      kl += 0.5f * z * z - 0.5f * eps * eps - sr;       // -log N(z;0,1) + log N(z; z_loc, z_std), constants cancel
      sqz = fmaf(z, z, sqz);
    }
    if (live) {
      for (uint32_t j = Z + j8; j < a.ldz; j += kMmaTpe) {      // ones column of [z | 1] (db4 of the dW4 GEMM) + padding
        a.z_hi[(size_t)r * a.ldz + j] = j == Z ? 1.0f : 0.f;
        a.z_lo[(size_t)r * a.ldz + j] = 0.f;
      }
      if (j8 < 4) {                                       // ones column of [H1 | 1] (bias row of the dW2 / dW3 GEMM)
        a.h1_hi[(size_t)r * a.ldh + H + j8] = j8 == 0 ? 1.0f : 0.f;
        a.h1_lo[(size_t)r * a.ldh + H + j8] = 0.f;
      }
    }
#pragma unroll
    for (int o = 1; o < kMmaTpe; o <<= 1) { kl += __shfl_xor_sync(0xffffffffu, kl, o); sqz += __shfl_xor_sync(0xffffffffu, sqz, o); }
    if (j8 == 0 && live) { a.loss_kl[r] = kl; a.sq_z[r] = sqz; }
  }
  __syncthreads();
  // ---- phase 3: decoder hidden layer h2 = softplus(z W4 + b4); warp w takes column blocks w, w + 4, ... --------
  {
    uint32_t zh[4][4], zl[4][4];
#pragma unroll
    for (int ks = 0; ks < 4; ++ks)
      if ((uint32_t)ks < fd.ks4) {
        load_a_pair(&s_z[0][g][0], &s_z[0][g + 8][0], 8 * ks + 2 * t, zh[ks]);
        load_a_pair(&s_z[1][g][0], &s_z[1][g + 8][0], 8 * ks + 2 * t, zl[ks]);
      }
    float sq0 = 0.f, sq1 = 0.f;
    const bool live0 = r0 + g < a.Bl, live1 = r0 + g + 8 < a.Bl;
    for (uint32_t nt = warp; nt < fd.nt4; nt += kMmaWarps) {
      float acc[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
      for (int ks = 0; ks < 4; ++ks)
        if ((uint32_t)ks < fd.ks4) mma3(acc, zh[ks], zl[ks], __ldg(a.wf4 + ((size_t)ks * fd.nt4 + nt) * 32 + lane));
      const uint32_t n = 8 * nt + 2 * t;
      const float2 b = make_float2(a.params[a.off_b4 + n], a.params[a.off_b4 + n + 1]);
      const float v00 = softplus_f(acc[0] + b.x), v01 = softplus_f(acc[1] + b.y);
      const float v10 = softplus_f(acc[2] + b.x), v11 = softplus_f(acc[3] + b.y);
      sq0 = fmaf(v00, v00, fmaf(v01, v01, sq0));
      sq1 = fmaf(v10, v10, fmaf(v11, v11, sq1));
      const float h00 = tc::tf32_hi(v00), h01 = tc::tf32_hi(v01), h10 = tc::tf32_hi(v10), h11 = tc::tf32_hi(v11);
      if (live0) {
        *reinterpret_cast<float2*>(a.h2_hi + (size_t)(r0 + g) * H + n) = make_float2(v00, v01);     // unmasked
        *reinterpret_cast<float2*>(a.h2_lo + (size_t)(r0 + g) * H + n) = make_float2(v00 - h00, v01 - h01);
      }
      if (live1) {
        *reinterpret_cast<float2*>(a.h2_hi + (size_t)(r0 + g + 8) * H + n) = make_float2(v10, v11);
        *reinterpret_cast<float2*>(a.h2_lo + (size_t)(r0 + g + 8) * H + n) = make_float2(v10 - h10, v11 - h11);
      }
    }
    sq0 += __shfl_xor_sync(0xffffffffu, sq0, 1); sq0 += __shfl_xor_sync(0xffffffffu, sq0, 2);
    sq1 += __shfl_xor_sync(0xffffffffu, sq1, 1); sq1 += __shfl_xor_sync(0xffffffffu, sq1, 2);
    if (t == 0) { s_sq[warp][g] = sq0; s_sq[warp][g + 8] = sq1; }
  }
  __syncthreads();
  if (threadIdx.x < kMmaRows && r0 + threadIdx.x < a.Bl)
    a.sq_h2[r0 + threadIdx.x] = sum_warps<kMmaWarps>(s_sq, threadIdx.x);
}

// S2 on MMA: back-propagation through the z layer and the encoder heads, ghost norm, clip factor, scaled operands
// of the clipped-sum GEMMs, 16 examples per CTA.  Dynamic shared memory: raw delta1 [16][H].
__global__ void __launch_bounds__(kMmaThreads) vae_mid_bwd_mma_kernel(VaeArgs a) {
  extern __shared__ __align__(16) float s_d1[];        // [16][H]
  __shared__ float s_red[kMmaWarps][kMmaRows][34];
  __shared__ __align__(8) float s_dh[2][kMmaRows][64]; // [delta2 | delta3] hi / lo (A operand of the dh1 product)
  __shared__ float s_d23[kMmaRows][64];                // unsplit [delta2 | delta3]
  __shared__ float s_sq1[kMmaWarps][kMmaRows];
  __shared__ float s_sq23[kMmaRows], s_cc[kMmaRows];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, g = lane >> 2, t = lane & 3;
  const uint32_t H = a.H, Z = a.Z, Z2 = 2 * a.Z;
  const MidFragDims fd(H, Z);
  const uint32_t r0 = blockIdx.x * kMmaRows;
  const uint32_t e8 = threadIdx.x / kMmaTpe, j8 = threadIdx.x % kMmaTpe;
  const uint32_t rg = min(r0 + g, a.Bl - 1), rg8 = min(r0 + g + 8, a.Bl - 1);
  const bool live0 = r0 + g < a.Bl, live1 = r0 + g + 8 < a.Bl;
  // ---- phase 1: delta4 W4^T, [16, H] x [H, Z]; warp w takes k-steps w, w + 4, ... ------------------------------
  {
    float acc[4][4];
#pragma unroll
    for (int nt = 0; nt < 4; ++nt) { acc[nt][0] = acc[nt][1] = acc[nt][2] = acc[nt][3] = 0.f; }
    const float* p0 = a.d4 + (size_t)rg * H;
    const float* p1 = a.d4 + (size_t)rg8 * H;
#pragma unroll 4
    for (uint32_t ks = warp; ks < fd.ks4t; ks += kMmaWarps) {
      uint32_t ah[4], al[4];
      const uint32_t k = 8 * ks + 2 * t;
      split_a(*reinterpret_cast<const float2*>(p0 + k), *reinterpret_cast<const float2*>(p1 + k), ah, al);
      const float4* bf = a.wf4t + (size_t)ks * fd.nt4t * 32 + lane;
#pragma unroll
      for (int nt = 0; nt < 4; ++nt)
        if ((uint32_t)nt < fd.nt4t) mma3(acc[nt], ah, al, __ldg(bf + nt * 32));
    }
#pragma unroll
    for (int nt = 0; nt < 4; ++nt)
      if ((uint32_t)nt < fd.nt4t) {
        s_red[warp][g][8 * nt + 2 * t] = acc[nt][0]; s_red[warp][g][8 * nt + 2 * t + 1] = acc[nt][1];
        s_red[warp][g + 8][8 * nt + 2 * t] = acc[nt][2]; s_red[warp][g + 8][8 * nt + 2 * t + 1] = acc[nt][3];
      }
  }
  __syncthreads();
  // ---- phase 2: delta_z = z + delta4 W4^T, delta3 = delta_z u - 1 ----------------------------------------------
  {
    const uint32_t r = r0 + e8;
    const bool live = r < a.Bl;
    float sq23 = 0.f;
    for (uint32_t j = j8; j < Z; j += kMmaTpe) {
      const float zv = live ? a.z_hi[(size_t)r * a.ldz + j] + a.z_lo[(size_t)r * a.ldz + j] : 0.f;
      const float uv = live ? a.u[(size_t)r * Z + j] : 0.f;
      float dz = s_red[0][e8][j];
#pragma unroll
      for (int w = 1; w < kMmaWarps; ++w) dz += s_red[w][e8][j];
      dz += zv;
      const float d3 = fmaf(dz, uv, -1.0f);
      s_d23[e8][j] = dz; s_d23[e8][Z + j] = d3;
      const float hz = tc::tf32_hi(dz), h3 = tc::tf32_hi(d3);
      s_dh[0][e8][j] = hz; s_dh[1][e8][j] = dz - hz;
      s_dh[0][e8][Z + j] = h3; s_dh[1][e8][Z + j] = d3 - h3;
      sq23 = fmaf(dz, dz, fmaf(d3, d3, sq23));
    }
#pragma unroll
    for (int o = 1; o < kMmaTpe; o <<= 1) sq23 += __shfl_xor_sync(0xffffffffu, sq23, o);
    if (j8 == 0) s_sq23[e8] = sq23;
  }
  __syncthreads();
  // ---- phase 3: delta_h1 = delta2 W2^T + delta3 W3^T; delta1 = delta_h1 softplus'(pre1); raw delta1 kept in smem -----
  {
    float sq0 = 0.f, sq1 = 0.f;
    const float* ph0 = a.h1_hi + (size_t)rg * a.ldh;
    const float* ph1 = a.h1_hi + (size_t)rg8 * a.ldh;
    const float* pl0 = a.h1_lo + (size_t)rg * a.ldh;
    const float* pl1 = a.h1_lo + (size_t)rg8 * a.ldh;
    for (uint32_t nt = warp; nt < fd.nt23t; nt += kMmaWarps) {
      float acc[4] = {0.f, 0.f, 0.f, 0.f};
      // h1 of this column block is requested before the MMA loop (the MMAs are opaque to the compiler, which would
      // otherwise leave these loads behind them and expose their full latency in every iteration)
      const uint32_t n = 8 * nt + 2 * t;
      const float2 hh0 = __ldg(reinterpret_cast<const float2*>(ph0 + n)), hl0 = __ldg(reinterpret_cast<const float2*>(pl0 + n));
      const float2 hh1 = __ldg(reinterpret_cast<const float2*>(ph1 + n)), hl1 = __ldg(reinterpret_cast<const float2*>(pl1 + n));
      for (uint32_t ks = 0; ks < fd.ks23t; ++ks) {
        uint32_t ah[4], al[4];
        load_a_pair(&s_dh[0][g][0], &s_dh[0][g + 8][0], 8 * ks + 2 * t, ah);
        load_a_pair(&s_dh[1][g][0], &s_dh[1][g + 8][0], 8 * ks + 2 * t, al);
        mma3(acc, ah, al, __ldg(a.wf23t + ((size_t)ks * fd.nt23t + nt) * 32 + lane));
      }
      const float d00 = live0 ? acc[0] * (-expm1f(-(hh0.x + hl0.x))) : 0.f;
      const float d01 = live0 ? acc[1] * (-expm1f(-(hh0.y + hl0.y))) : 0.f;
      const float d10 = live1 ? acc[2] * (-expm1f(-(hh1.x + hl1.x))) : 0.f;
      const float d11 = live1 ? acc[3] * (-expm1f(-(hh1.y + hl1.y))) : 0.f;
      sq0 = fmaf(d00, d00, fmaf(d01, d01, sq0));
      sq1 = fmaf(d10, d10, fmaf(d11, d11, sq1));
      *reinterpret_cast<float2*>(s_d1 + (size_t)g * H + n) = make_float2(d00, d01);
      *reinterpret_cast<float2*>(s_d1 + (size_t)(g + 8) * H + n) = make_float2(d10, d11);
    }
    sq0 += __shfl_xor_sync(0xffffffffu, sq0, 1); sq0 += __shfl_xor_sync(0xffffffffu, sq0, 2);
    sq1 += __shfl_xor_sync(0xffffffffu, sq1, 1); sq1 += __shfl_xor_sync(0xffffffffu, sq1, 2);
    if (t == 0) { s_sq1[warp][g] = sq0; s_sq1[warp][g + 8] = sq1; }
  }
  __syncthreads();
  // ---- phase 4: ghost norm, clip factor, per-example loss -----------------------------------------------------
  {
    const uint32_t r = r0 + e8;
    const bool live = r < a.Bl;
    const uint32_t nv = a.num_valid ? (uint32_t)max(*a.num_valid, 0) : 0xffffffffu;
    const float ratio = a.site_scale * a.inv_S;                   // (1 / obs_scale) * site scale
    float sq_h1 = 0.f, sq_d4 = 0.f, sq_d5 = 0.f, lrec = 0.f;
    if (live) {
      for (uint32_t q = j8; q < a.ns_h; q += kMmaTpe) { sq_h1 += a.sq_h1[(size_t)q * a.Bl + r]; sq_d4 += a.sq_d4[(size_t)q * a.Bl + r]; }
      for (uint32_t q = j8; q < a.ns_d; q += kMmaTpe) { sq_d5 += a.sq_d5[(size_t)q * a.Bl + r]; lrec += a.loss_rec[(size_t)q * a.Bl + r]; }
    }
#pragma unroll
    for (int o = 1; o < kMmaTpe; o <<= 1) {
      sq_h1 += __shfl_xor_sync(0xffffffffu, sq_h1, o); sq_d4 += __shfl_xor_sync(0xffffffffu, sq_d4, o);
      sq_d5 += __shfl_xor_sync(0xffffffffu, sq_d5, o); lrec += __shfl_xor_sync(0xffffffffu, lrec, o);
    }
    if (j8 == 0) {
      float cc = 0.f;
      if (live) {
        const float s1 = sum_warps<kMmaWarps>(s_sq1, e8);
        const float n2 = (a.sq_h2[r] + 1.0f) * sq_d5 + (a.sq_z[r] + 1.0f) * sq_d4 + (sq_h1 + 1.0f) * s_sq23[e8] +
                         (a.sq_x[r] + 1.0f) * s1;
        const float norm = fabsf(ratio) * sqrtf(n2);
        const uint32_t p = a.pos_begin + r;
        const bool valid = (p < nv) && (!a.mask || a.mask[p]);
        const float c = valid ? 1.0f / fmaxf(1.0f, norm / a.C) : 0.f;
        cc = c * ratio;
        const float loss_s = valid ? a.site_scale * (a.loss_kl[r] + lrec) : 0.f;   // = obs_scale * loss_i
        a.lossv[r] = loss_s;
        a.cnt[r] = valid ? 1.0f : 0.f;
        if (a.px_norms) a.px_norms[p] = valid ? norm : 0.f;
        if (a.px_loss) a.px_loss[p] = loss_s;
      }
      s_cc[e8] = cc;
    }
  }
  __syncthreads();
  // ---- phase 5: scaled hi / lo operands of the clipped-sum GEMMs (streaming) ---------------------------------------
  const uint32_t H4 = H / 4;
  const uint32_t n_stream = min((uint32_t)kMmaRows, a.Bl - r0) * H4;      // the rows of this CTA that exist
#pragma unroll 4
  for (uint32_t i = threadIdx.x; i < n_stream; i += kMmaThreads) {
    const uint32_t e = i / H4, h = 4 * (i - e * H4), r = r0 + e;
    const float cc = s_cc[e];
    const float4 d1 = *reinterpret_cast<const float4*>(s_d1 + (size_t)e * H + h);
    const float4 d4 = *reinterpret_cast<const float4*>(a.d4 + (size_t)r * H + h);
    const float4 hh = *reinterpret_cast<const float4*>(a.h2_hi + (size_t)r * H + h);      // h2, unmasked
    float4 o_hi, o_lo;
#define D3P_SPLIT4(src_x, src_y, src_z, src_w)                                                     \
    { const float vx = (src_x), vy = (src_y), vz = (src_z), vw = (src_w);                          \
      o_hi = make_float4(tc::tf32_hi(vx), tc::tf32_hi(vy), tc::tf32_hi(vz), tc::tf32_hi(vw));      \
      o_lo = make_float4(vx - o_hi.x, vy - o_hi.y, vz - o_hi.z, vw - o_hi.w); }
    // c delta1 and c h2 go out unsplit: the dW1 / dW5 GEMMs make their lo parts in shared memory (GemmOperand::split)
    *reinterpret_cast<float4*>(a.cd1_hi + (size_t)r * H + h) = make_float4(cc * d1.x, cc * d1.y, cc * d1.z, cc * d1.w);
    D3P_SPLIT4(cc * d4.x, cc * d4.y, cc * d4.z, cc * d4.w)
    *reinterpret_cast<float4*>(a.cd4_hi + (size_t)r * H + h) = o_hi;
    *reinterpret_cast<float4*>(a.cd4_lo + (size_t)r * H + h) = o_lo;
    *reinterpret_cast<float4*>(a.ch2_hi + (size_t)r * a.ldh + h) =
        make_float4(cc * hh.x, cc * hh.y, cc * hh.z, cc * hh.w);
#undef D3P_SPLIT4
  }
  {
    const uint32_t r = r0 + e8;
    if (r < a.Bl) {
      const float cc = s_cc[e8];
      if (j8 < 4) {
        const float v = j8 == 0 ? cc : 0.f;
        a.ch2_hi[(size_t)r * a.ldh + H + j8] = v;          // unmasked; the dW5 GEMM never reads ch2_lo

      }
      for (uint32_t j = j8; j < a.ld23; j += kMmaTpe) {
        const float v = j < Z2 ? cc * s_d23[e8][j] : 0.f;
        const float hi = tc::tf32_hi(v);
        a.cd23_hi[(size_t)r * a.ld23 + j] = hi;
        a.cd23_lo[(size_t)r * a.ld23 + j] = v - hi;
      }
    }
  }
}

// DPSVI.evaluate: loss = site scale of the evaluation trace (N / B) * (1 / N) = 1 / B, times sum_i (kl_i + rec_i);
// one CTA, fixed order.
__global__ void __launch_bounds__(1024) vae_eval_reduce_kernel(VaeArgs a, float* __restrict__ loss_out) {
  __shared__ float red[32];
  float s = 0.f;
  for (uint32_t r = threadIdx.x; r < a.Bl; r += 1024) {
    float l = a.loss_kl[r];
    for (uint32_t t = 0; t < a.ns_d; ++t) l += a.loss_rec[(size_t)t * a.Bl + r];
    s += l;
  }
  s = group_sum<32>(s);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = s;
  __syncthreads();
  if (threadIdx.x == 0) {
    float tot = 0.f;
#pragma unroll
    for (int w = 0; w < 32; ++w) tot += red[w];
    *loss_out = tot * (a.site_scale / (float)a.B);
  }
}

// loss / count columns of the partial rows: slab s = a contiguous range of examples, summed in a fixed order
__global__ void __launch_bounds__(256) vae_loss_kernel(VaeArgs a) {
  __shared__ float red[2][8];
  const uint32_t per = (a.Bl + a.S - 1) / a.S;
  const uint32_t i0 = blockIdx.x * per, i1 = min(a.Bl, i0 + per);
  float ls = 0.f, cn = 0.f;
  for (uint32_t i = i0 + threadIdx.x; i < i1; i += 256) { ls += a.lossv[i]; cn += a.cnt[i]; }
  ls = group_sum<32>(ls);
  cn = group_sum<32>(cn);
  if ((threadIdx.x & 31) == 0) { red[0][threadIdx.x >> 5] = ls; red[1][threadIdx.x >> 5] = cn; }
  __syncthreads();
  if (threadIdx.x == 0) {
    float l = 0.f, c = 0.f;
    for (int w = 0; w < 8; ++w) { l += red[0][w]; c += red[1][w]; }
    a.partials[(size_t)blockIdx.x * (a.P + 2) + a.P] = l;
    a.partials[(size_t)blockIdx.x * (a.P + 2) + a.P + 1] = c;
  }
}

// ---- host --------------------------------------------------------------------------------------------
constexpr int kHeavyEW = 16;           // epilogue warps of the GEMMs with transcendental epilogues
constexpr int kThinBN = 64;            // N tile of the two thin clipped-sum GEMMs (N = 2Z and Z + 1)

struct VaeLayout {
  size_t total;
  size_t partials, w1_hi, w1_lo, w5_hi, w5_lo, x_hi, x_lo, flag, h1_hi, h1_lo, h2_hi, h2_lo, ch2_hi, ch2_lo, d5_hi, d5_lo,
      d4, cd4_hi, cd4_lo, cd1_hi, cd1_lo, z_hi, z_lo, u, cd23_hi, cd23_lo, sq_x, sq_h1, sq_h2, sq_z, sq_d5, loss_rec, sq_d4,
      loss_kl, lossv, cnt, wf23, wf4, wf4t, wf23t;
  uint32_t S, ns_h, ns_d;
  size_t ldx, ldh, ldz, ld23;
};

// Batch splits of the clipped-sum GEMMs = partial rows.  The four GEMMs (dW1, dW5, dW2|dW3, dW4) are independent and
// run concurrently (forked streams), every CTA owns one SM (the operand ring takes the whole shared memory), so the
// split count is chosen to put all their CTAs on the GPU in ONE wave with as many k-blocks per CTA as possible
// (784-400-20: 36 tiles -> 4 splits = 144 CTAs of 32 k-blocks; the old 10 splits ran 140-CTA grids of 13 k-blocks back
// to back, each paying its prologue, pipeline fill and epilogue).
static uint32_t vae_splits(const d3p_vae_desc* d, uint32_t Bl) {
  const uint32_t kb = (Bl + tc::kKB - 1) / tc::kKB;
  auto tiles = [](uint32_t m, uint32_t n, uint32_t bn) { return ((m + tc::kBM - 1) / tc::kBM) * ((n + bn - 1) / bn); };
  const uint32_t D = d->out_dim, H = d->hidden_dim, Z = d->z_dim;
  const uint32_t total = tiles(D + 1, H, kVaeBN) + tiles(D, H + 1, kVaeBN) + tiles(H + 1, 2 * Z, kThinBN) + tiles(H, Z + 1, kThinBN);
  uint32_t s = (uint32_t)sm_count() / (total ? total : 1);
  if (s > 10) s = 10;
  if (s > kb) s = kb;
  return s ? s : 1;
}

static VaeLayout vae_layout(const d3p_vae_desc* d, uint32_t Bl) {
  VaeLayout L;
  const size_t D = d->out_dim, H = d->hidden_dim, Z = d->z_dim, P = d->n_params;
  L.S = vae_splits(d, Bl);
  L.ns_h = (uint32_t)((H + kVaeBNH - 1) / kVaeBNH) * (kHeavyEW / 4);
  L.ns_d = (uint32_t)((D + kVaeBN - 1) / kVaeBN) * (kHeavyEW / 4);
  L.ldx = D + 4; L.ldh = H + 4; L.ldz = (Z + 1 + 3) / 4 * 4; L.ld23 = (2 * Z + 3) / 4 * 4;
  size_t off = 0;
  auto take = [&](size_t floats) { size_t o = off; off += align_up(floats * sizeof(float), 256); return o; };
  L.partials = take((size_t)L.S * (P + 2));
  L.w1_hi = take(D * H); L.w1_lo = take(D * H); L.w5_hi = take(H * D); L.w5_lo = take(H * D);
  L.x_hi = take((size_t)Bl * L.ldx); L.x_lo = take((size_t)Bl * L.ldx); L.flag = take(4);
  L.h1_hi = take((size_t)Bl * L.ldh); L.h1_lo = take((size_t)Bl * L.ldh);
  L.h2_hi = take((size_t)Bl * H); L.h2_lo = take((size_t)Bl * H);
  L.ch2_hi = take((size_t)Bl * L.ldh); L.ch2_lo = take((size_t)Bl * L.ldh);
  L.d5_hi = take((size_t)Bl * D); L.d5_lo = take((size_t)Bl * D);
  L.d4 = take((size_t)Bl * H); L.cd4_hi = take((size_t)Bl * H); L.cd4_lo = take((size_t)Bl * H);
  L.cd1_hi = take((size_t)Bl * H); L.cd1_lo = take((size_t)Bl * H);
  L.z_hi = take((size_t)Bl * L.ldz); L.z_lo = take((size_t)Bl * L.ldz); L.u = take((size_t)Bl * Z);
  L.cd23_hi = take((size_t)Bl * L.ld23); L.cd23_lo = take((size_t)Bl * L.ld23);
  L.sq_x = take(Bl); L.sq_h1 = take((size_t)L.ns_h * Bl); L.sq_h2 = take(Bl); L.sq_z = take(Bl);
  L.sq_d5 = take((size_t)L.ns_d * Bl); L.loss_rec = take((size_t)L.ns_d * Bl); L.sq_d4 = take((size_t)L.ns_h * Bl);
  L.loss_kl = take(Bl); L.lossv = take(Bl); L.cnt = take(Bl);
  {
    const MidFragDims fd((uint32_t)H, (uint32_t)Z);          // float4 entries (sized for every shape: a few hundred KB)
    L.wf23 = take(4 * fd.n23()); L.wf4 = take(4 * fd.n4()); L.wf4t = take(4 * fd.n4t()); L.wf23t = take(4 * fd.n23t());
  }
  L.total = off;
  return L;
}

static size_t mid_fwd_smem_bytes(uint32_t H, uint32_t Z) {
  return ((size_t)H * 2 * Z + (size_t)Z * H + 64 + H + (size_t)kMidWarps * kMidE * (H + 3 * 64)) * sizeof(float);
}
static size_t mid_bwd_smem_bytes(uint32_t H, uint32_t Z) {
  return (3 * (size_t)Z * H + (size_t)kMidWarps * kMidE * (H + 128)) * sizeof(float);
}

}  // namespace d3p

// Side streams for the four independent clipped-sum GEMMs (and the small preparation kernels): CALLER-OWNED
// (d3p_vae_ctx_create / _destroy; the library keeps no global state).  `mu` serialises the fork / join bookkeeping
// should two host threads share one context.
struct d3p_vae_ctx {
  std::mutex mu;
  cudaStream_t s[3];
  cudaEvent_t fork, join[3];
};

namespace d3p {
using VaeSideStreams = d3p_vae_ctx;

static bool vae_supported(const d3p_vae_desc* d) {
  return d && d->out_dim >= 4 && d->hidden_dim >= 4 && d->z_dim >= 1 && d->z_dim <= 32 && (d->out_dim % 4) == 0 &&
         (d->hidden_dim % 4) == 0 && mid_fwd_smem_bytes(d->hidden_dim, d->z_dim) <= 220 * 1024 &&
         mid_bwd_smem_bytes(d->hidden_dim, d->z_dim) <= 220 * 1024;
}

}  // namespace d3p

using namespace d3p;

extern "C" size_t d3p_vae_workspace_bytes(const d3p_vae_desc* desc, uint32_t batch_rows, uint32_t* n_partials_out) {
  if (!vae_supported(desc) || batch_rows == 0) return 0;
  VaeLayout L = vae_layout(desc, batch_rows);
  if (n_partials_out) *n_partials_out = L.S;
  return L.total;
}

extern "C" int32_t d3p_vae_ctx_create(d3p_vae_ctx** ctx_out) {
  if (!ctx_out) return D3P_ERR_INVALID_ARGUMENT;
  d3p_vae_ctx* v = new (std::nothrow) d3p_vae_ctx();
  if (!v) return D3P_ERR_CUDA;
  bool ok = cudaEventCreateWithFlags(&v->fork, cudaEventDisableTiming) == cudaSuccess;
  int made = 0;
  for (int i = 0; i < 3 && ok; ++i) {
    ok = cudaStreamCreateWithFlags(&v->s[i], cudaStreamNonBlocking) == cudaSuccess &&
         cudaEventCreateWithFlags(&v->join[i], cudaEventDisableTiming) == cudaSuccess;
    if (ok) ++made;
  }
  if (!ok) {
    for (int i = 0; i < made; ++i) { cudaStreamDestroy(v->s[i]); cudaEventDestroy(v->join[i]); }
    delete v;
    return D3P_ERR_CUDA;
  }
  *ctx_out = v;
  return D3P_OK;
}

// Returns at once; streams and events are released by the runtime when the work queued on them has drained.
extern "C" int32_t d3p_vae_ctx_destroy(d3p_vae_ctx* ctx) {
  if (!ctx) return D3P_ERR_INVALID_ARGUMENT;
  for (int i = 0; i < 3; ++i) { cudaStreamDestroy(ctx->s[i]); cudaEventDestroy(ctx->join[i]); }
  cudaEventDestroy(ctx->fork);
  delete ctx;
  return D3P_OK;
}

int32_t d3p::step_vae_impl(const d3p_vae_desc* desc, const float* params_d, const float* x_d, size_t x_row_stride,
                           const int32_t* idx_d, const uint8_t* mask_d, const int32_t* num_valid_d, uint32_t B,
                           uint32_t pos_begin, uint32_t pos_end, const uint32_t* threefry_key_h,
                           const uint32_t* threefry_key_d, float obs_scale, float C, float* px_norms_d,
                           float* px_loss_d, void* ws_d, size_t ws_bytes, void* const* profile_events_h,
                           d3p_vae_ctx* ctx, void* stream, float* eval_loss_d) {
  if (!desc || !params_d || !x_d || (!threefry_key_h && !threefry_key_d) || !ws_d) return D3P_ERR_INVALID_ARGUMENT;
  if (!vae_supported(desc)) return D3P_ERR_UNSUPPORTED;
  if (pos_end > B || pos_begin >= pos_end || !(C > 0.f) || !(obs_scale != 0.f)) return D3P_ERR_INVALID_ARGUMENT;
  if (reinterpret_cast<uintptr_t>(ws_d) & 255) return D3P_ERR_INVALID_ARGUMENT;
  const uint32_t Bl = pos_end - pos_begin;
  const VaeLayout L = vae_layout(desc, Bl);
  if (ws_bytes < L.total) return D3P_ERR_WORKSPACE;
  cudaStream_t s = (cudaStream_t)stream;
  char* ws = static_cast<char*>(ws_d);
  auto F = [&](size_t off) { return reinterpret_cast<float*>(ws + off); };
  const uint32_t D = desc->out_dim, H = desc->hidden_dim, Z = desc->z_dim, P = desc->n_params;

  VaeArgs a;
  memset(&a, 0, sizeof(a));
  a.D = D; a.H = H; a.Z = Z; a.B = B; a.Bl = Bl; a.pos_begin = pos_begin;
  a.ldx = L.ldx; a.ldh = L.ldh; a.ldz = L.ldz; a.ld23 = L.ld23;
  a.params = params_d;
  a.off_w4 = desc->off_w4; a.off_b4 = desc->off_b4; a.off_w5 = desc->off_w5; a.off_b5 = desc->off_b5;
  a.off_w1 = desc->off_w1; a.off_b1 = desc->off_b1; a.off_w2 = desc->off_w2; a.off_b2 = desc->off_b2;
  a.off_w3 = desc->off_w3; a.off_b3 = desc->off_b3; a.P = P;
  a.x = x_d; a.x_stride = x_row_stride; a.idx = idx_d; a.mask = mask_d; a.num_valid = num_valid_d;
  a.k0 = threefry_key_h ? threefry_key_h[0] : 0u; a.k1 = threefry_key_h ? threefry_key_h[1] : 0u;
  a.key_d = threefry_key_d;
  a.eval_mode = eval_loss_d ? 1 : 0;
  a.site_scale = desc->site_scale; a.inv_S = 1.0f / obs_scale; a.C = C;
  a.ns_h = L.ns_h; a.ns_d = L.ns_d; a.S = L.S;
  a.x_hi = F(L.x_hi); a.x_lo = F(L.x_lo); a.x_lo_flag = reinterpret_cast<int*>(ws + L.flag);
  a.h1_hi = F(L.h1_hi); a.h1_lo = F(L.h1_lo); a.h2_hi = F(L.h2_hi); a.h2_lo = F(L.h2_lo);
  a.ch2_hi = F(L.ch2_hi); a.ch2_lo = F(L.ch2_lo); a.d5_hi = F(L.d5_hi); a.d5_lo = F(L.d5_lo);
  a.d4 = F(L.d4); a.cd4_hi = F(L.cd4_hi); a.cd4_lo = F(L.cd4_lo); a.cd1_hi = F(L.cd1_hi); a.cd1_lo = F(L.cd1_lo);
  a.z_hi = F(L.z_hi); a.z_lo = F(L.z_lo); a.u = F(L.u); a.cd23_hi = F(L.cd23_hi); a.cd23_lo = F(L.cd23_lo);
  a.sq_x = F(L.sq_x); a.sq_h1 = F(L.sq_h1); a.sq_h2 = F(L.sq_h2); a.sq_z = F(L.sq_z); a.sq_d5 = F(L.sq_d5);
  a.loss_rec = F(L.loss_rec); a.sq_d4 = F(L.sq_d4); a.loss_kl = F(L.loss_kl); a.lossv = F(L.lossv); a.cnt = F(L.cnt);
  a.partials = F(L.partials);
  a.px_norms = px_norms_d; a.px_loss = px_loss_d;
  a.wf23 = reinterpret_cast<float4*>(ws + L.wf23); a.wf4 = reinterpret_cast<float4*>(ws + L.wf4);
  a.wf4t = reinterpret_cast<float4*>(ws + L.wf4t); a.wf23t = reinterpret_cast<float4*>(ws + L.wf23t);
  // thin layers: warp-MMA kernels for the shapes they tile (H % 8 == 0, Z % 4 == 0), SIMT kernels otherwise
  const bool mid_mma = (H % 8) == 0 && (Z % 4) == 0 && Z <= 32;
  float* w1_hi = F(L.w1_hi); float* w1_lo = F(L.w1_lo); float* w5_hi = F(L.w5_hi); float* w5_lo = F(L.w5_lo);

  const int sms = sm_count();
  int32_t rc;
  // parameter splits + X preparation: four independent small kernels; the weight splits and the thin-layer fragments
  // run on side streams beside the X preparation (the longest of them)
  VaeSideStreams* ss = ctx;               // nullptr: everything on the caller's stream
  {
    std::unique_lock<std::mutex> lk;
    cudaStream_t sw = s, sm = s;
    if (ss) {
      lk = std::unique_lock<std::mutex>(ss->mu);
      if (cudaEventRecord(ss->fork, s) != cudaSuccess) return D3P_ERR_CUDA;
      for (int i = 0; i < 2; ++i)
        if (cudaStreamWaitEvent(ss->s[i], ss->fork, 0) != cudaSuccess) return D3P_ERR_CUDA;
      sw = ss->s[0]; sm = ss->s[1];
    }
    if ((rc = d3p_split_tf32(params_d + a.off_w1, nullptr, 0, w1_hi, w1_lo, (size_t)D * H, sw)) != D3P_OK) return rc;
    if ((rc = d3p_split_tf32(params_d + a.off_w5, nullptr, 0, w5_hi, w5_lo, (size_t)H * D, sw)) != D3P_OK) return rc;
    if (mid_mma) {
      const MidFragDims fd(H, Z);
      const size_t n = fd.n23() + fd.n4() + fd.n4t() + fd.n23t();
      vae_prep_mid_kernel<<<(unsigned)((n + 255) / 256), 256, 0, sm>>>(a);
      if ((rc = check_launch()) != D3P_OK) return rc;
    }
    if (cudaMemsetAsync(a.x_lo_flag, 0, sizeof(int), s) != cudaSuccess) return D3P_ERR_CUDA;
    unsigned grid = (Bl + 7) / 8;
    if (grid > (unsigned)sms * 8) grid = sms * 8;
    if ((reinterpret_cast<uintptr_t>(x_d) & 15) == 0 && (x_row_stride & 3) == 0) vae_prep_x_kernel<true><<<grid, 256, 0, s>>>(a);
    else vae_prep_x_kernel<false><<<grid, 256, 0, s>>>(a);
    if ((rc = check_launch()) != D3P_OK) return rc;
    if (ss)
      for (int i = 0; i < 2; ++i)
        if (cudaEventRecord(ss->join[i], ss->s[i]) != cudaSuccess || cudaStreamWaitEvent(s, ss->join[i], 0) != cudaSuccess)
          return D3P_ERR_CUDA;
  }
  // G1: pre1 = X W1  (A = X K-major [Bl, D]; B = W1 stored [K = D, N = H])
  {
    tc::GemmOperand A{a.x_hi, a.x_lo, 0, a.ldx}, Bo{w1_hi, w1_lo, 1, H};
    EpiFwd1::Args ea{params_d + a.off_b1, a.h1_hi, a.h1_lo, a.ldh, a.sq_h1, Bl};
    if ((rc = tc::launch_tc_gemm<false, true, kVaeBNH, EpiFwd1, kHeavyEW>(A, Bo, Bl, H, D, 1, ea, s, a.x_lo_flag)) != D3P_OK)
      return rc;
  }
  const size_t mid_fwd_smem = mid_fwd_smem_bytes(H, Z), mid_bwd_smem = mid_bwd_smem_bytes(H, Z);
  unsigned mid_grid = ((Bl + kMidE - 1) / kMidE + kMidWarps - 1) / kMidWarps;
  if (mid_grid > (unsigned)sms) mid_grid = sms;
  const unsigned mma_grid = (Bl + kMmaRows - 1) / kMmaRows;
  if (mid_mma) {
    vae_mid_fwd_mma_kernel<<<mma_grid, kMmaThreads, 0, s>>>(a);
    if ((rc = check_launch()) != D3P_OK) return rc;
  } else {
    if (cudaFuncSetAttribute(vae_mid_fwd_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)mid_fwd_smem) != cudaSuccess)
      return D3P_ERR_CUDA;
    vae_mid_fwd_kernel<<<mid_grid, kMidWarps * 32, mid_fwd_smem, s>>>(a);
    if ((rc = check_launch()) != D3P_OK) return rc;
  }
  // G5: logits = H2 W5  (B = W5 stored [K = H, N = D])
  {
    tc::GemmOperand A{a.h2_hi, nullptr, 0, H, 1}, Bo{params_d + a.off_w5, nullptr, 1, D, 1};   // both split in the kernel
    EpiFwd5::Args ea{params_d + a.off_b5, a.x_hi, a.ldx, a.d5_hi, a.d5_lo, D, a.sq_d5, a.loss_rec, Bl};
    if ((rc = tc::launch_tc_gemm<false, true, kVaeBN, EpiFwd5, kHeavyEW>(A, Bo, Bl, D, H, 1, ea, s, nullptr)) != D3P_OK)
      return rc;
  }
  if (eval_loss_d) {       // DPSVI.evaluate: the forward pass is all there is; loss = (1 / B) sum_i (kl_i + rec_i) * N * (1 / N)
    vae_eval_reduce_kernel<<<1, 1024, 0, s>>>(a, eval_loss_d);
    return check_launch();
  }
  // G5b: dh2 = delta5 W5^T  (B[n = h, k = d] = W5[h, d]: K-major)
  {
    tc::GemmOperand A{a.d5_hi, a.d5_lo, 0, D}, Bo{w5_hi, w5_lo, 0, D};     // pre-split: the in-kernel split measured slower here
    EpiBwd5::Args ea{a.h2_hi, a.h2_lo, H, a.d4, a.sq_d4, Bl};
    if ((rc = tc::launch_tc_gemm<false, false, kVaeBNH, EpiBwd5, kHeavyEW>(A, Bo, Bl, H, D, 1, ea, s, nullptr)) != D3P_OK)
      return rc;
  }
  if (mid_mma) {
    const size_t smem = (size_t)kMmaRows * H * sizeof(float);
    if (smem > 24 * 1024 &&
        cudaFuncSetAttribute(vae_mid_bwd_mma_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess)
      return D3P_ERR_CUDA;
    vae_mid_bwd_mma_kernel<<<mma_grid, kMmaThreads, smem, s>>>(a);
    if ((rc = check_launch()) != D3P_OK) return rc;
  } else {
    if (cudaFuncSetAttribute(vae_mid_bwd_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)mid_bwd_smem) != cudaSuccess)
      return D3P_ERR_CUDA;
    vae_mid_bwd_kernel<<<mid_grid, kMidWarps * 32, mid_bwd_smem, s>>>(a);
    if ((rc = check_launch()) != D3P_OK) return rc;
  }
  // The four clipped-sum GEMMs are independent: GW1 stays on the caller's stream, GW5 / GW23 / GW4 run on side streams
  // forked from it and joined at the end of the step (one wave of CTAs, see vae_splits).  The optional profile events
  // (bench) bracket the whole concurrent group on the caller's stream.
  if (profile_events_h && cudaEventRecord((cudaEvent_t)profile_events_h[0], s) != cudaSuccess) return D3P_ERR_CUDA;
  std::unique_lock<std::mutex> ss_lock;
  cudaStream_t s5 = s, s23 = s, s4 = s;
  if (ss) {
    ss_lock = std::unique_lock<std::mutex>(ss->mu);
    if (cudaEventRecord(ss->fork, s) != cudaSuccess) return D3P_ERR_CUDA;
    for (int i = 0; i < 3; ++i)
      if (cudaStreamWaitEvent(ss->s[i], ss->fork, 0) != cudaSuccess) return D3P_ERR_CUDA;
    s5 = ss->s[0]; s23 = ss->s[1]; s4 = ss->s[2];
  }
  // GW23: [H1 | 1]^T (c [delta2 | delta3]) -> dW2, dW3 [H, Z] and db2, db3   (thin GEMMs first: they are short)
  {
    tc::GemmOperand A{a.h1_hi, a.h1_lo, 1, a.ldh}, Bo{a.cd23_hi, a.cd23_lo, 1, a.ld23};
    EpiGrad::Args ea{a.partials, (size_t)P + 2, a.off_w2, a.off_b2, Z, H, 0, Z, a.off_w3, a.off_b3};
    if ((rc = tc::launch_tc_gemm<true, true, kThinBN, EpiGrad>(A, Bo, H + 1, 2 * Z, Bl, L.S, ea, s23, nullptr)) != D3P_OK) return rc;
  }
  // the (loss, count) columns of the partial rows need the thin-layer kernel's per-example values only, and no GEMM
  // epilogue touches those two columns: behind the short GW23 on its side stream, off the critical path
  vae_loss_kernel<<<L.S, 256, 0, s23>>>(a);
  if ((rc = check_launch()) != D3P_OK) return rc;
  // GW4: (c delta4)^T [z | 1] -> dW4^T (stored [Z, H]) and db4
  {
    tc::GemmOperand A{a.cd4_hi, a.cd4_lo, 1, H}, Bo{a.z_hi, a.z_lo, 1, a.ldz};
    EpiGrad::Args ea{a.partials, (size_t)P + 2, a.off_w4, a.off_b4, H, Z, 1, 0, 0, 0};
    if ((rc = tc::launch_tc_gemm<true, true, kThinBN, EpiGrad>(A, Bo, H, Z + 1, Bl, L.S, ea, s4, nullptr)) != D3P_OK) return rc;
  }
  // GW1: [X | 1]^T (c delta1) -> dW1 [D, H] and db1; contraction over the batch
  {
    tc::GemmOperand A{a.x_hi, a.x_lo, 1, a.ldx}, Bo{a.cd1_hi, nullptr, 1, H, 1};      // c delta1: split in the kernel
    EpiGrad::Args ea{a.partials, (size_t)P + 2, a.off_w1, a.off_b1, H, D, 0, 0, 0, 0};
    if ((rc = tc::launch_tc_gemm<true, true, kVaeBN, EpiGrad, kHeavyEW>(A, Bo, D + 1, H, Bl, L.S, ea, s, a.x_lo_flag)) != D3P_OK) return rc;
  }
  // GW5: delta5^T [c h2 | c] -> dW5^T (stored [H, D]) and db5
  {
    tc::GemmOperand A{a.d5_hi, nullptr, 1, D, 1}, Bo{a.ch2_hi, nullptr, 1, a.ldh, 1};   // both split in the kernel
    EpiGrad::Args ea{a.partials, (size_t)P + 2, a.off_w5, a.off_b5, D, H, 1, 0, 0, 0};
    if ((rc = tc::launch_tc_gemm<true, true, kVaeBN, EpiGrad, kHeavyEW>(A, Bo, D, H + 1, Bl, L.S, ea, s5, nullptr)) != D3P_OK) return rc;
  }
  if (ss) {
    for (int i = 0; i < 3; ++i)
      if (cudaEventRecord(ss->join[i], ss->s[i]) != cudaSuccess || cudaStreamWaitEvent(s, ss->join[i], 0) != cudaSuccess)
        return D3P_ERR_CUDA;
    ss_lock.unlock();
  }
  if (profile_events_h && cudaEventRecord((cudaEvent_t)profile_events_h[1], s) != cudaSuccess) return D3P_ERR_CUDA;
  return D3P_OK;
}

extern "C" int32_t d3p_dpsvi_step_vae(const d3p_vae_desc* desc, const float* params_d, const float* x_d,
                                      size_t x_row_stride, const int32_t* idx_d, const uint8_t* mask_d,
                                      const int32_t* num_valid_d, uint32_t B, uint32_t pos_begin, uint32_t pos_end,
                                      const uint32_t threefry_key_h[2], float obs_scale, float C, float* px_norms_d,
                                      float* px_loss_d, void* ws_d, size_t ws_bytes, void* const* profile_events_h,
                                      d3p_vae_ctx* ctx, void* stream) {
  if (!threefry_key_h) return D3P_ERR_INVALID_ARGUMENT;
  return step_vae_impl(desc, params_d, x_d, x_row_stride, idx_d, mask_d, num_valid_d, B, pos_begin, pos_end, threefry_key_h,
                       nullptr, obs_scale, C, px_norms_d, px_loss_d, ws_d, ws_bytes, profile_events_h, ctx, stream);
}

// Device-key form (see d3p_dpsvi_step_meanfield_dk).
extern "C" int32_t d3p_dpsvi_step_vae_dk(const d3p_vae_desc* desc, const float* params_d, const float* x_d,
                                         size_t x_row_stride, const int32_t* idx_d, const uint8_t* mask_d,
                                         const int32_t* num_valid_d, uint32_t B, uint32_t pos_begin, uint32_t pos_end,
                                         const uint32_t* threefry_key_d, float obs_scale, float C, float* px_norms_d,
                                         float* px_loss_d, void* ws_d, size_t ws_bytes, void* const* profile_events_h,
                                         d3p_vae_ctx* ctx, void* stream) {
  if (!threefry_key_d) return D3P_ERR_INVALID_ARGUMENT;
  return step_vae_impl(desc, params_d, x_d, x_row_stride, idx_d, mask_d, num_valid_d, B, pos_begin, pos_end, nullptr,
                       threefry_key_d, obs_scale, C, px_norms_d, px_loss_d, ws_d, ws_bytes, profile_events_h, ctx, stream);
}

// DPSVI.evaluate for the VAE (d3p/svi.py:436-449; examples/vae.py:236-247 evaluates the test loss every epoch): the
// forward half of the step on the whole batch with ONE guide draw z [B, Z] from `threefry_key_h` = numpyro's
// rng_key_eval; *loss_d = -ELBO under the evaluation trace's scale (N / B) * (1 / N).  Workspace as for the step.
extern "C" int32_t d3p_elbo_evaluate_vae(const d3p_vae_desc* desc, const float* params_d, const float* x_d,
                                         size_t x_row_stride, const int32_t* idx_d, uint32_t B,
                                         const uint32_t threefry_key_h[2], float* loss_d, void* ws_d, size_t ws_bytes,
                                         d3p_vae_ctx* ctx, void* stream) {
  if (!loss_d || !threefry_key_h || B == 0) return D3P_ERR_INVALID_ARGUMENT;
  return step_vae_impl(desc, params_d, x_d, x_row_stride, idx_d, nullptr, nullptr, B, 0, B, threefry_key_h, nullptr, 1.0f, 1.0f,
                       nullptr, nullptr, ws_d, ws_bytes, nullptr, ctx, stream, loss_d);
}
