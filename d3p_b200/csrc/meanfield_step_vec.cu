// K5a/K5b fast path: the fused mean-field step for "full" shapes d = 64 * NQ (256, 512, 1024),
// one warp per example, 4 consecutive latent elements per lane and float4 everywhere
// (LDG.128 row loads, LDS.128 parameter reads).  Same math and same random streams as the generic
// kernel in meanfield_step.cu (that file documents the algebra), and the same per-example ELBO terms
// (meanfield_common.cuh); this one removes the per-slot
// predicates, keeps the Gaussian transform branch-free (one warp-uniform tail fix-up per 4
// variates) and exposes 4-8 independent Threefry / erf_inv chains per lane to the scheduler.
#include "common.cuh"
#include "launch.cuh"
#include "meanfield_common.cuh"

namespace d3p {

D3P_D float4 ld4(const float* p) { return *reinterpret_cast<const float4*>(p); }
D3P_D float4 ldg4(const float* p) { return __ldg(reinterpret_cast<const float4*>(p)); }

#define D3P_F4_FOREACH(OP) OP(x) OP(y) OP(z) OP(w)

// 4 Threefry calls (q, q + HALF), q = q0..q0+3 -> normals for the low and the high half.
D3P_D void normals8(const TfKey& km, uint32_t q0, uint32_t half, float4& lo, float4& hi) {
  uint32_t a0, b0, a1, b1, a2, b2, a3, b3;
  threefry2x32(km, q0 + 0u, q0 + 0u + half, a0, b0);
  threefry2x32(km, q0 + 1u, q0 + 1u + half, a1, b1);
  threefry2x32(km, q0 + 2u, q0 + 2u + half, a2, b2);
  threefry2x32(km, q0 + 3u, q0 + 3u + half, a3, b3);
  float4 ul = make_float4(unit_to_u(a0), unit_to_u(a1), unit_to_u(a2), unit_to_u(a3));
  float4 uh = make_float4(unit_to_u(b0), unit_to_u(b1), unit_to_u(b2), unit_to_u(b3));
  float4 wl, wh;
#define D3P_CENTRAL(c) lo.c = normal_central(ul.c, wl.c); hi.c = normal_central(uh.c, wh.c);
  D3P_F4_FOREACH(D3P_CENTRAL)
#undef D3P_CENTRAL
  const float wmin = fminf(fminf(fminf(wl.x, wl.y), fminf(wl.z, wl.w)), fminf(fminf(wh.x, wh.y), fminf(wh.z, wh.w)));
  if (__any_sync(0xffffffffu, wmin <= D3P_TAIL_L2)) {        // warp-uniform, ~58 % of the groups
#define D3P_TAIL1(v, u_, w_)                                                        \
    if (__any_sync(0xffffffffu, w_ <= D3P_TAIL_L2)) {      /* warp-uniform, ~10 % */  \
      const float tv = normal_tail(u_, w_);                                          \
      v = (w_ <= D3P_TAIL_L2) ? tv : v;                                              \
    }
#define D3P_TAIL(c) D3P_TAIL1(lo.c, ul.c, wl.c) D3P_TAIL1(hi.c, uh.c, wh.c)
    D3P_F4_FOREACH(D3P_TAIL)
#undef D3P_TAIL
#undef D3P_TAIL1
  }
}

D3P_D void cp_async16(float* smem_dst, const float* gsrc) {
  unsigned sa = (unsigned)__cvta_generic_to_shared(smem_dst);
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;\n" ::"r"(sa), "l"(gsrc));
}
D3P_D void st4(float* p, const float4& v) { *reinterpret_cast<float4*>(p) = v; }

// Per-warp staging in shared memory: the example's row x (later overwritten by g_loc) and the scaled
// noise u (later overwritten by g_rho).  Every lane only touches its own 16-byte slots, so no intra-warp synchronisation is
// needed; the loops over chunks stay rolled, which keeps the hot loop inside the instruction cache
// (the fully unrolled variant was fetch-bound: ncu `no_instruction` stalls, profiles/r1_*).
//
// LPE = lanes per example.  d = 2 * LPE * NQ: with LPE = 32 a warp works on one example at a time; with
// LPE = 8 / 16 it works on 4 / 2 examples at once (one per group of LPE lanes), every lane still owning
// NQ elements per half.  Short rows (d = 256) then amortise the per-example work that does not scale
// with d (key shuffles, reductions, loop control, the link scalars) over 4 examples: d = 256 ran 17 % more
// cycles per element than d = 1024 with one example per warp.
template <int FAMILY, int LINK, int NQ, int LPE>
__global__ void __launch_bounds__(kStepThreads, 2) meanfield_step_vec_kernel(StepArgs a) {
  static_assert(NQ % 4 == 0, "NQ must be a multiple of 4");
  static_assert(LPE == 8 || LPE == 16 || LPE == 32, "LPE must be 8, 16 or 32");
  constexpr int NCH = NQ / 4;          // float4 chunks per half per lane
  constexpr int HALF = LPE * NQ;       // d / 2
  constexpr int D = 2 * HALF;
  constexpr int G = 32 / LPE;          // examples in flight per warp
  constexpr int TILE = 16;
  constexpr bool kExp = LINK == D3P_LINK_EXP;
  extern __shared__ __align__(16) float smem[];
  float* s_loc = smem;
  float* s_scl = s_loc + D;
  float* s_a = s_scl + D;                       // softplus only
  float* s_sa = s_a + (kExp ? 0 : D);
  float* s_bt = s_sa + (kExp ? 0 : D);
  float* s_stage = s_bt + (kExp ? 0 : D);       // [kStepWarps][G][2 * D]
  __shared__ float s_red[kStepWarps];
  __shared__ float s_scal[kStepWarps][4];

  // let a programmatic dependent (the finalize kernel) be placed on the SMs as this grid drains; it waits for the
  // whole grid to complete before it reads the partial rows
  asm volatile("griddepcontrol.launch_dependents;");
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int sl = lane & (LPE - 1), sub = lane / LPE;       // lane within its example group, group index
  float* xs = s_stage + (warp * G + sub) * 2 * D;          // x, then gl
  float* us = xs + D;                                      // u = eps * s'

  float log_s_part = 0.f;
  for (int e = threadIdx.x; e < D; e += kStepThreads) {
    float s, aa, bt, ls;
    link_terms<LINK>(a.params[a.rho_off + e], a.inv_S, s, aa, bt, ls);
    s_loc[e] = a.params[a.loc_off + e];
    s_scl[e] = s;
    // s' underflows to 0 below rho ~ -88.7 while s stays a denormal: theta = loc there, as in the generic kernel
    if (!kExp) { s_a[e] = aa; s_sa[e] = (aa != 0.f) ? s / aa : 0.f; s_bt[e] = bt; }
    log_s_part += ls;
  }
  InterceptGuide b{0.f, 0.f, 0.f, 0.f};
  if (a.has_b) {
    float ls;
    b.loc = a.params[a.b_loc_off];
    link_terms<LINK>(a.params[a.b_rho_off], a.inv_S, b.s, b.a, b.bt, ls);
    if (threadIdx.x == 0) log_s_part += ls;
  }
  log_s_part = gsum<32>(log_s_part, 0xffffffffu);
  if (lane == 0) s_red[warp] = log_s_part;
  __syncthreads();
  float sum_log_s = 0.f;
#pragma unroll
  for (int w = 0; w < kStepWarps; ++w) sum_log_s += s_red[w];

  float4 accL[2 * NCH], accR[2 * NCH];
#pragma unroll
  for (int i = 0; i < 2 * NCH; ++i) { accL[i] = make_float4(0.f, 0.f, 0.f, 0.f); accR[i] = accL[i]; }
  float acc_bloc = 0.f, acc_brho = 0.f, acc_loss = 0.f, acc_cnt = 0.f;

  const TfKey K = tf_key_arg(a.k0, a.k1, a.key_d);
  const uint32_t npos = a.pos_end - a.pos_begin;
  const uint32_t nv = a.num_valid ? (uint32_t)max(*a.num_valid, 0) : 0xffffffffu;
  const uint32_t total_warps = gridDim.x * kStepWarps;
  const float Linv = a.L * a.inv_var;

  // Each warp owns one contiguous run of floor(npos / total_warps) (+1 for npos % total_warps of the
  // warps) positions and walks it in tiles of 16: per-warp loads differ by at most one example, which
  // matters when a rank holds only a few examples per warp (sharded batches: 5.3 at N = 8 on C2).
  const uint32_t gw = blockIdx.x * kStepWarps + warp;
  // the npos % total_warps longer runs are spread evenly over the grid (Bresenham), so that every SM holds the
  // same number of examples +-1 whichever CTAs it hosts (the first-come form gave 88 vs 80 per SM at N = 8)
  const uint32_t per_q = npos / total_warps, per_r = npos % total_warps;
  const uint32_t x_lo = (uint32_t)(((unsigned long long)gw * per_r) / total_warps);
  const uint32_t x_hi = (uint32_t)(((unsigned long long)(gw + 1u) * per_r) / total_warps);
  const uint32_t w_begin = gw * per_q + x_lo;
  const uint32_t w_end = a.pos_begin + w_begin + per_q + (x_hi - x_lo);
  for (uint32_t base = a.pos_begin + w_begin; base < w_end; base += TILE) {
    const uint32_t my_p = base + lane;
    bool my_valid = (lane < TILE) && (my_p < w_end) && (my_p < nv) && (!a.mask || a.mask[my_p]);
    uint32_t my_k0, my_k1, my_row = 0;
    float my_eb = 0.f, my_y = 0.f;
    {
      // Key chain of example base + (lane & 15); it must equal the guide_rng / next_site chain of common.cuh
      // that the generic kernel runs: split(K,B)[p] -> split -> guide_seed -> split -> (rng, k_main)
      // [-> split(rng) -> k_b -> eps_b].  Every level is two independent Threefry calls ((0,2) and (1,3)); the
      // lower / upper half-warp take one each and swap by shuffle, so the chain costs 3 (5 with an intercept)
      // calls per tile of 16 examples instead of 6 (9) per example.
      const uint32_t tl = lane & 15u, part = lane >> 4;
      const uint32_t w = tf_split_word(K, a.B, 2u * (base + tl) + part);
      TfKey kk(__shfl_sync(0xffffffffu, w, tl), __shfl_sync(0xffffffffu, w, tl + 16u));
      uint32_t y0, y1;
      threefry2x32(kk, part, part + 2u, y0, y1);                 // (model_seed, guide_seed)
      kk = TfKey(__shfl_sync(0xffffffffu, y1, tl), __shfl_sync(0xffffffffu, y1, tl + 16u));
      threefry2x32(kk, part, part + 2u, y0, y1);                 // (rng, k_main)
      my_k0 = __shfl_sync(0xffffffffu, y1, tl);
      my_k1 = __shfl_sync(0xffffffffu, y1, tl + 16u);
      if (a.has_b) {
        kk = TfKey(__shfl_sync(0xffffffffu, y0, tl), __shfl_sync(0xffffffffu, y0, tl + 16u));
        threefry2x32(kk, part, part + 2u, y0, y1);               // (rng2, k_b)
        kk = TfKey(__shfl_sync(0xffffffffu, y1, tl), __shfl_sync(0xffffffffu, y1, tl + 16u));
        threefry2x32(kk, 0u, 0u, y0, y1);
        my_eb = bits_to_normal_fast(y0);
      }
    }
    if (my_valid) {
      my_row = a.idx ? (uint32_t)a.idx[my_p] : my_p;
      if (FAMILY == D3P_FAMILY_LOGREG) my_y = (float)a.y[my_row];
    }
    const unsigned valid_bits = __ballot_sync(0xffffffffu, my_valid);
    const uint32_t any_row = __shfl_sync(0xffffffffu, my_row, __ffs(valid_bits | 0x10000u) - 1);   // a readable row
#pragma unroll 1
    for (int t0 = 0; t0 < TILE; t0 += G) {
      if (!((valid_bits >> t0) & ((1u << G) - 1u))) continue;   // warp-uniform: none of the G examples is valid
      const int t = t0 + sub;                                    // this lane group's example
      // a group whose example is masked out runs along on a readable row with weight 0 (it must take part
      // in the warp-wide votes of the tail fix-up); with LPE = 32 this never happens
      const bool act = (valid_bits >> t) & 1u;
      const TfKey km(__shfl_sync(0xffffffffu, my_k0, t), __shfl_sync(0xffffffffu, my_k1, t));
      const uint32_t row_t = __shfl_sync(0xffffffffu, my_row, t);
      const uint32_t row = act ? row_t : any_row;
      const float eb = __shfl_sync(0xffffffffu, my_eb, t);
      const float yv = __shfl_sync(0xffffffffu, my_y, t);
      const float* __restrict__ xr = a.x + (size_t)row * a.x_stride;

      // the row goes straight to this lane's staging slots (no register staging)
#pragma unroll
      for (int i = 0; i < 2 * NCH; ++i) {
        const int e0 = (i & 1) * HALF + 4 * (sl + LPE * (i >> 1));
        cp_async16(xs + e0, xr + e0);
      }
      asm volatile("cp.async.commit_group;\n" ::: "memory");

      // ---- loop A: noise + pass 1 ----------------------------------------------------------------
      float zdot = 0.f, s_th2 = 0.f, s_e2 = 0.f, s_res2 = 0.f, nrm = 0.f;
#pragma unroll 1
      for (int kk = 0; kk < NCH; ++kk) {
        const int q0 = 4 * (sl + LPE * kk);
        float4 ev[2];
        normals8(km, (uint32_t)q0, HALF, ev[0], ev[1]);
        if (kk == 0) asm volatile("cp.async.wait_group 0;\n" ::: "memory");
#pragma unroll
        for (int h = 0; h < 2; ++h) {
          const int e0 = h * HALF + q0;
          const float4 xv = ld4(xs + e0);
          const float4 loc = ld4(s_loc + e0), sc = ld4(s_scl + e0);
          float4 aa = sc, bt = sc;
          if (!kExp) { aa = ld4(s_a + e0); if (FAMILY == D3P_FAMILY_GAUSS) bt = ld4(s_bt + e0); }
          float4 u, gl;
          // Gaussian family: the gradient needs no reduction over the row (h = L (theta - x) / var element-wise), so
          // loop B is folded in here: g_loc goes over x, g_rho goes where logreg parks u
#define D3P_P1(c)                                                      \
          {                                                            \
            const float th = fmaf(ev[h].c, sc.c, loc.c);               \
            s_e2 = fmaf(ev[h].c, ev[h].c, s_e2);                       \
            s_th2 = fmaf(th, th, s_th2);                               \
            u.c = ev[h].c * aa.c;                                      \
            if (FAMILY == D3P_FAMILY_LOGREG) zdot = fmaf(xv.c, th, zdot); \
            else {                                                     \
              const float r = xv.c - th;                               \
              s_res2 = fmaf(r, r, s_res2);                             \
              gl.c = fmaf(th, a.inv_S, -(Linv * r));                   \
              u.c = fmaf(gl.c, u.c, -(kExp ? a.inv_S : bt.c));         \
              nrm = fmaf(gl.c, gl.c, fmaf(u.c, u.c, nrm));             \
            }                                                          \
          }
          D3P_F4_FOREACH(D3P_P1)
#undef D3P_P1
          st4(us + e0, u);
          if (FAMILY == D3P_FAMILY_GAUSS) st4(xs + e0, gl);
        }
      }
      if (FAMILY == D3P_FAMILY_LOGREG) zdot = gsum<LPE>(zdot, 0xffffffffu);
      else s_res2 = gsum<LPE>(s_res2, 0xffffffffu);
      s_th2 = gsum<LPE>(s_th2, 0xffffffffu);
      s_e2 = gsum<LPE>(s_e2, 0xffffffffu);

      float th_b, Lr;
      const float loss_i = example_loss<FAMILY>(a, b, eb, yv, FAMILY == D3P_FAMILY_LOGREG ? zdot : s_res2, s_th2, s_e2,
                                                sum_log_s, D, th_b, Lr);

      // ---- loop B (logreg: needs the logit first): gradients (g_loc overwrites x, g_rho overwrites u), norm ----
#pragma unroll 2
      for (int kk = 0; kk < (FAMILY == D3P_FAMILY_LOGREG ? NCH : 0); ++kk) {
#pragma unroll
        for (int h = 0; h < 2; ++h) {
          const int e0 = h * HALF + 4 * (sl + LPE * kk);
          const float4 loc = ld4(s_loc + e0), xv = ld4(xs + e0), u = ld4(us + e0);
          float4 sa = loc, bt = loc, gl, gs;
          if (!kExp) { sa = ld4(s_sa + e0); bt = ld4(s_bt + e0); }
#define D3P_P2(c)                                                                            \
          {                                                                                  \
            const float th = kExp ? (loc.c + u.c) : fmaf(u.c, sa.c, loc.c);                  \
            const float hh = (FAMILY == D3P_FAMILY_LOGREG) ? Lr * xv.c : Linv * (th - xv.c); \
            gl.c = fmaf(th, a.inv_S, hh);                                                    \
            gs.c = fmaf(gl.c, u.c, -(kExp ? a.inv_S : bt.c));                                \
            nrm = fmaf(gl.c, gl.c, fmaf(gs.c, gs.c, nrm));                                   \
          }
          D3P_F4_FOREACH(D3P_P2)
#undef D3P_P2
          st4(xs + e0, gl);
          st4(us + e0, gs);
        }
      }
      if (a.px_grads && act) {             // stage-method API only (tests): materialise this example's gradient row
        float* pg = a.px_grads + (size_t)(base + t) * a.P;
#pragma unroll 1
        for (int i = 0; i < 2 * NCH; ++i) {
          const int e0 = (i & 1) * HALF + 4 * (sl + LPE * (i >> 1));
          const float4 gl = ld4(xs + e0), gs = ld4(us + e0);
#define D3P_PG(c, k) pg[a.loc_off + e0 + k] = gl.c; pg[a.rho_off + e0 + k] = gs.c;
          D3P_PG(x, 0) D3P_PG(y, 1) D3P_PG(z, 2) D3P_PG(w, 3)
#undef D3P_PG
        }
      }
      float glb, gsb;
      nrm = intercept_grad(a, b, th_b, eb, Lr, gsum<LPE>(nrm, 0xffffffffu), glb, gsb);
      const float norm = sqrtf(nrm);
      const float c = act ? 1.0f / fmaxf(1.0f, norm / a.C) : 0.f;

      // ---- loop C: clipped accumulation (unrolled: the accumulators live in registers) ---------
#pragma unroll
      for (int i = 0; i < 2 * NCH; ++i) {
        const int e0 = (i & 1) * HALF + 4 * (sl + LPE * (i >> 1));
        const float4 gl = ld4(xs + e0), gs = ld4(us + e0);
#define D3P_P3(c_)                                                     \
        accL[i].c_ = fmaf(c, gl.c_, accL[i].c_);                       \
        accR[i].c_ = fmaf(c, gs.c_, accR[i].c_);
        D3P_F4_FOREACH(D3P_P3)
#undef D3P_P3
      }
      if (sl == 0 && act) {
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

  // ---- epilogue: lane groups fold into group 0 (fixed order), then warps add into the CTA partial -----------
  if (G > 1) {
#pragma unroll
    for (int o = LPE; o < 32; o <<= 1) {
#pragma unroll
      for (int i = 0; i < 2 * NCH; ++i) {
#define D3P_FOLD(c_)                                                   \
        accL[i].c_ += __shfl_xor_sync(0xffffffffu, accL[i].c_, o);     \
        accR[i].c_ += __shfl_xor_sync(0xffffffffu, accR[i].c_, o);
        D3P_F4_FOREACH(D3P_FOLD)
#undef D3P_FOLD
      }
      acc_bloc += __shfl_xor_sync(0xffffffffu, acc_bloc, o);
      acc_brho += __shfl_xor_sync(0xffffffffu, acc_brho, o);
      acc_loss += __shfl_xor_sync(0xffffffffu, acc_loss, o);
      acc_cnt += __shfl_xor_sync(0xffffffffu, acc_cnt, o);
    }
  }
  // every warp parks its sums in its own staging slot (it is done with it), then all threads add the 8 slots of
  // their columns in warp order (fixed order => run-to-run deterministic) and write the CTA partial
  float* slot = s_stage + (size_t)warp * G * 2 * D;
  if (sub == 0) {
#pragma unroll
    for (int i = 0; i < 2 * NCH; ++i) {
      const int e0 = (i & 1) * HALF + 4 * (sl + LPE * (i >> 1));
      st4(slot + e0, accL[i]);
      st4(slot + D + e0, accR[i]);
    }
  }
  if (lane == 0) {
    s_scal[warp][0] = acc_bloc; s_scal[warp][1] = acc_brho; s_scal[warp][2] = acc_loss; s_scal[warp][3] = acc_cnt;
  }
  __syncthreads();
  float* out = a.partials + (size_t)blockIdx.x * (a.P + 2);
  for (int j = threadIdx.x; j < 2 * D; j += kStepThreads) {
    float v = 0.f;
#pragma unroll
    for (int w = 0; w < kStepWarps; ++w) v += s_stage[(size_t)w * G * 2 * D + j];
    out[(j < D ? a.loc_off : a.rho_off - D) + j] = v;
  }
  if (threadIdx.x < 4) {
    float v = 0.f;
#pragma unroll
    for (int w = 0; w < kStepWarps; ++w) v += s_scal[w][threadIdx.x];
    if (threadIdx.x >= 2) out[a.P + threadIdx.x - 2] = v;
    else if (a.has_b) out[threadIdx.x == 0 ? a.b_loc_off : a.b_rho_off] = v;
  }
}

template <int FAMILY, int LINK, int NQ, int LPE>
static int32_t launch_vec_one(const StepArgs& a, unsigned grid, cudaStream_t s) {
  constexpr int D = 2 * LPE * NQ;
  constexpr int G = 32 / LPE;
  size_t smem = ((LINK == D3P_LINK_EXP ? 2 : 5) * (size_t)D + (size_t)kStepWarps * G * 2 * D) * sizeof(float);
  auto kern = meanfield_step_vec_kernel<FAMILY, LINK, NQ, LPE>;
  if (smem > 48 * 1024 &&
      cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess)
    return D3P_ERR_CUDA;
  kern<<<grid, kStepThreads, smem, s>>>(a);
  return check_launch();
}

template <int FAMILY, int LINK>
static int32_t launch_vec_nq(const StepArgs& a, unsigned grid, cudaStream_t s) {
  switch (a.d) {
    case 256: return launch_vec_one<FAMILY, LINK, 16, 8>(a, grid, s);     // 4 examples per warp
    case 512: return launch_vec_one<FAMILY, LINK, 16, 16>(a, grid, s);    // 2 examples per warp
    case 1024: return launch_vec_one<FAMILY, LINK, 16, 32>(a, grid, s);
    default: return D3P_ERR_UNSUPPORTED;
  }
}

// Eligibility: full shape (single main site of exactly d = 256/512/1024 elements) and 16-byte
// aligned rows.  Returns D3P_ERR_UNSUPPORTED when the generic kernel has to be used.
int32_t launch_meanfield_vec(int family, int link, const StepArgs& a, unsigned grid, cudaStream_t s) {
  if (a.n_main != a.d || (a.d != 256 && a.d != 512 && a.d != 1024)) return D3P_ERR_UNSUPPORTED;
  if ((reinterpret_cast<uintptr_t>(a.x) & 15) || (a.x_stride & 3)) return D3P_ERR_UNSUPPORTED;
  if (family == D3P_FAMILY_LOGREG) {
    if (link == D3P_LINK_EXP) return launch_vec_nq<D3P_FAMILY_LOGREG, D3P_LINK_EXP>(a, grid, s);
    return launch_vec_nq<D3P_FAMILY_LOGREG, D3P_LINK_SOFTPLUS>(a, grid, s);
  }
  if (link == D3P_LINK_EXP) return launch_vec_nq<D3P_FAMILY_GAUSS, D3P_LINK_EXP>(a, grid, s);
  return launch_vec_nq<D3P_FAMILY_GAUSS, D3P_LINK_SOFTPLUS>(a, grid, s);
}

}  // namespace d3p
