// K8: fixed-order reduction of the per-CTA partial sums + mean + ChaCha20 Gaussian perturbation
// + rescale + optimizer step, in one launch.  Replaces DPSVI._combine_gradients
// (d3p/svi.py:327-348), _perturb_and_reassemble_gradients (:350-377), perturbation_function
// (:470-498) and _apply_gradient (:379-393) with numpyro.optim.SGD / Adam / Momentum / Adagrad / RMSProp /
// RMSPropMomentum / ClippedAdam and d3p's ADADP.
#include "comm.cuh"
#include "common.cuh"
#include "launch.cuh"

namespace d3p {

struct LeafTable {
  uint32_t n_leaves;
  uint32_t off[D3P_MAX_LEAVES];
  uint32_t len[D3P_MAX_LEAVES];
};

struct FinalizeArgs {
  const float* partials;
  uint32_t n_partials, P, B;
  float dp_scale, C, obs_scale;
  int add_noise;
  float* grad_out;
  int opt_kind;        // D3P_OPT_* without D3P_OPT_SCHEDULED
  float step_size;     // lr of this step: the schedule is evaluated on the host, once per launch
  float b1, b2, eps;
  float mom, gamma, clip;   // MOMENTUM .. CLIPPED_ADAM (header)
  int step;
  float* params;
  float* m;
  float* v;
  float* stats;
  int use_override;
  float n_override, f_override;
  const float* lr;     // ADADP: device step size
  float* err_ws;       // ADADP odd steps: [0] = number of CTA partials, [1 + cta] = partial error sums
};

// d3p/optimizers.py:58-70 (even step) and :72-78,108 (odd step, before the accept/reject decision taken by
// adadp_finish_kernel).  m = x_stepped, v = x_prev.  Returns this element's squared error term (odd steps).
D3P_D float adadp_element(const FinalizeArgs& a, float lr, uint32_t j, float x, float g) {
  const float new_x = x - (0.5f * lr) * g;
  a.params[j] = new_x;
  if ((a.step & 1) == 0) {
    a.v[j] = x;
    a.m[j] = x - lr * g;
    return 0.f;
  }
  const float xs = a.m[j];
  const float e = __fdiv_rn(xs - new_x, fmaxf(1.0f, xs));
  return e * e;
}

// Which old state an optimizer kind reads (ADADP's is handled by adadp_element).
__host__ __device__ inline bool opt_uses_x(int k) { return k != D3P_OPT_NONE && k != D3P_OPT_ADADP; }
__host__ __device__ inline bool opt_uses_m(int k) {
  return k == D3P_OPT_ADAM || k == D3P_OPT_MOMENTUM || k == D3P_OPT_ADAGRAD || k == D3P_OPT_RMSPROP_MOMENTUM ||
         k == D3P_OPT_CLIPPED_ADAM;
}
__host__ __device__ inline bool opt_uses_v(int k) {
  return k == D3P_OPT_ADAM || k == D3P_OPT_ADAGRAD || k == D3P_OPT_RMSPROP || k == D3P_OPT_RMSPROP_MOMENTUM ||
         k == D3P_OPT_CLIPPED_ADAM;
}

// One element of the numpyro optimizers (jax.example_libraries.optimizers; header, D3P_OPT_*): x, m, v are the old
// state, loaded by the kernel's prologue; bc1 / bc2 are Adam's bias corrections of this step.  quad_adam: Adam's
// moments are rounded as finalize_quad_kernel has always rounded them, fma(g, 1 - b1, b1 * m) and
// fma(g * g, 1 - b2, b2 * v).  Everywhere else (finalize_kernel, and ClippedAdam in both kernels) the compiler
// contracts the plain expressions the other way round, fma(m, b1, (1 - b1) * g): the two differ in the last bit.
D3P_D void optim_element(const FinalizeArgs& a, float bc1, float bc2, uint32_t j, float g, float x, float m, float v,
                         float* __restrict__ prm, float* __restrict__ pm, float* __restrict__ pv, bool quad_adam) {
  const int k = a.opt_kind;                              // NONE and ADADP do nothing here
  if (k == D3P_OPT_SGD) {
    prm[j] = x - a.step_size * g;
  } else if (k == D3P_OPT_ADAM || k == D3P_OPT_CLIPPED_ADAM) {
    // jnp.clip (a NaN stays NaN); only the moments see the clipped value, grad_out got g already
    if (k == D3P_OPT_CLIPPED_ADAM) g = g < -a.clip ? -a.clip : (g > a.clip ? a.clip : g);
    if (quad_adam && k == D3P_OPT_ADAM) {
      m = __fmaf_rn(1.0f - a.b1, g, __fmul_rn(a.b1, m));
      v = __fmaf_rn(1.0f - a.b2, __fmul_rn(g, g), __fmul_rn(a.b2, v));
    } else {
      m = (1.0f - a.b1) * g + a.b1 * m;
      v = (1.0f - a.b2) * (g * g) + a.b2 * v;
    }
    float mhat = m / bc1;
    float vhat = v / bc2;
    prm[j] = x - a.step_size * mhat / (sqrtf(vhat) + a.eps);
    pm[j] = m;
    pv[j] = v;
  } else if (k == D3P_OPT_MOMENTUM) {
    m = a.mom * m + g;
    prm[j] = x - a.step_size * m;
    pm[j] = m;
  } else if (k == D3P_OPT_ADAGRAD) {
    v = v + g * g;
    const float r = v > 0.f ? 1.0f / sqrtf(v) : 0.f;     // an element that never had a gradient: 0, not 0 * inf
    m = (1.0f - a.mom) * (g * r) + a.mom * m;
    prm[j] = x - a.step_size * m;
    pm[j] = m;
    pv[j] = v;
  } else if (k == D3P_OPT_RMSPROP) {
    v = v * a.gamma + (g * g) * (1.0f - a.gamma);
    prm[j] = x - a.step_size * g / sqrtf(v + a.eps);     // eps inside the root
    pv[j] = v;
  } else if (k == D3P_OPT_RMSPROP_MOMENTUM) {
    v = v * a.gamma + (g * g) * (1.0f - a.gamma);
    m = a.mom * m + a.step_size * g / sqrtf(v + a.eps);
    prm[j] = x - m;
    pm[j] = m;
    pv[j] = v;
  }
}

// Adam's bias corrections of this step (bc1 / bc2 are left alone for the other kinds).
D3P_D void adam_bias(const FinalizeArgs& a, float& bc1, float& bc2) {
  if (a.opt_kind == D3P_OPT_ADAM || a.opt_kind == D3P_OPT_CLIPPED_ADAM) {
    const float t = (float)(a.step + 1);
    bc1 = 1.0f - powf(a.b1, t); bc2 = 1.0f - powf(a.b2, t);
  }
}

// Fixed-order CTA sum of the partial rows' (count, loss) columns: rows strided over the NT threads, a shuffle tree per
// warp, then thread 0 adds the warp sums in warp order into s_n / s_loss.  The caller synchronizes before reading them.
template <int NT>
D3P_D void reduce_count_loss(const FinalizeArgs& a, float (&red)[2][NT / 32], float& s_n, float& s_loss) {
  const uint32_t stride = a.P + 2;
  float cnt = 0.f, loss = 0.f;
  for (uint32_t p = threadIdx.x; p < a.n_partials; p += NT) {
    loss += a.partials[(size_t)p * stride + a.P];
    cnt += a.partials[(size_t)p * stride + a.P + 1];
  }
  cnt = group_sum<32>(cnt);
  loss = group_sum<32>(loss);
  if ((threadIdx.x & 31) == 0) { red[0][threadIdx.x >> 5] = cnt; red[1][threadIdx.x >> 5] = loss; }
  __syncthreads();
  if (threadIdx.x == 0) {
    float c = 0.f, l = 0.f;
#pragma unroll
    for (int w = 0; w < NT / 32; ++w) { c += red[0][w]; l += red[1][w]; }
    s_n = c; s_loss = l;
  }
}

// One-shot all-reduce of the CTA's (n, loss) over NVLink peer memory (comm.cuh): thread 0 pushes them as tagged words
// jn, jn + 1 to every peer, every thread polls its own window for the peers' copies and adds all copies in rank order
// (identical on every rank).  Returns the start value of the caller's per-column sums: 0, or NaN when an earlier
// time-out on this rank (sampler counts, a previous exchange) has poisoned everything from here on.  The caller pushes
// its columns first and adds them in rank order after this.
D3P_D float exchange_n_loss(const CommDev& comm, float& n, float& loss) {
  const float my_n = n, my_loss = loss;
  const size_t jn = comm.extra_off + 2 * (size_t)blockIdx.x;
  if (threadIdx.x == 0) { ll_push(comm, jn, my_n); ll_push(comm, jn + 1, my_loss); }
  const float zero = comm_poisoned(comm) ? __uint_as_float(0x7fc00000u) : 0.f;
  n = 0.f; loss = zero;
  for (int r = 0; r < comm.world; ++r) {
    const bool me = r == comm.rank;
    n += me ? my_n : ll_wait(comm, r, jn);
    loss += me ? my_loss : ll_wait(comm, r, jn + 1);
  }
  return zero;
}

constexpr int kFinThreads = 512;   // 16 warps share the partial rows of a 32-column strip: the row loop is latency-bound

// Fixed-order sum of column j over n_rows rows (kFinThreads threads, 32 columns per CTA): warp w adds rows w, w + 16,
// ... in row order, four loads in flight, and warp 0 adds the 16 warp sums in warp order.  The result is warp 0's.
D3P_D float column_sum(const float* __restrict__ rows, uint32_t n_rows, size_t stride, uint32_t j, bool live) {
  constexpr uint32_t W = kFinThreads / 32;
  __shared__ float colred[W][32];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  float part = 0.f;
  if (live) {
    uint32_t p = warp;
    for (; p + 3 * W < n_rows; p += 4 * W) {
      float v0 = rows[p * stride + j];
      float v1 = rows[(p + W) * stride + j];
      float v2 = rows[(p + 2 * W) * stride + j];
      float v3 = rows[(p + 3 * W) * stride + j];
      part += v0; part += v1; part += v2; part += v3;
    }
    for (; p < n_rows; p += W) part += rows[p * stride + j];
  }
  colred[warp][lane] = part;
  __syncthreads();
  float sum = 0.f;
  if (warp == 0)
#pragma unroll
    for (int w = 0; w < (int)W; ++w) sum += colred[w][lane];
  return sum;
}

// The release scale of this step from the all-reduced (n, loss), and the loss / n / f statistics (thread 0 of CTA 0).
struct Release { float Bf, f, sigma; };
D3P_D Release release_scale(const FinalizeArgs& a, float n_all, float loss_all) {
  const float n = a.use_override ? a.n_override : n_all;
  const float Bf = (float)a.B;
  const float f = a.use_override ? a.f_override : ((n == 0.f) ? 0.f : __fdiv_rn(Bf, n));   // svi.py:305
  const float sigma = __fmul_rn(a.dp_scale, __fdiv_rn(a.C, n));        // svi.py:365-366 (inf when n == 0)
  if (blockIdx.x == 0 && threadIdx.x == 0 && a.stats) {
    a.stats[0] = __fmul_rn(__fdiv_rn(loss_all, Bf), f);                // svi.py:306,342
    a.stats[1] = n;
    a.stats[2] = f;
  }
  return {Bf, f, sigma};
}

// One released element: sum = its column sum over all ranks, xi = its Gaussian draw when `noisy`.
D3P_D float release_element(const FinalizeArgs& a, const Release& r, uint32_t j, float sum, bool noisy, float xi) {
  float g = __fdiv_rn(sum, r.Bf);                                      // mean over the padded batch size
  if (noisy) g = __fadd_rn(g, __fmul_rn(xi, r.sigma));                // svi.py:485-486
  g = __fmul_rn(__fmul_rn(g, a.obs_scale), r.f);                       // svi.py:374-375
  if (a.grad_out) a.grad_out[j] = g;
  return g;
}

// The optimizer update of element j from its released gradient g and old state x, m, v; ADADP adds its squared error
// term to err2.
D3P_D void update_element(const FinalizeArgs& a, float bc1, float bc2, float lr, uint32_t j, float g, float x, float m,
                          float v, float& err2, bool quad_adam) {
  optim_element(a, bc1, bc2, j, g, x, m, v, a.params, a.m, a.v, quad_adam);
  if (a.opt_kind == D3P_OPT_ADADP) err2 += adadp_element(a, lr, j, x, g);
}

// A CTA's sum of the ADADP error terms (odd steps), for adadp_finish_kernel.
D3P_D void store_err_partial(const FinalizeArgs& a, float e) {
  a.err_ws[1 + blockIdx.x] = e;
  if (blockIdx.x == 0) a.err_ws[0] = (float)gridDim.x;
}

// site states live in constant-bank kernel parameters next to the leaf table
struct SiteStates { uint32_t w[D3P_MAX_LEAVES][16]; };

// `sites_d` (the *_dk entry point): the per-leaf ChaCha states live in device memory ([n_leaves][16] words, written by
// d3p_dpsvi_keys_dk) instead of the kernel parameters.
__global__ void __launch_bounds__(kFinThreads) finalize_kernel(const __grid_constant__ FinalizeArgs a,
                                                               const __grid_constant__ LeafTable leaves,
                                                               const __grid_constant__ SiteStates sites,
                                                               const uint32_t* __restrict__ sites_d,
                                                               const __grid_constant__ CommDev comm) {
  __shared__ float red[2][kFinThreads / 32];
  __shared__ float s_n, s_loss;
  // Launched as a programmatic dependent of the step kernel, this CTA is resident while that kernel is still running.
  // Everything that does not depend on its partial rows happens NOW, under the producer's tail instead of behind it:
  // the column's Gaussian draw (a ChaCha block: keys only), the Adam bias corrections and the loads of the parameter
  // and the optimizer state its kind keeps (written by the previous finalize, which completed before the step kernel
  // started).
  float xi_pre = 0.f, x_pre = 0.f, m_pre = 0.f, v_pre = 0.f, bc1 = 1.f, bc2 = 1.f;
  bool have_xi = false;
  {
    const uint32_t jp = blockIdx.x * 32 + (threadIdx.x & 31);
    if ((threadIdx.x >> 5) == 0 && jp < a.P) {
      if (a.add_noise) {
        int leaf = -1;
#pragma unroll 1
        for (uint32_t l = 0; l < leaves.n_leaves; ++l)
          if (jp >= leaves.off[l] && jp < leaves.off[l] + leaves.len[l]) leaf = (int)l;
        if (leaf >= 0) {
          uint32_t e = jp - leaves.off[leaf];
          uint32_t ks[16], st[16];
#pragma unroll
          for (int i = 0; i < 16; ++i) st[i] = sites_d ? __ldg(sites_d + 16 * leaf + i) : sites.w[leaf][i];
          chacha20_block(st, st[12] + (e >> 4), ks);
          uint32_t bits = ks[0];
#pragma unroll
          for (int i = 1; i < 16; ++i) bits = ((e & 15u) == (uint32_t)i) ? ks[i] : bits;
          xi_pre = bits_to_normal<false>(bits);
          have_xi = true;
        }
      }
      if (opt_uses_x(a.opt_kind)) x_pre = a.params[jp];
      if (opt_uses_m(a.opt_kind)) m_pre = a.m[jp];
      if (opt_uses_v(a.opt_kind)) v_pre = a.v[jp];
      adam_bias(a, bc1, bc2);
    }
  }
  asm volatile("griddepcontrol.wait;" ::: "memory");    // no-op unless launched as a programmatic dependent
  // every CTA reduces the (count, loss) columns itself: n_partials is a few hundred at most
  reduce_count_loss<kFinThreads>(a, red, s_n, s_loss);
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const uint32_t j = blockIdx.x * 32 + lane;
  const bool live = j < a.P;
  float sum = column_sum(a.partials, a.n_partials, a.P + 2, j, live);   // its barrier also publishes s_n / s_loss
  if (warp != 0) return;
  float n_all = s_n, loss_all = s_loss;
  if (comm.world > 1) {
    const float mine = sum;
    if (live) ll_push(comm, j, mine);
    sum = exchange_n_loss(comm, n_all, loss_all);
    for (int r = 0; r < comm.world; ++r)
      if (live) sum += r == comm.rank ? mine : ll_wait(comm, r, j);
  }
  const Release rel = release_scale(a, n_all, loss_all);
  float err2 = 0.f;
  if (live) {
    const bool adadp = a.opt_kind == D3P_OPT_ADADP;     // ADADP reads its parameter here, after griddepcontrol.wait
    update_element(a, bc1, bc2, adadp ? *a.lr : 0.f, j, release_element(a, rel, j, sum, have_xi, xi_pre),
                   adadp ? a.params[j] : x_pre, m_pre, v_pre, err2, false);
  }
  if (a.opt_kind == D3P_OPT_ADADP && (a.step & 1)) {
    err2 = group_sum<32>(err2);
    if (lane == 0) store_err_partial(a, err2);
  }
}

// Large-P variant (VAE: P = 652 824, few partial rows).  finalize_kernel recomputes a whole ChaCha block
// (~1000 instructions) for each of its 16 elements: fine at P ~ 2 k, 90 us at P ~ 650 k.  Here FOUR lanes
// cooperate on one block, each holding one column of the 4 x 4 state (column round = local quarter round,
// diagonal round = rotate rows 1-3 across the 4 lanes with shuffles), and then finalize the 4 elements whose
// keystream words they hold with finalize_kernel's release_element; partial rows are summed in row order.
struct ChunkTable { uint32_t n_chunks; uint32_t chunk_start[D3P_MAX_LEAVES + 1]; };   // chunk = one 16-element block

D3P_D void quad_qr(uint32_t& a, uint32_t& b, uint32_t& c, uint32_t& d) { D3P_QR(a, b, c, d) }

// (the tables are __grid_constant__: indexing a by-value kernel parameter with a run-time leaf number otherwise makes
// every thread copy it to local memory first)
__global__ void __launch_bounds__(256) finalize_quad_kernel(const __grid_constant__ FinalizeArgs a,
                                                            const __grid_constant__ LeafTable leaves,
                                                            const __grid_constant__ SiteStates sites,
                                                            const uint32_t* __restrict__ sites_d,
                                                            const __grid_constant__ ChunkTable ct,
                                                            const __grid_constant__ CommDev comm) {
  __shared__ float red[2][8];
  __shared__ float s_n, s_loss;
  const uint32_t stride = a.P + 2;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  reduce_count_loss<256>(a, red, s_n, s_loss);
  __syncthreads();
  const uint32_t t = blockIdx.x * 256 + threadIdx.x;
  const uint32_t chunk = t >> 2, q = t & 3;
  const bool live = chunk < ct.n_chunks;                  // uniform per 4-lane group; shuffles stay full-warp
  uint32_t leaf = 0;
#pragma unroll 1
  for (uint32_t l = 1; l < leaves.n_leaves; ++l)
    if (live && chunk >= ct.chunk_start[l]) leaf = l;
  const uint32_t b = live ? chunk - ct.chunk_start[leaf] : 0u;
  const bool adadp_odd = a.opt_kind == D3P_OPT_ADADP && (a.step & 1);
  const uint32_t len = leaves.len[leaf], off = leaves.off[leaf];
  const float* __restrict__ parts = a.partials;
  float* __restrict__ prm = a.params;
  float* __restrict__ pm = a.m;
  float* __restrict__ pv = a.v;
  const float lr_adadp = (a.opt_kind == D3P_OPT_ADADP) ? *a.lr : 0.f;
  float sum[4], x[4], m0[4], v0[4];
  uint32_t jj[4];
  bool ok[4];
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const uint32_t e = b * 16 + 4 * i + q;
    ok[i] = live && e < len;
    jj[i] = off + (ok[i] ? e : 0u);
    sum[i] = 0.f;
    x[i] = (ok[i] && a.opt_kind != D3P_OPT_NONE) ? prm[jj[i]] : 0.f;
    m0[i] = (ok[i] && opt_uses_m(a.opt_kind)) ? pm[jj[i]] : 0.f;
    v0[i] = (ok[i] && opt_uses_v(a.opt_kind)) ? pv[jj[i]] : 0.f;
  }
  // The partial rows are requested before the ChaCha rounds below.  Up to 4 rows (the VAE's concurrent wave writes 4)
  // are only LOADED here and added after the rounds, so that the 200 dependent instructions of the rounds run under
  // the loads' latency instead of behind it; more rows are added 5 at a time (20 independent loads per thread).
  const bool few = a.n_partials <= 4;
  float pre[4][4];
#pragma unroll
  for (int p = 0; p < 4; ++p)
#pragma unroll
    for (int i = 0; i < 4; ++i)
      pre[p][i] = (few && (uint32_t)p < a.n_partials && ok[i]) ? __ldg(parts + (size_t)p * stride + jj[i]) : 0.f;
  if (!few) {
#pragma unroll 5
    for (uint32_t p = 0; p < a.n_partials; ++p) {
#pragma unroll
      for (int i = 0; i < 4; ++i) sum[i] += ok[i] ? __ldg(parts + (size_t)p * stride + jj[i]) : 0.f;
    }
  }
  // column q of the state: rows 0..3
  const uint32_t* sw = sites_d ? sites_d + 16 * leaf : sites.w[leaf];
  const uint32_t i0 = sw[q], i1 = sw[4 + q], i2 = sw[8 + q];
  const uint32_t i3 = (q == 0) ? sw[12] + b : sw[12 + q];
  uint32_t x0 = i0, x1 = i1, x2 = i2, x3 = i3;
  const int base = lane & ~3;
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    quad_qr(x0, x1, x2, x3);                              // column round
    x1 = __shfl_sync(0xffffffffu, x1, base + ((q + 1) & 3));
    x2 = __shfl_sync(0xffffffffu, x2, base + ((q + 2) & 3));
    x3 = __shfl_sync(0xffffffffu, x3, base + ((q + 3) & 3));
    quad_qr(x0, x1, x2, x3);                              // diagonal round
    x1 = __shfl_sync(0xffffffffu, x1, base + ((q + 3) & 3));
    x2 = __shfl_sync(0xffffffffu, x2, base + ((q + 2) & 3));
    x3 = __shfl_sync(0xffffffffu, x3, base + ((q + 1) & 3));
  }
  const uint32_t ks[4] = {x0 + i0, x1 + i1, x2 + i2, x3 + i3};   // keystream words q, 4 + q, 8 + q, 12 + q
#pragma unroll
  for (int p = 0; p < 4; ++p)                                    // rows in row order, as the loop above adds them
#pragma unroll
    for (int i = 0; i < 4; ++i) sum[i] += pre[p][i];
  float n_all = s_n, loss_all = s_loss;
  if (comm.world > 1) {
    float mine[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) { mine[i] = sum[i]; if (ok[i]) ll_push(comm, jj[i], mine[i]); }
    const float zero = exchange_n_loss(comm, n_all, loss_all);
#pragma unroll
    for (int i = 0; i < 4; ++i) sum[i] = zero;
    for (int r = 0; r < comm.world; ++r)
#pragma unroll
      for (int i = 0; i < 4; ++i) if (ok[i]) sum[i] += r == comm.rank ? mine[i] : ll_wait(comm, r, jj[i]);
  }
  const Release rel = release_scale(a, n_all, loss_all);
  float bc1 = 1.f, bc2 = 1.f;
  adam_bias(a, bc1, bc2);
  float err2 = 0.f;
#pragma unroll
  for (int i = 0; i < 4; ++i)
    if (ok[i])
      update_element(a, bc1, bc2, lr_adadp, jj[i],
                     release_element(a, rel, jj[i], sum[i], true, bits_to_normal<false>(ks[i])), x[i], m0[i], v0[i],
                     err2, true);
  if (adadp_odd) {                                              // fixed-order CTA sum of the error terms
    err2 = group_sum<32>(err2);
    if (lane == 0) red[0][warp] = err2;
    __syncthreads();
    if (threadIdx.x == 0) {
      float e = 0.f;
#pragma unroll
      for (int w = 0; w < 8; ++w) e += red[0][w];
      store_err_partial(a, e);
    }
  }
}

// ADADP odd step, second half (d3p/optimizers.py:80-99): every CTA adds the error partials in the same
// order, so all of them take the same accept/reject decision; CTA 0 also updates the step size.
__global__ void __launch_bounds__(256) adadp_finish_kernel(const float* __restrict__ err_ws, float* lr, float tol,
                                                           int stability_check, float* __restrict__ params,
                                                           const float* __restrict__ x_prev, uint32_t P) {
  __shared__ float red[8];
  __shared__ float s_err;
  const uint32_t n = (uint32_t)err_ws[0];
  float part = 0.f;
  for (uint32_t p = threadIdx.x; p < n; p += 256) part += err_ws[1 + p];
  part = group_sum<32>(part);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = part;
  __syncthreads();
  if (threadIdx.x == 0) {
    float e = 0.f;
#pragma unroll
    for (int w = 0; w < 8; ++w) e += red[w];
    s_err = sqrtf(e);
  }
  __syncthreads();
  const float err = s_err;
  if (blockIdx.x == 0 && threadIdx.x == 0)
    *lr = *lr * fminf(fmaxf(sqrtf(__fdiv_rn(tol, err)), 0.9f), 1.1f);
  if (!(stability_check && err > tol)) return;
  for (uint32_t j = blockIdx.x * 256 + threadIdx.x; j < P; j += gridDim.x * 256) params[j] = x_prev[j];
}

// out[j] = sum_p partials[p][j] for j < row_len, in finalize_kernel's order.
__global__ void __launch_bounds__(kFinThreads) reduce_partials_kernel(const float* __restrict__ partials,
                                                                      uint32_t n_partials, uint32_t row_len,
                                                                      float* __restrict__ out) {
  const uint32_t j = blockIdx.x * 32 + (threadIdx.x & 31);
  const float sum = column_sum(partials, n_partials, row_len, j, j < row_len);
  if ((threadIdx.x >> 5) == 0 && j < row_len) out[j] = sum;
}

}  // namespace d3p

using namespace d3p;

extern "C" int32_t d3p_reduce_partials_f32(const float* partials_d, uint32_t n_partials, uint32_t P, float* out_d,
                                           void* stream) {
  if (!partials_d || !out_d || n_partials == 0) return D3P_ERR_INVALID_ARGUMENT;
  uint32_t row_len = P + 2;
  reduce_partials_kernel<<<(row_len + 31) / 32, kFinThreads, 0, (cudaStream_t)stream>>>(partials_d, n_partials, row_len,
                                                                                        out_d);
  return check_launch();
}

// jax.example_libraries.optimizers' schedules (constant, exponential_decay, inverse_time_decay, polynomial_decay,
// piecewise_constant), restated in float32.
extern "C" int32_t d3p_optim_step_size(const d3p_optim_desc* o, int32_t step, float* out_h) {
  if (!o || !out_h) return D3P_ERR_INVALID_ARGUMENT;
  const int32_t kind = o->kind & ~D3P_OPT_SCHEDULED;
  if (kind < D3P_OPT_NONE || kind > D3P_OPT_CLIPPED_ADAM) return D3P_ERR_UNSUPPORTED;
  if (kind == D3P_OPT_CLIPPED_ADAM && !(o->clip_norm > 0.f)) return D3P_ERR_INVALID_ARGUMENT;
  if (!(o->kind & D3P_OPT_SCHEDULED)) { *out_h = o->step_size; return D3P_OK; }
  if (kind == D3P_OPT_NONE || kind == D3P_OPT_ADADP || step < 0) return D3P_ERR_INVALID_ARGUMENT;
  const float s = o->step_size, i = (float)step, ds = o->decay_steps;
  switch (o->schedule) {
    case D3P_SCHED_CONSTANT:
      *out_h = s;
      return D3P_OK;
    case D3P_SCHED_EXPONENTIAL:
    case D3P_SCHED_INVERSE_TIME:
    case D3P_SCHED_POLYNOMIAL:
      if (!(ds > 0.f)) return D3P_ERR_INVALID_ARGUMENT;
      break;
    case D3P_SCHED_PIECEWISE:
      if (o->n_boundaries > D3P_MAX_BOUNDARIES) return D3P_ERR_INVALID_ARGUMENT;
      break;
    default:
      return D3P_ERR_UNSUPPORTED;
  }
  if (o->schedule == D3P_SCHED_EXPONENTIAL) {
    *out_h = s * powf(o->decay_rate, i / ds);
  } else if (o->schedule == D3P_SCHED_INVERSE_TIME) {
    *out_h = o->staircase ? s / (1.f + o->decay_rate * floorf(i / ds)) : s / (1.f + o->decay_rate * i / ds);
  } else if (o->schedule == D3P_SCHED_POLYNOMIAL) {
    const float n = fminf(i, ds);
    const float mult = powf(1.f - n / ds, o->power);
    *out_h = mult * (s - o->final_step_size) + o->final_step_size;
  } else {
    uint32_t k = 0;
    for (uint32_t b = 0; b < o->n_boundaries; ++b) k += i > o->boundaries[b] ? 1u : 0u;
    *out_h = o->values[k];
  }
  return D3P_OK;
}

int32_t d3p::optim_check(const d3p_optim_desc* o, const float* params_d, const float* m_d, const float* v_d) {
  if (!o) return D3P_OK;
  const int32_t kind = o->kind & ~D3P_OPT_SCHEDULED;
  if (kind != D3P_OPT_NONE && !params_d) return D3P_ERR_INVALID_ARGUMENT;
  if ((opt_uses_m(kind) && !m_d) || (opt_uses_v(kind) && !v_d)) return D3P_ERR_INVALID_ARGUMENT;
  if (kind == D3P_OPT_ADADP && (!m_d || !v_d || !o->lr_d || !o->err_ws_d || o->step < 0))
    return D3P_ERR_INVALID_ARGUMENT;
  float lr;
  return d3p_optim_step_size(o, o->step, &lr);
}

extern "C" int32_t d3p_perturb_finalize_f32(const float* partials_d, uint32_t n_partials, uint32_t P, uint32_t B,
                                            const d3p_leaf_table* leaves_h, float dp_scale, float C, float obs_scale,
                                            int32_t add_noise, float* grad_out_d, const d3p_optim_desc* optim_h,
                                            float* params_d, float* m_d, float* v_d, float* stats_d,
                                            const float* nf_override_h, void* stream) {
  return d3p_perturb_finalize_p2p_f32(partials_d, n_partials, P, B, leaves_h, dp_scale, C, obs_scale, add_noise,
                                      grad_out_d, optim_h, params_d, m_d, v_d, stats_d, nf_override_h, nullptr, stream);
}

int32_t d3p::perturb_finalize_impl(const float* partials_d, uint32_t n_partials, uint32_t P, uint32_t B,
                                   const d3p_leaf_table* leaves_h, const uint32_t* site_states_d, float dp_scale, float C,
                                   float obs_scale, int32_t add_noise, float* grad_out_d,
                                   const d3p_optim_desc* optim_h, float* params_d, float* m_d,
                                   float* v_d, float* stats_d, const float* nf_override_h,
                                   d3p_comm* comm, void* stream) {
  if (!partials_d || n_partials == 0 || B == 0) return D3P_ERR_INVALID_ARGUMENT;
  if (add_noise && !leaves_h) return D3P_ERR_INVALID_ARGUMENT;
  if (leaves_h && leaves_h->n_leaves > D3P_MAX_LEAVES) return D3P_ERR_UNSUPPORTED;
  FinalizeArgs a;
  a.partials = partials_d; a.n_partials = n_partials; a.P = P; a.B = B;
  a.dp_scale = dp_scale; a.C = C; a.obs_scale = obs_scale; a.add_noise = add_noise;
  a.grad_out = grad_out_d;
  if (const int32_t rc = optim_check(optim_h, params_d, m_d, v_d); rc != D3P_OK) return rc;
  a.opt_kind = optim_h ? optim_h->kind & ~D3P_OPT_SCHEDULED : D3P_OPT_NONE;
  a.step_size = 0.f;
  if (optim_h) d3p_optim_step_size(optim_h, optim_h->step, &a.step_size);   // validated by optim_check
  a.b1 = optim_h ? optim_h->b1 : 0.f; a.b2 = optim_h ? optim_h->b2 : 0.f; a.eps = optim_h ? optim_h->eps : 0.f;
  const bool appended = a.opt_kind >= D3P_OPT_MOMENTUM;     // fields past err_ws_d exist only for the new kinds
  a.mom = appended ? optim_h->momentum : 0.f;
  a.gamma = appended ? optim_h->gamma : 0.f;
  a.clip = appended ? optim_h->clip_norm : 0.f;
  a.step = optim_h ? optim_h->step : 0;
  a.params = params_d; a.m = m_d; a.v = v_d; a.stats = stats_d;
  a.use_override = nf_override_h ? 1 : 0;
  a.n_override = nf_override_h ? nf_override_h[0] : 0.f;
  a.f_override = nf_override_h ? nf_override_h[1] : 0.f;
  a.lr = nullptr; a.err_ws = nullptr;
  if (a.opt_kind == D3P_OPT_ADADP) { a.lr = optim_h->lr_d; a.err_ws = optim_h->err_ws_d; }
  LeafTable lt;
  SiteStates ss;
  CommDev cd;
  memset(&cd, 0, sizeof(cd));
  cd.world = 1;
  memset(&lt, 0, sizeof(lt));
  memset(&ss, 0, sizeof(ss));
  if (leaves_h) {
    lt.n_leaves = leaves_h->n_leaves;
    for (uint32_t l = 0; l < lt.n_leaves; ++l) {
      lt.off[l] = leaves_h->leaf_off[l];
      lt.len[l] = leaves_h->leaf_len[l];
      if ((uint64_t)lt.off[l] + lt.len[l] > P) return D3P_ERR_INVALID_ARGUMENT;
      for (int i = 0; i < 16; ++i) ss.w[l][i] = leaves_h->site_state[l][i];
    }
  }
  if (add_noise) {
    // every coordinate must get its noise: the leaves have to tile [0, P) exactly (disjoint, no gap).  A table that
    // leaves a coordinate uncovered would release that clipped sum un-noised (round-1 ADVICE)
    uint64_t covered = 0;
    for (uint32_t l = 0; l < lt.n_leaves; ++l) {
      covered += lt.len[l];
      for (uint32_t k = 0; k < l; ++k)
        if (lt.off[l] < lt.off[k] + lt.len[k] && lt.off[k] < lt.off[l] + lt.len[l] && lt.len[l] && lt.len[k])
          return D3P_ERR_INVALID_ARGUMENT;
    }
    if (covered != P) return D3P_ERR_INVALID_ARGUMENT;
  }
  // large parameter vectors (with noise, so the leaf table tiles [0, P) as checked above): four threads per keystream
  // block
  if (add_noise && P >= 32768 && n_partials <= 64) {
    ChunkTable ct;
    memset(&ct, 0, sizeof(ct));
    uint32_t nc = 0;
    for (uint32_t l = 0; l < lt.n_leaves; ++l) {
      ct.chunk_start[l] = nc;
      nc += (lt.len[l] + 15) / 16;
    }
    ct.chunk_start[lt.n_leaves] = nc;
    ct.n_chunks = nc;
    const unsigned qgrid = (nc * 4 + 255) / 256;
    if (comm) { const int32_t rc = comm_next(comm, P, qgrid, &cd); if (rc != D3P_OK) return rc; }
    finalize_quad_kernel<<<qgrid, 256, 0, (cudaStream_t)stream>>>(a, lt, ss, site_states_d, ct, cd);
    return check_launch();
  }
  unsigned grid = P ? (P + 31) / 32 : 1;
  if (comm) { const int32_t rc = comm_next(comm, P, grid, &cd); if (rc != D3P_OK) return rc; }
  // Programmatic dependent launch: when the preceding kernel on the stream releases its dependents early (the
  // fused step kernels do, at their first instruction), the CTAs of this latency-bound kernel are placed on SMs as
  // those drain and wait in griddepcontrol.wait for the producer grid to complete and flush, which takes the
  // launch latency off the step's critical path.  After any other predecessor this is an ordinary launch.
  cudaLaunchConfig_t cfg;
  memset(&cfg, 0, sizeof(cfg));
  cfg.gridDim = dim3(grid); cfg.blockDim = dim3(kFinThreads); cfg.dynamicSmemBytes = 0; cfg.stream = (cudaStream_t)stream;
  cudaLaunchAttribute attr;
  attr.id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr.val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = &attr; cfg.numAttrs = 1;
  if (cudaLaunchKernelEx(&cfg, finalize_kernel, a, lt, ss, site_states_d, cd) != cudaSuccess) return D3P_ERR_CUDA;
  return check_launch();
}

extern "C" int32_t d3p_perturb_finalize_p2p_f32(const float* partials_d, uint32_t n_partials, uint32_t P, uint32_t B,
                                                const d3p_leaf_table* leaves_h, float dp_scale, float C,
                                                float obs_scale, int32_t add_noise, float* grad_out_d,
                                                const d3p_optim_desc* optim_h, float* params_d, float* m_d,
                                                float* v_d, float* stats_d, const float* nf_override_h,
                                                d3p_comm* comm, void* stream) {
  return perturb_finalize_impl(partials_d, n_partials, P, B, leaves_h, nullptr, dp_scale, C, obs_scale, add_noise,
                               grad_out_d, optim_h, params_d, m_d, v_d, stats_d, nf_override_h, comm, stream);
}

// Device-key form: leaves_h carries the leaf layout only (its site_state words are ignored); the per-leaf ChaCha states
// are read from site_states_d ([n_leaves][16] words, e.g. written by d3p_dpsvi_keys_dk).
extern "C" int32_t d3p_perturb_finalize_dk_f32(const float* partials_d, uint32_t n_partials, uint32_t P, uint32_t B,
                                               const d3p_leaf_table* leaves_h, const uint32_t* site_states_d,
                                               float dp_scale, float C, float obs_scale, float* grad_out_d,
                                               const d3p_optim_desc* optim_h, float* params_d, float* m_d, float* v_d,
                                               float* stats_d, d3p_comm* comm, void* stream) {
  if (!leaves_h || !site_states_d) return D3P_ERR_INVALID_ARGUMENT;
  return perturb_finalize_impl(partials_d, n_partials, P, B, leaves_h, site_states_d, dp_scale, C, obs_scale, 1, grad_out_d,
                               optim_h, params_d, m_d, v_d, stats_d, nullptr, comm, stream);
}

extern "C" size_t d3p_adadp_workspace_floats(uint32_t P) { return (size_t)(P + 31) / 32 + 2; }

extern "C" int32_t d3p_adadp_finish_f32(const d3p_optim_desc* optim_h, uint32_t P, float* params_d,
                                        const float* x_prev_d, void* stream) {
  if (!optim_h || optim_h->kind != D3P_OPT_ADADP || !optim_h->lr_d || !optim_h->err_ws_d || !params_d || !x_prev_d)
    return D3P_ERR_INVALID_ARGUMENT;
  unsigned grid = (P + 255) / 256;
  if (grid == 0) grid = 1;
  if (grid > 1184) grid = 1184;
  adadp_finish_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(optim_h->err_ws_d, optim_h->lr_d, optim_h->tol,
                                                              optim_h->stability_check, params_d, x_prev_d, P);
  return check_launch();
}
