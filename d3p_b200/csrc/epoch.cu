// Row f2 of the scope table: the whole `fori_loop(fetch -> update)` body of the examples
// (examples/logistic_regression.py:149-160, README.md:119-126) driven from C for the mean-field
// families.  One call = n_steps x { fold_in + minibatch sampler, 3-way key split, key conversion,
// fused per-example-gradient/clip/sum, per-leaf noise keys, finalize (+ ADADP finish) }, queued with no host
// synchronisation and no interpreter between the launches.  Host work per step is a handful of ChaCha blocks
// (<10 us); every device piece is the same entry point DPSVI.update uses, so the parameter trajectory is
// bit-identical to calling get_batch / update step by step.
//
// get_batch(i, state) depends on the batch key and on i only, never on the parameters, so the index sampler of
// step i + 1 is queued on a second (forked) stream and runs while step i's gradient kernel drains and its finalize
// kernel (latency-bound, a few CTAs; at N > 1 it also waits for the peers) holds the main stream.  idx / counts /
// mask are double-buffered; events order sampler(i) -> step(i) and step(i) -> sampler(i + 2).
#include <string.h>

#include <new>

#include "comm.cuh"
#include "common.cuh"
#include "launch.cuh"

using namespace d3p;

namespace {

struct EpochWs {
  uint8_t* base;
  size_t poisson_bytes, step_bytes, total;
  uint8_t* poisson;   // sampler scratch (Poisson only; used by the sampler stream alone)
  int32_t* idx[2];    // [batch], double-buffered over the step parity
  int32_t* counts[2]; // [2]
  uint8_t* mask[2];   // [batch]
  float* step;        // [n_partials, P + 2]
  // device-key mode (*_dk): per-step keys made on the device
  uint32_t* bkey[2];  // fold_in(batch_key, step) per sampler buffer
  uint32_t* rc[2];    // Feistel round constants per sampler buffer
  uint32_t* tf;       // Threefry key of the step
  uint32_t* sites;    // [D3P_MAX_LEAVES][16] per-leaf noise keys of the step
};

size_t align256(size_t v) { return (v + 255) & ~(size_t)255; }

bool layout_ws(size_t step_bytes, const d3p_sampler_desc* s, void* base, EpochWs& w) {
  w.step_bytes = step_bytes;
  if (w.step_bytes == 0) return false;
  w.poisson_bytes = s->kind == D3P_SAMPLER_POISSON ? d3p_poisson_workspace_bytes(s->n_records) : 0;
  size_t off = 0;
  w.base = static_cast<uint8_t*>(base);
  auto take = [&](size_t bytes) { size_t o = off; off += align256(bytes); return o; };
  const size_t o_poi = take(w.poisson_bytes), o_step = take(w.step_bytes);
  size_t o_idx[2], o_cnt[2], o_mask[2];
  for (int b = 0; b < 2; ++b) { o_idx[b] = take((size_t)s->batch * 4); o_cnt[b] = take(8); o_mask[b] = take(s->batch); }
  const size_t o_keys = take((2 * 16 + 2 * 32 + 64 + D3P_MAX_LEAVES * 16) * sizeof(uint32_t));
  w.total = off;
  if (base) {
    w.poisson = w.base + o_poi;
    w.step = reinterpret_cast<float*>(w.base + o_step);
    for (int b = 0; b < 2; ++b) {
      w.idx[b] = reinterpret_cast<int32_t*>(w.base + o_idx[b]);
      w.counts[b] = reinterpret_cast<int32_t*>(w.base + o_cnt[b]);
      w.mask[b] = w.base + o_mask[b];
    }
    uint32_t* k = reinterpret_cast<uint32_t*>(w.base + o_keys);
    w.bkey[0] = k; w.bkey[1] = k + 16; w.rc[0] = k + 32; w.rc[1] = k + 64; w.tf = k + 96; w.sites = k + 160;
  }
  return true;
}

bool sampler_ok(const d3p_sampler_desc* s) {
  if (!s || s->n_records == 0 || s->batch == 0) return false;
  if (s->kind == D3P_SAMPLER_POISSON) return s->q >= 0.f && s->q <= 1.f;
  if (s->kind == D3P_SAMPLER_SUBSAMPLE) return s->batch <= s->n_records;
  if (s->kind == D3P_SAMPLER_SPLIT) return s->batch <= s->n_records && s->perm_d != nullptr;
  return false;
}

}  // namespace

// Caller-owned resources of the epoch drivers: the forked sampler stream with its events and (VAE) the side streams of
// the step.  Creating a stream costs tens of microseconds, so a caller that runs many short epochs keeps one context;
// entry points called with ctx = NULL make a temporary one.
struct d3p_epoch_ctx {
  cudaStream_t samp = nullptr;
  cudaEvent_t ev_fork = nullptr, ev_sampled[2] = {nullptr, nullptr}, ev_consumed[2] = {nullptr, nullptr};
  d3p_vae_ctx* vae = nullptr;
};

extern "C" int32_t d3p_epoch_ctx_destroy(d3p_epoch_ctx* c) {
  if (!c) return D3P_OK;
  for (int b = 0; b < 2; ++b) {
    if (c->ev_sampled[b]) cudaEventDestroy(c->ev_sampled[b]);
    if (c->ev_consumed[b]) cudaEventDestroy(c->ev_consumed[b]);
  }
  if (c->ev_fork) cudaEventDestroy(c->ev_fork);
  if (c->samp) cudaStreamDestroy(c->samp);     // returns at once; the stream is released when its work has drained
  if (c->vae) d3p_vae_ctx_destroy(c->vae);
  delete c;
  return D3P_OK;
}

extern "C" int32_t d3p_epoch_ctx_create(d3p_epoch_ctx** out) {
  if (!out) return D3P_ERR_INVALID_ARGUMENT;
  *out = nullptr;
  d3p_epoch_ctx* c = new (std::nothrow) d3p_epoch_ctx();
  if (!c) return D3P_ERR_CUDA;
  bool ok = cudaStreamCreateWithFlags(&c->samp, cudaStreamNonBlocking) == cudaSuccess;
  ok = ok && cudaEventCreateWithFlags(&c->ev_fork, cudaEventDisableTiming) == cudaSuccess;
  for (int b = 0; b < 2 && ok; ++b)
    ok = cudaEventCreateWithFlags(&c->ev_sampled[b], cudaEventDisableTiming) == cudaSuccess &&
         cudaEventCreateWithFlags(&c->ev_consumed[b], cudaEventDisableTiming) == cudaSuccess;
  if (!ok) { d3p_epoch_ctx_destroy(c); return D3P_ERR_CUDA; }
  *out = c;
  return D3P_OK;
}

namespace {
// a context for the duration of one call when the caller passed none
struct CtxGuard {
  d3p_epoch_ctx* ctx; bool own = false;
  CtxGuard(d3p_epoch_ctx* c, bool needed) : ctx(c) {
    if (!ctx && needed) own = d3p_epoch_ctx_create(&ctx) == D3P_OK;
  }
  ~CtxGuard() { if (own) d3p_epoch_ctx_destroy(ctx); }
};

// rows of the batch handled by one rank of `world` (contiguous position ranges, the last one may be shorter)
uint32_t rows_per_rank(uint32_t B, int world) { return world > 1 ? (B + (uint32_t)world - 1) / (uint32_t)world : B; }

// The family-specific part of a step: the size of its workspace, and the launch of the fused per-example-gradient /
// clip / sum kernels of batch positions [pos_begin, pos_end) into the partial rows at `ws`.
struct StepLauncher {
  const float* x; size_t stride; float* params; uint32_t P;
  bool vae = false;       // the VAE step: side streams of a d3p_vae_ctx, a 256-byte aligned workspace
  StepLauncher(const float* x, size_t stride, float* params, uint32_t P) : x(x), stride(stride), params(params), P(P) {}
  // workspace of one step for `rows` batch rows per rank (partial rows first); 0 = unsupported description
  virtual size_t workspace(uint32_t rows, uint32_t* n_part) const = 0;
  // (tf_h, tf_d): the Threefry key of the step on the host or in device memory, one of them non-null
  virtual int32_t launch(const int32_t* idx, const uint8_t* mask, uint32_t B, uint32_t pos_begin, uint32_t pos_end,
                         const uint32_t* tf_h, const uint32_t* tf_d, float obs_scale, float C, void* ws, size_t ws_bytes,
                         d3p_vae_ctx* vae_ctx, cudaStream_t s) const = 0;
  virtual ~StepLauncher() {}
};

struct MeanfieldLauncher : StepLauncher {
  const d3p_meanfield_desc* desc; const int32_t* y;
  explicit MeanfieldLauncher(const d3p_meanfield_desc* d, const float* x = nullptr, size_t stride = 0,
                             const int32_t* y = nullptr, float* params = nullptr)
      : StepLauncher(x, stride, params, d->n_params), desc(d), y(y) {}
  size_t workspace(uint32_t, uint32_t* n_part) const override { return d3p_meanfield_workspace_bytes(desc, n_part); }
  int32_t launch(const int32_t* idx, const uint8_t* mask, uint32_t B, uint32_t pos_begin, uint32_t pos_end,
                 const uint32_t* tf_h, const uint32_t* tf_d, float obs_scale, float C, void* ws, size_t ws_bytes,
                 d3p_vae_ctx*, cudaStream_t s) const override {
    return step_meanfield_impl(desc, params, x, stride, y, idx, mask, nullptr, B, pos_begin, pos_end, tf_h, tf_d, obs_scale,
                               C, nullptr, nullptr, nullptr, ws, ws_bytes, s);
  }
};
struct GmmLauncher : StepLauncher {
  const d3p_gmm_desc* desc;
  explicit GmmLauncher(const d3p_gmm_desc* d, const float* x = nullptr, size_t stride = 0, float* params = nullptr)
      : StepLauncher(x, stride, params, d->n_params), desc(d) {}
  size_t workspace(uint32_t, uint32_t* n_part) const override { return d3p_gmm_workspace_bytes(desc, n_part); }
  int32_t launch(const int32_t* idx, const uint8_t* mask, uint32_t B, uint32_t pos_begin, uint32_t pos_end,
                 const uint32_t* tf_h, const uint32_t* tf_d, float obs_scale, float C, void* ws, size_t ws_bytes,
                 d3p_vae_ctx*, cudaStream_t s) const override {
    return step_gmm_impl(desc, params, x, stride, idx, mask, nullptr, B, pos_begin, pos_end, tf_h, tf_d, obs_scale, C,
                         nullptr, nullptr, nullptr, ws, ws_bytes, s);
  }
};
struct VaeLauncher : StepLauncher {
  const d3p_vae_desc* desc;
  explicit VaeLauncher(const d3p_vae_desc* d, const float* x = nullptr, size_t stride = 0, float* params = nullptr)
      : StepLauncher(x, stride, params, d->n_params), desc(d) { vae = true; }
  size_t workspace(uint32_t rows, uint32_t* n_part) const override { return d3p_vae_workspace_bytes(desc, rows, n_part); }
  int32_t launch(const int32_t* idx, const uint8_t* mask, uint32_t B, uint32_t pos_begin, uint32_t pos_end,
                 const uint32_t* tf_h, const uint32_t* tf_d, float obs_scale, float C, void* ws, size_t ws_bytes,
                 d3p_vae_ctx* vae_ctx, cudaStream_t s) const override {
    return step_vae_impl(desc, params, x, stride, idx, mask, nullptr, B, pos_begin, pos_end, tf_h, tf_d, obs_scale, C,
                         nullptr, nullptr, ws, ws_bytes, nullptr, vae_ctx, s);
  }
};

size_t epoch_ws_bytes(const StepLauncher& fam, const d3p_sampler_desc* sampler, int32_t world) {
  EpochWs w;
  uint32_t n_part = 0;
  if (!sampler_ok(sampler) || world < 1 ||
      !layout_ws(fam.workspace(rows_per_rank(sampler->batch, world), &n_part), sampler, nullptr, w))
    return 0;
  return w.total;
}

// The set-up and loop shared by the d3p_dpsvi_run_epoch_* entry points.  Keys: host words (batch_key_h, rng_key_io_h)
// or, for the *_dk entry points, device words (batch_key_d, rng_key_io_d).
int32_t run_epoch(const StepLauncher& fam, const d3p_sampler_desc* sampler, const uint32_t* batch_key_h,
                  uint32_t* rng_key_io_h, const uint32_t* batch_key_d, uint32_t* rng_key_io_d, uint32_t first_step,
                  uint32_t n_steps, float obs_scale, float C, float dp_scale, const d3p_leaf_table* leaves_h,
                  d3p_optim_desc* optim_io_h, float* m_d, float* v_d, float* stats_out_d, d3p_comm* comm, void* ws_d,
                  size_t ws_bytes, d3p_epoch_ctx* ctx, void* stream) {
  const bool dk = rng_key_io_d != nullptr;           // keys in device memory
  const bool split = sampler && sampler->kind == D3P_SAMPLER_SPLIT;      // pre-shuffled epoch: no sampler, no batch key
  if (!fam.x || !fam.params || (dk ? !batch_key_d : ((!split && !batch_key_h) || !rng_key_io_h)) || !leaves_h ||
      !optim_io_h || !ws_d)
    return D3P_ERR_INVALID_ARGUMENT;
  // a descriptor the finalize would refuse is refused before the first step kernel is queued
  if (const int32_t rc = optim_check(optim_io_h, fam.params, m_d, v_d); rc != D3P_OK) return rc;
  if (fam.vae && (reinterpret_cast<uintptr_t>(ws_d) & 255)) return D3P_ERR_INVALID_ARGUMENT;
  if (split && (uint64_t)(first_step + n_steps) * sampler->batch > sampler->n_records) return D3P_ERR_INVALID_ARGUMENT;
  if (!sampler_ok(sampler) || leaves_h->n_leaves == 0 || leaves_h->n_leaves > D3P_MAX_LEAVES)
    return D3P_ERR_INVALID_ARGUMENT;
  EpochWs w;
  uint32_t n_part = 0;
  if (!layout_ws(fam.workspace(rows_per_rank(sampler->batch, comm ? comm->world : 1), &n_part), sampler, ws_d, w))
    return D3P_ERR_UNSUPPORTED;
  if (ws_bytes < w.total) return D3P_ERR_WORKSPACE;
  const uint32_t B = sampler->batch, P = fam.P;

  d3p_leaf_table lt = *leaves_h;
  // sharded batch (SURVEY 8e): this rank handles a contiguous range of batch positions; the sampler and
  // all key derivations are replicated, the clipped sums meet inside the finalize kernel (comm.cuh)
  uint32_t pos_begin = 0, pos_end = B;
  if (comm && comm->world > 1) {
    const uint32_t per = (B + comm->world - 1) / comm->world;
    pos_begin = per * comm->rank < B ? per * comm->rank : B;
    pos_end = pos_begin + per < B ? pos_begin + per : B;
  }
  const bool fork = n_steps > 1 && !split;
  cudaStream_t main_s = (cudaStream_t)stream, samp_s = main_s;
  cudaEvent_t ev_sampled[2] = {nullptr, nullptr}, ev_consumed[2] = {nullptr, nullptr}, ev_fork = nullptr;
  CtxGuard guard(ctx, fork || fam.vae);          // a context only for the sampler stream or the VAE's side streams
  if ((fork || fam.vae) && !guard.ctx) return D3P_ERR_CUDA;
  if (fam.vae && !guard.ctx->vae && d3p_vae_ctx_create(&guard.ctx->vae) != D3P_OK) return D3P_ERR_CUDA;
  d3p_vae_ctx* const vae_ctx = fam.vae ? guard.ctx->vae : nullptr;
  if (fork) {
    samp_s = guard.ctx->samp;
    ev_fork = guard.ctx->ev_fork;
    for (int b = 0; b < 2; ++b) { ev_sampled[b] = guard.ctx->ev_sampled[b]; ev_consumed[b] = guard.ctx->ev_consumed[b]; }
    // the sampler stream starts after everything already queued on the caller's stream
    if (cudaEventRecord(ev_fork, main_s) != cudaSuccess || cudaStreamWaitEvent(samp_s, ev_fork, 0) != cudaSuccess)
      return D3P_ERR_CUDA;
  }
  // get_batch(i, batchifier_state): fold_in, then the index sampler (minibatch.py:103-131,217-237), into buffer i & 1
  auto queue_sampler = [&](uint32_t s) -> int32_t {
    const int b = s & 1;
    const bool poisson = sampler->kind == D3P_SAMPLER_POISSON;
    uint32_t bkey[16], rcs[30];
    int32_t r = D3P_OK;
    if (!dk && (r = d3p_chacha_fold_in_h(batch_key_h, first_step + s, bkey)) != D3P_OK) return r;
    if (fork && s >= 2 && cudaStreamWaitEvent(samp_s, ev_consumed[b], 0) != cudaSuccess) return D3P_ERR_CUDA;
    if (dk) {
      // the same keys made by one-block kernels, into the buffers of parity b (free once step s - 2 has consumed them)
      if ((r = d3p_chacha_fold_in_dk(batch_key_d, nullptr, first_step + s, w.bkey[b], samp_s)) != D3P_OK) return r;
      if (!poisson && (r = d3p_feistel_round_constants_dk(w.bkey[b], w.rc[b], samp_s)) != D3P_OK) return r;
    } else if (!poisson && (r = d3p_feistel_round_constants_h(bkey, rcs)) != D3P_OK) {
      return r;
    }
    const uint32_t* key_h = dk ? nullptr : bkey;
    const uint32_t* key_d = dk ? w.bkey[b] : nullptr;
    if (poisson) {
      r = D3P_ERR_UNSUPPORTED;
      if (comm && comm->world > 1)             // selector draw split over the ranks (samplers.cu)
        r = poisson_sample_sharded_impl(comm, key_h, key_d, sampler->q, sampler->n_records, B, sampler->suppress,
                                        pos_begin, pos_end, w.idx[b], w.counts[b], w.mask[b], w.poisson, w.poisson_bytes,
                                        samp_s);
      if (r == D3P_ERR_UNSUPPORTED)            // same decision on every rank (window size, tiles >= ranks)
        r = poisson_sample_impl(key_h, key_d, sampler->q, sampler->n_records, B, sampler->suppress, w.idx[b], w.counts[b],
                                w.mask[b], w.poisson, w.poisson_bytes, samp_s);
    } else {
      r = feistel_sample_impl(dk ? nullptr : rcs, dk ? w.rc[b] : nullptr, sampler->n_records, 0, B, w.idx[b], samp_s);
    }
    if (r == D3P_OK && fork && cudaEventRecord(ev_sampled[b], samp_s) != cudaSuccess) r = D3P_ERR_CUDA;
    return r;
  };
  int32_t rc = D3P_OK;
  if (fork) rc = queue_sampler(0);
  for (uint32_t s = 0; s < n_steps && rc == D3P_OK; ++s) {
    const int b = s & 1;
    if (split) {
      // nothing to sample: this step's records are a slice of the epoch's shuffle
    } else if (fork) {
      if (s + 1 < n_steps && (rc = queue_sampler(s + 1)) != D3P_OK) break;      // runs ahead on the sampler stream
      if (cudaStreamWaitEvent(main_s, ev_sampled[b], 0) != cudaSuccess) { rc = D3P_ERR_CUDA; break; }
    } else if ((rc = queue_sampler(s)) != D3P_OK) {
      break;
    }
    const uint8_t* mask = sampler->kind == D3P_SAMPLER_POISSON ? w.mask[b] : nullptr;
    const int32_t* idx = split ? sampler->perm_d + (size_t)(first_step + s) * B : w.idx[b];
    // ---- DPSVI.update (svi.py:395-434) ----------------------------------------------------------------------
    // carry / k_grad -> Threefry key / k_noise -> per-leaf keys: in host C, or all on the device with the state key
    // advanced in place
    uint32_t keys[3][16], tf[2];
    if (dk) {
      if ((rc = d3p_dpsvi_keys_dk(rng_key_io_d, lt.n_leaves, w.tf, w.sites, main_s)) != D3P_OK) break;
    } else {
      if ((rc = d3p_chacha_split_h(rng_key_io_h, 3, &keys[0][0])) != D3P_OK) break;           // carry, k_grad, k_noise
      if ((rc = d3p_chacha_random_bits_h(keys[1], 0, tf, 2)) != D3P_OK) break;                // convert_to_jax_rng_key
    }
    rc = fam.launch(idx, mask, B, pos_begin, pos_end, dk ? nullptr : tf, dk ? w.tf : nullptr, obs_scale, C, w.step,
                    w.step_bytes, vae_ctx, main_s);
    if (rc != D3P_OK) break;
    if (!dk && (rc = d3p_chacha_split_h(keys[2], (int32_t)lt.n_leaves, &lt.site_state[0][0])) != D3P_OK) break;
    rc = perturb_finalize_impl(w.step, n_part, P, B, &lt, dk ? w.sites : nullptr, dp_scale, C, obs_scale, 1, nullptr,
                               optim_io_h, fam.params, m_d, v_d, stats_out_d ? stats_out_d + 3 * (size_t)s : nullptr,
                               nullptr, comm, main_s);
    if (rc != D3P_OK) break;
    // recorded after the finalize launch so that nothing sits between the step kernel and its programmatic dependent
    if (fork && cudaEventRecord(ev_consumed[b], main_s) != cudaSuccess) { rc = D3P_ERR_CUDA; break; }
    if (optim_io_h->kind == D3P_OPT_ADADP && (optim_io_h->step & 1))
      if ((rc = d3p_adadp_finish_f32(optim_io_h, P, fam.params, v_d, main_s)) != D3P_OK) break;
    optim_io_h->step += 1;
    if (!dk) memcpy(rng_key_io_h, keys[0], sizeof(keys[0]));
  }
  if (fork) {
    // join: whatever is still queued on the sampler stream (only after an error) precedes later work of the caller
    if (cudaEventRecord(ev_fork, samp_s) == cudaSuccess) cudaStreamWaitEvent(main_s, ev_fork, 0);
  }
  return rc;
}

}  // namespace

extern "C" size_t d3p_dpsvi_epoch_workspace_bytes(const d3p_meanfield_desc* desc, const d3p_sampler_desc* sampler) {
  return desc ? epoch_ws_bytes(MeanfieldLauncher(desc), sampler, 1) : 0;
}

extern "C" size_t d3p_dpsvi_epoch_vae_workspace_bytes(const d3p_vae_desc* desc, const d3p_sampler_desc* sampler,
                                                      int32_t world) {
  return desc ? epoch_ws_bytes(VaeLauncher(desc), sampler, world) : 0;
}

extern "C" int32_t d3p_dpsvi_run_epoch_meanfield(const d3p_meanfield_desc* desc, const d3p_sampler_desc* sampler,
                                                 const float* x_d, size_t x_row_stride, const int32_t* y_d,
                                                 const uint32_t batch_key_h[16], uint32_t rng_key_io_h[16],
                                                 uint32_t first_step, uint32_t n_steps, float obs_scale, float C,
                                                 float dp_scale, const d3p_leaf_table* leaves_h,
                                                 d3p_optim_desc* optim_io_h, float* params_d, float* m_d, float* v_d,
                                                 float* stats_out_d, d3p_comm* comm, void* ws_d, size_t ws_bytes,
                                                 d3p_epoch_ctx* ctx, void* stream) {
  if (!desc) return D3P_ERR_INVALID_ARGUMENT;
  return run_epoch(MeanfieldLauncher(desc, x_d, x_row_stride, y_d, params_d), sampler, batch_key_h, rng_key_io_h, nullptr,
                   nullptr, first_step, n_steps, obs_scale, C, dp_scale, leaves_h, optim_io_h, m_d, v_d, stats_out_d, comm,
                   ws_d, ws_bytes, ctx, stream);
}

// Device-key form: the batchifier key and the DPSVI state key live in device memory (rng_key_io_d is advanced in place),
// every per-step key is derived by one-block kernels on the stream: the loop body of a jitted fori_loop with traced
// keys (examples/logistic_regression.py:149-160) without a host round trip.  Same kernels, same results.
extern "C" int32_t d3p_dpsvi_run_epoch_meanfield_dk(const d3p_meanfield_desc* desc, const d3p_sampler_desc* sampler,
                                                    const float* x_d, size_t x_row_stride, const int32_t* y_d,
                                                    const uint32_t* batch_key_d, uint32_t* rng_key_io_d,
                                                    uint32_t first_step, uint32_t n_steps, float obs_scale, float C,
                                                    float dp_scale, const d3p_leaf_table* leaves_h,
                                                    d3p_optim_desc* optim_io_h, float* params_d, float* m_d, float* v_d,
                                                    float* stats_out_d, d3p_comm* comm, void* ws_d, size_t ws_bytes,
                                                    d3p_epoch_ctx* ctx, void* stream) {
  if (!desc) return D3P_ERR_INVALID_ARGUMENT;
  return run_epoch(MeanfieldLauncher(desc, x_d, x_row_stride, y_d, params_d), sampler, nullptr, nullptr, batch_key_d,
                   rng_key_io_d, first_step, n_steps, obs_scale, C, dp_scale, leaves_h, optim_io_h, m_d, v_d, stats_out_d,
                   comm, ws_d, ws_bytes, ctx, stream);
}

// The same loop for the mixture model (examples/gaussian_mixture_model.py:205-218).
extern "C" size_t d3p_dpsvi_epoch_gmm_workspace_bytes(const d3p_gmm_desc* desc, const d3p_sampler_desc* sampler) {
  return desc ? epoch_ws_bytes(GmmLauncher(desc), sampler, 1) : 0;
}

extern "C" int32_t d3p_dpsvi_run_epoch_gmm(const d3p_gmm_desc* desc, const d3p_sampler_desc* sampler, const float* x_d,
                                           size_t x_row_stride, const uint32_t batch_key_h[16],
                                           uint32_t rng_key_io_h[16], uint32_t first_step, uint32_t n_steps,
                                           float obs_scale, float C, float dp_scale, const d3p_leaf_table* leaves_h,
                                           d3p_optim_desc* optim_io_h, float* params_d, float* m_d, float* v_d,
                                           float* stats_out_d, d3p_comm* comm, void* ws_d, size_t ws_bytes, d3p_epoch_ctx* ctx,
                                           void* stream) {
  if (!desc) return D3P_ERR_INVALID_ARGUMENT;
  return run_epoch(GmmLauncher(desc, x_d, x_row_stride, params_d), sampler, batch_key_h, rng_key_io_h, nullptr, nullptr,
                   first_step, n_steps, obs_scale, C, dp_scale, leaves_h, optim_io_h, m_d, v_d, stats_out_d, comm, ws_d,
                   ws_bytes, ctx, stream);
}

// The same loop for the VAE family (examples/vae.py:216-233 runs fori_loop(get_batch -> update) per epoch).
extern "C" int32_t d3p_dpsvi_run_epoch_vae(const d3p_vae_desc* desc, const d3p_sampler_desc* sampler, const float* x_d,
                                           size_t x_row_stride, const uint32_t batch_key_h[16],
                                           uint32_t rng_key_io_h[16], uint32_t first_step, uint32_t n_steps,
                                           float obs_scale, float C, float dp_scale, const d3p_leaf_table* leaves_h,
                                           d3p_optim_desc* optim_io_h, float* params_d, float* m_d, float* v_d,
                                           float* stats_out_d, d3p_comm* comm, void* ws_d, size_t ws_bytes, d3p_epoch_ctx* ctx,
                                           void* stream) {
  if (!desc) return D3P_ERR_INVALID_ARGUMENT;
  return run_epoch(VaeLauncher(desc, x_d, x_row_stride, params_d), sampler, batch_key_h, rng_key_io_h, nullptr, nullptr,
                   first_step, n_steps, obs_scale, C, dp_scale, leaves_h, optim_io_h, m_d, v_d, stats_out_d, comm, ws_d,
                   ws_bytes, ctx, stream);
}

extern "C" int32_t d3p_dpsvi_run_epoch_vae_dk(const d3p_vae_desc* desc, const d3p_sampler_desc* sampler, const float* x_d,
                                              size_t x_row_stride, const uint32_t* batch_key_d, uint32_t* rng_key_io_d,
                                              uint32_t first_step, uint32_t n_steps, float obs_scale, float C,
                                              float dp_scale, const d3p_leaf_table* leaves_h, d3p_optim_desc* optim_io_h,
                                              float* params_d, float* m_d, float* v_d, float* stats_out_d, d3p_comm* comm,
                                              void* ws_d, size_t ws_bytes, d3p_epoch_ctx* ctx, void* stream) {
  if (!desc) return D3P_ERR_INVALID_ARGUMENT;
  return run_epoch(VaeLauncher(desc, x_d, x_row_stride, params_d), sampler, nullptr, nullptr, batch_key_d, rng_key_io_d,
                   first_step, n_steps, obs_scale, C, dp_scale, leaves_h, optim_io_h, m_d, v_d, stats_out_d, comm, ws_d,
                   ws_bytes, ctx, stream);
}
