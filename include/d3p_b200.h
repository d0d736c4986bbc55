/* d3p_b200 — C ABI of the B200-native DP-VI update path.
 *
 * This is the drop-in boundary for the hot path of DPBayes/d3p (reference paths are relative
 * to the d3p repository root).  Every entry point
 *   - is `extern "C"`, takes plain pointers and sizes (no torch / jax types),
 *   - returns D3P_OK (0) or a negative D3P_ERR_* code, never throws,
 *   - never allocates device memory and never synchronises the device (pointer arguments
 *     with suffix `_d` are DEVICE pointers, suffix `_h` HOST pointers; scratch space comes
 *     from the caller, sized by the matching `*_workspace_bytes` query),
 *   - enqueues its kernels on `stream` (a `cudaStream_t` passed as `void*`; NULL = default),
 *   - keeps no global mutable state (the only statics are write-once caches of immutable facts: the SM count of a
 *     device, the driver's cuTensorMapEncodeTiled entry point) and is re-entrant across streams and threads;
 *     handles (d3p_comm, d3p_vae_ctx, d3p_epoch_ctx) are caller-owned and serve one caller at a time.
 * One process per GPU; the caller selects the device with cudaSetDevice before calling.
 *
 * ChaCha states are 16 x uint32 in RFC 8439 layout (constants | 8 key words | counter |
 * 3 nonce words), i.e. jax-chacha-prng's 4x4 `RNGState` flattened row-major.
 */
#ifndef D3P_B200_H_
#define D3P_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define D3P_OK 0
#define D3P_ERR_INVALID_ARGUMENT (-1)
#define D3P_ERR_CUDA (-2)
#define D3P_ERR_UNSUPPORTED (-3)
#define D3P_ERR_WORKSPACE (-4)
#define D3P_ERR_PEER_TIMEOUT (-5) /* sticky: a peer-memory exchange of this window timed out earlier */

#define D3P_MAX_LEAVES 16

/* Library / build identification. */
typedef struct d3p_comm d3p_comm;       /* peer-memory window of a sharded run, see d3p_comm_create */
typedef struct d3p_epoch_ctx d3p_epoch_ctx; /* streams / events of the epoch drivers, see d3p_epoch_ctx_create */
typedef struct d3p_vae_ctx d3p_vae_ctx; /* side streams of the VAE step, see d3p_vae_ctx_create */

int32_t d3p_abi_version(void);
const char* d3p_error_string(int32_t code);

/* CUDA events for callers without a CUDA binding (device timing on the launching stream). */
int32_t d3p_event_create(void** event_out);
int32_t d3p_event_record(void* event, void* stream);
int32_t d3p_event_elapsed_ms(void* begin, void* end, float* ms_out); /* synchronises on `end` */
int32_t d3p_event_destroy(void* event);

/* ------------------------------------------------------------------------------------------
 * ChaCha20 rng suite — replaces jax-chacha-prng behind d3p/random/__init__.py:28-32.
 * ------------------------------------------------------------------------------------------ */

/* d3p.random.PRNGKey (d3p/random/__init__.py:35-47): <=32 seed bytes, zero padded. */
int32_t d3p_chacha_key_from_seed_h(const uint8_t* seed_h, size_t len, uint32_t out_h[16]);
/* rng_suite.fold_in (d3p/random/__init__.py:30; call sites d3p/minibatch.py:115,207,230). */
int32_t d3p_chacha_fold_in_h(const uint32_t in_h[16], uint32_t data, uint32_t out_h[16]);
/* rng_suite.split (d3p/random/__init__.py:29; call sites d3p/svi.py:210,447,491). out = num x 16. */
int32_t d3p_chacha_split_h(const uint32_t in_h[16], int32_t num, uint32_t* out_h);
/* Host keystream (few words): rng_suite.random_bits for tiny outputs, e.g.
 * convert_to_jax_rng_key (d3p/random/__init__.py:149-155) and the Feistel round constants
 * (d3p/util.py:240-246). */
int32_t d3p_chacha_random_bits_h(const uint32_t state_h[16], uint64_t first_block, uint32_t* out_h,
                                 size_t n_words);
/* Device keystream: rng_suite.random_bits(key, 32, shape) (d3p/random/__init__.py:31). */
int32_t d3p_chacha_random_bits(const uint32_t state_h[16], uint64_t first_block, uint32_t* out_d,
                               size_t n_words, void* stream);
/* rng_suite.uniform(key, shape, float32, lo, hi) (d3p/random/__init__.py:32). */
int32_t d3p_chacha_uniform_f32(const uint32_t state_h[16], uint64_t first_block, float lo, float hi,
                               float* out_d, size_t n, void* stream);
/* d3p.random.normal (d3p/random/__init__.py:50-81): sqrt(2) * erf_inv(uniform(lo=-1+ulp, hi=1)). */
int32_t d3p_chacha_normal_f32(const uint32_t state_h[16], uint64_t first_block, float* out_d, size_t n,
                              void* stream);
/* One rejection round of d3p.random._randint (d3p/random/__init__.py:128-143) for 32-bit
 * outputs: vals[i] = (first || vals[i] > delta) ? bits(round_key)[i] & bitmask : vals[i];
 * *pending_d = number of lanes still > delta afterwards. */
int32_t d3p_chacha_randint_round_u32(const uint32_t round_state_h[16], uint32_t bitmask, uint32_t delta,
                                     int32_t first, uint32_t* vals_d, size_t n, int32_t* pending_d,
                                     void* stream);
/* vals -> int32 indices: idx = int32(vals) + minval. */
int32_t d3p_randint_finish_i32(const uint32_t* vals_d, int32_t minval, int32_t* out_d, size_t n, void* stream);
/* The same pair for the other result widths of d3p.random.randint (d3p/random/__init__.py:113-124: nbits = bits of
 * the result dtype, draws are random_bits(round_key, nbits, shape)): nbits = 8, 16 or 32; vals_d stays uint32 per
 * element; out_d is int8 / int16 / int32 and the addition wraps in that type. */
int32_t d3p_chacha_randint_round(const uint32_t round_state_h[16], uint32_t nbits, uint32_t bitmask, uint32_t delta,
                                 int32_t first, uint32_t* vals_d, size_t n, int32_t* pending_d, void* stream);
int32_t d3p_randint_finish(const uint32_t* vals_d, int32_t minval, uint32_t nbits, void* out_d, size_t n, void* stream);
/* The whole of d3p.random.randint(key, (n,), minval, maxval, int{nbits}) (d3p/random/__init__.py:84-146) in one launch,
 * with no host synchronisation: key_h is the key randint receives (the kernel does the first split itself); out_d is
 * int8 / int16 / int32 for nbits = 8, 16, 32 and gets the values of the per-round loop above bit for bit.
 * nbits outside {8, 16, 32}: D3P_ERR_UNSUPPORTED; n == 0: D3P_OK without a launch; a null pointer with n > 0:
 * D3P_ERR_INVALID_ARGUMENT.  Both refusals come before any launch. */
int32_t d3p_chacha_randint(const uint32_t key_h[16], uint32_t nbits, int64_t minval, int64_t maxval, void* out_d,
                           size_t n, void* stream);
/* randint's rejection mask for delta = (maxval - 1 - minval) mod 2^nbits: 2^log_po2 - 1 with
 * log_po2 = min(int(float32(log2(float32(delta))) + 1), nbits) and 0 for delta == 0 (host only, no device work). */
uint32_t d3p_randint_bitmask(uint32_t nbits, uint32_t delta);

/* ------------------------------------------------------------------------------------------
 * Minibatch samplers — replace d3p/util.py:216-301 and d3p/minibatch.py:29-39,103-131,217-237.
 * ------------------------------------------------------------------------------------------ */

/* Round constants of sample_from_array (d3p/util.py:240-246): 30 keystream words, rc[3j] |= 1. */
int32_t d3p_feistel_round_constants_h(const uint32_t state_h[16], uint32_t rc_h[30]);
/* idx[p - first_pos] = walk(pi_rc(p)) for p in [first_pos, first_pos + n) (d3p/util.py:249-299). */
int32_t d3p_feistel_sample(const uint32_t rc_h[30], uint32_t capacity, uint32_t first_pos, uint32_t n,
                           int32_t* idx_d, void* stream);

/* poisson_sample_idxs + truncate/suppress + mask (d3p/minibatch.py:29-39,115-124).
 * idx_d[max_b]: selected indices in DESCENDING order, then unselected indices descending.
 * counts_d[0] = raw number selected, counts_d[1] = effective count after truncate / suppress.
 * mask_d[max_b] (may be NULL) = arange(max_b) < counts_d[1].
 * Multi-GPU: every rank runs the (cheap, ALU-only) sampler on the replicated key, so the
 * index list is bit-identical on all ranks without any collective. */
size_t d3p_poisson_workspace_bytes(uint32_t n_records);
int32_t d3p_poisson_sample(const uint32_t state_h[16], float q, uint32_t n_records, uint32_t max_b,
                           int32_t suppress, int32_t* idx_d, int32_t* counts_d, uint8_t* mask_d, void* ws_d,
                           size_t ws_bytes, void* stream);

/* mask * take(a, idxs, axis=0) (d3p/minibatch.py:126-131,210,233,306).
 * dst[r, :] = (num_valid_d == NULL || r < *num_valid_d) ? src[idx[r], :] : 0 ; any row_bytes > 0 (16-byte vectors
 * when rows and pointers allow, else 4-byte words, else bytes). */
int32_t d3p_gather_rows_masked(const void* src_d, size_t row_bytes, const int32_t* idx_d,
                               const int32_t* num_valid_d, uint32_t b, void* dst_d, void* stream);

/* ------------------------------------------------------------------------------------------
 * Per-example clipping on materialised gradients — replace d3p/svi.py:68-124,310-348.
 * px_grads is [B, P] row-major float32: the concatenation of the ravelled leaves per example.
 * ------------------------------------------------------------------------------------------ */

/* DPSVI._clip_gradients (d3p/svi.py:310-325): rows scaled in place by 1/max(1, norm/C).
 * norms_d (may be NULL) receives the pre-clip L2 norms (full_norm, d3p/svi.py:68-87). */
int32_t d3p_clip_rows_f32(float* px_grads_d, uint32_t B, uint32_t P, float C, float* norms_d, void* stream);
/* full_norm(parts, ord) for ord != 2 (d3p/svi.py:68-87): out_d[0] = ||x||_ord of n floats; ord = +-inf, 0, 1 or p. */
int32_t d3p_vector_norm_f32(const float* x_d, size_t n, float ord, float* out_d, void* stream);
/* Fused clip + sum over examples (d3p/svi.py:310-348 without the [B,P] round trip):
 * sum_d[P + 2] = { sum_i m_i c_i g_i , sum_i m_i loss_i (px_loss_d may be NULL), sum_i m_i }. */
size_t d3p_clip_and_sum_workspace_bytes(uint32_t B, uint32_t P);
int32_t d3p_clip_and_sum_f32(const float* px_grads_d, const float* px_loss_d, const uint8_t* mask_d,
                             uint32_t B, uint32_t P, float C, float* sum_d, void* ws_d, size_t ws_bytes,
                             void* stream);

/* ------------------------------------------------------------------------------------------
 * Fused per-example gradient + clip + sum for mean-field Normal guides — replaces
 * d3p/svi.py:238-348 for the model/guide pairs of examples/logistic_regression.py:49-86 and
 * examples/simple_gaussian_posterior.py:50-83 (and their AutoDiagonalNormal variants,
 * README.md:81,102).  No [B, P] tensor is materialised.
 * ------------------------------------------------------------------------------------------ */
#define D3P_FAMILY_LOGREG 0 /* Bernoulli(logits = x.w + b), N(0,1) priors          */
#define D3P_FAMILY_GAUSS 1  /* x ~ N(mu, lik_scale) per dimension, N(0,1) prior on mu */
#define D3P_LINK_EXP 0      /* scale = exp(rho)       (examples' hand-written guides) */
#define D3P_LINK_SOFTPLUS 1 /* scale = softplus(rho)  (AutoDiagonalNormal)            */

typedef struct {
  int32_t family;       /* D3P_FAMILY_*                                                    */
  int32_t link;         /* D3P_LINK_*                                                      */
  int32_t joint_site;   /* 0: one guide sample site per latent (w, then intercept);        */
                        /* 1: a single `_auto_latent` site holding [w..., intercept]        */
  uint32_t d;           /* data columns                                                    */
  uint32_t n_params;    /* P: length of the flat parameter vector                          */
  uint32_t loc_off;     /* offset of the d weight/mean location params in the flat vector  */
  uint32_t rho_off;     /* offset of the d unconstrained scale params                      */
  uint32_t b_loc_off;   /* LOGREG only: offset of the intercept location                   */
  uint32_t b_rho_off;   /* LOGREG only: offset of the intercept unconstrained scale        */
  float num_obs_total;  /* plate size N  (static kwarg `num_obs_total`)                    */
  float lik_scale;      /* GAUSS only: likelihood standard deviation                       */
} d3p_meanfield_desc;

/* Rows per row of the partial-sum workspace: P + 2 (grad sum | loss sum | valid count). */
size_t d3p_meanfield_workspace_bytes(const d3p_meanfield_desc* desc, uint32_t* n_partials_out);

/* One pass over a batch: for every position p < B with (mask_d == NULL || mask_d[p]) and
 * (num_valid_d == NULL || p < *num_valid_d):
 *     row = idx_d ? idx_d[p] : p ;  key_p = jax.random.split(threefry_key, B)[p]
 *     eps  = numpyro seed/Normal.sample plumbing ; g_p = grad of (1/obs_scale) * (-ELBO_p)
 *     c_p  = 1 / max(1, ||g_p|| / C)
 * and writes per-CTA partial sums of { c_p g_p , obs_scale * loss_p , 1 } to ws_d
 * ([n_partials, P + 2]); they are reduced in a fixed order by d3p_perturb_finalize_f32.
 * `pos_begin/pos_end` restrict the positions handled by this rank (sharded batch).
 * px_norms_d[B] (may be NULL) receives the pre-clip norms; px_grads_d[B, P] / px_loss_d[B] (may
 * be NULL) receive the UNCLIPPED per-example gradients and obs_scale * loss_p — the stage-method
 * form DPSVI._compute_per_example_gradients (d3p/svi.py:238-308).  Masked positions are not
 * written (the caller zero-fills). */
int32_t d3p_dpsvi_step_meanfield(const d3p_meanfield_desc* desc, const float* params_d, const float* x_d,
                                 size_t x_row_stride /* floats */, const int32_t* y_d, const int32_t* idx_d,
                                 const uint8_t* mask_d, const int32_t* num_valid_d, uint32_t B,
                                 uint32_t pos_begin, uint32_t pos_end, const uint32_t threefry_key_h[2],
                                 float obs_scale, float C, float* px_norms_d, float* px_grads_d, float* px_loss_d,
                                 void* ws_d, size_t ws_bytes, void* stream);

/* ------------------------------------------------------------------------------------------
 * AutoDiagonalNormal guide over a user model (d3p_b200.models.AutoDiagonalNormalModel): one
 * `_auto_latent` site of D real-valued elements, parameters auto_loc[D] and auto_scale[D]
 * (softplus link).  Everything but the model's log density runs here: the caller draws
 * theta_i = loc + softplus(rho) * eps_i with d3p_autodiag_draw_f32, evaluates the potential
 *     U_i = -log p(theta_i) - N log p(x_i | theta_i)
 * and its gradient h_i = dU_i / dtheta_i itself (autodiff of the model), and d3p_dpsvi_step_autodiag
 * forms (with S = obs_scale, s = softplus(rho), a = sigmoid(rho))
 *     gl_i = h_i / S ,   gs_i = gl_i * eps_i * a - (1/S) a / s
 *     S * loss_i = U_i - |eps_i|^2 / 2 - sum_e log s_e - D log sqrt(2 pi)
 * and clips and sums them as d3p_dpsvi_step_meanfield does.  Row r of theta_d / eps_d / grad_d /
 * potential_d belongs to batch position pos_begin + r; rows are `ld` floats apart.
 * ------------------------------------------------------------------------------------------ */
typedef struct {
  uint32_t latent_dim;  /* D: elements of the `_auto_latent` site                         */
  uint32_t n_params;    /* P: length of the flat parameter vector                          */
  uint32_t loc_off;     /* offset of auto_loc[D] in the flat vector                        */
  uint32_t scale_off;   /* offset of auto_scale[D] (unconstrained: scale = softplus)        */
  float num_obs_total;  /* plate size N, the factor of the log-likelihood inside U          */
} d3p_autodiag_desc;

/* The guide draws of batch positions [pos_begin, pos_end): eps_d / theta_d row r receive the
 * draw of key_p = jax.random.split(threefry_key, B)[pos_begin + r] through the seed-handler
 * plumbing of the fused AutoDiagonalNormal families ((model_seed, guide_seed) = split(key_p),
 * one site split; Threefry call j yields elements j and j + ceil(D/2)), with the step kernels'
 * normal transform.  Every position of the range is drawn (no mask).  B == 0: ONE draw from
 * threefry_key itself (no example split, pos_begin / pos_end ignored) with the exact transform of
 * d3p_elbo_evaluate_meanfield — SVI.evaluate's draw. */
int32_t d3p_autodiag_draw_f32(const d3p_autodiag_desc* desc, const float* params_d, const uint32_t threefry_key_h[2],
                              uint32_t B, uint32_t pos_begin, uint32_t pos_end, float* theta_d, float* eps_d,
                              size_t ld, void* stream);
/* Workspace of a step over `rows` batch rows; its first n_partials * (P + 2) floats are the
 * partial rows that d3p_perturb_finalize_* reduce. */
size_t d3p_autodiag_workspace_bytes(const d3p_autodiag_desc* desc, uint32_t rows, uint32_t* n_partials_out);
/* Partial rows { sum c_i gl_i | sum c_i gs_i | sum S loss_i | count } over the positions p of
 * [pos_begin, pos_end) with (mask_d == NULL || mask_d[p]) and (num_valid_d == NULL || p < *num_valid_d),
 * c_i = 1 / max(1, |(gl_i, gs_i)| / C); the other rows of eps_d / grad_d / potential_d are not
 * read.  px_norms_d[B], px_grads_d[B, P], px_loss_d[B] (may be NULL) as in d3p_dpsvi_step_meanfield. */
int32_t d3p_dpsvi_step_autodiag(const d3p_autodiag_desc* desc, const float* params_d, const float* eps_d,
                                const float* grad_d, size_t ld, const float* potential_d, const uint8_t* mask_d,
                                const int32_t* num_valid_d, uint32_t B, uint32_t pos_begin, uint32_t pos_end,
                                float obs_scale, float C, float* px_norms_d, float* px_grads_d, float* px_loss_d,
                                void* ws_d, size_t ws_bytes, void* stream);

/* ------------------------------------------------------------------------------------------
 * Reduce + perturb + rescale (+ optimizer) — replaces d3p/svi.py:327-393,470-498.
 * ------------------------------------------------------------------------------------------ */
#define D3P_OPT_NONE 0
#define D3P_OPT_SGD 1
#define D3P_OPT_ADAM 2
#define D3P_OPT_ADADP 3 /* d3p.optimizers.ADADP (d3p/optimizers.py:29-131) */
/* numpyro.optim wrappers of jax.example_libraries.optimizers; g = the released noisy gradient, lr = step_size(i):
 *   MOMENTUM          m = momentum * m + g;                           x -= lr * m            (momentum = numpyro's mass)
 *   ADAGRAD           v += g^2; r = v > 0 ? 1 / sqrt(v) : 0;
 *                     m = (1 - momentum) * (g * r) + momentum * m;     x -= lr * m
 *   RMSPROP           v = v * gamma + g^2 * (1 - gamma);               x -= lr * g / sqrt(v + eps)
 *   RMSPROP_MOMENTUM  v as RMSPROP; m = momentum * m + lr * g / sqrt(v + eps);  x -= m
 *   CLIPPED_ADAM      Adam (b1, b2, eps) on clip(g, -clip_norm, clip_norm); grad_out_d still receives g */
#define D3P_OPT_MOMENTUM 4
#define D3P_OPT_ADAGRAD 5
#define D3P_OPT_RMSPROP 6
#define D3P_OPT_RMSPROP_MOMENTUM 7
#define D3P_OPT_CLIPPED_ADAM 8
/* OR-ed into `kind`: step_size is the schedule `schedule` (fields below) evaluated at `step`, not a constant.  Not
 * valid with NONE or ADADP (whose step size is device state). */
#define D3P_OPT_SCHEDULED 0x100
/* Step-size schedules of jax.example_libraries.optimizers, s = step_size, i = step, float32 arithmetic: */
#define D3P_SCHED_CONSTANT 0     /* s                                                                              */
#define D3P_SCHED_EXPONENTIAL 1  /* s * decay_rate ** (i / decay_steps)                                            */
#define D3P_SCHED_INVERSE_TIME 2 /* s / (1 + decay_rate * i / decay_steps); staircase: i / decay_steps floored     */
#define D3P_SCHED_POLYNOMIAL 3   /* n = min(i, decay_steps): (1 - n / decay_steps) ** power * (s - final) + final  */
#define D3P_SCHED_PIECEWISE 4    /* values[#{b in boundaries : i > b}]                                             */
#define D3P_MAX_BOUNDARIES 16

typedef struct {
  uint32_t n_leaves;
  uint32_t leaf_off[D3P_MAX_LEAVES]; /* offset of each leaf in the flat vector (pytree order) */
  uint32_t leaf_len[D3P_MAX_LEAVES];
  uint32_t site_state[D3P_MAX_LEAVES][16]; /* rng_suite.split(k_noise, n_leaves) (d3p/svi.py:491) */
} d3p_leaf_table;

typedef struct {
  int32_t kind;       /* D3P_OPT_*                               */
  float step_size;
  float b1, b2, eps;  /* Adam                                     */
  int32_t step;       /* numpyro optimizer step counter i (>= 0)  */
  /* ADADP only (d3p/optimizers.py:29-116).  State mapping: params_d = x, m_d = x_stepped,
   * v_d = x_prev; the adaptive step size lives on the device so that no step synchronises.   */
  float tol;               /* error tolerance                                                */
  int32_t stability_check; /* reject the odd step when err > tol (optimizers.py:92-97)       */
  float* lr_d;             /* device scalar: current step size, updated by d3p_adadp_finish  */
  float* err_ws_d;         /* device scratch, >= d3p_adadp_workspace_floats(P) floats        */
  /* Appended fields: read only when `kind` names MOMENTUM .. CLIPPED_ADAM or carries D3P_OPT_SCHEDULED, so a caller
   * that knows only the fields above never has them read. */
  float momentum;          /* MOMENTUM: mass; ADAGRAD, RMSPROP_MOMENTUM: momentum             */
  float gamma;             /* RMSPROP, RMSPROP_MOMENTUM: decay of the squared-gradient average */
  float clip_norm;         /* CLIPPED_ADAM: element-wise clip bound (> 0)                     */
  int32_t schedule;        /* D3P_SCHED_* (with D3P_OPT_SCHEDULED)                            */
  float decay_steps;       /* EXPONENTIAL, INVERSE_TIME, POLYNOMIAL (> 0)                     */
  float decay_rate;        /* EXPONENTIAL, INVERSE_TIME                                       */
  int32_t staircase;       /* INVERSE_TIME                                                    */
  float final_step_size;   /* POLYNOMIAL                                                      */
  float power;             /* POLYNOMIAL                                                      */
  uint32_t n_boundaries;   /* PIECEWISE: <= D3P_MAX_BOUNDARIES                                */
  float boundaries[D3P_MAX_BOUNDARIES];
  float values[D3P_MAX_BOUNDARIES + 1]; /* PIECEWISE: n_boundaries + 1 step sizes            */
} d3p_optim_desc;

/* The step size of `optim_h` at optimizer step `step` (its own counter, starting at 0): step_size, or with
 * D3P_OPT_SCHEDULED the schedule, evaluated in float32 on the host.  d3p_perturb_finalize_* evaluate it this way once
 * per launch.  Also validates the descriptor: unknown kind or schedule -> D3P_ERR_UNSUPPORTED; D3P_OPT_SCHEDULED on
 * NONE / ADADP, step < 0, decay_steps <= 0, n_boundaries > D3P_MAX_BOUNDARIES or a clip_norm that is not > 0 ->
 * D3P_ERR_INVALID_ARGUMENT. */
int32_t d3p_optim_step_size(const d3p_optim_desc* optim_h, int32_t step, float* out_h);

/* ADADP needs the global error norm before an odd step can be accepted, so an odd step is two
 * launches: d3p_perturb_finalize_f32 (kind = D3P_OPT_ADADP, odd `step`) stores the tentative
 * x - lr/2 * g in params_d and per-CTA partial sums of ((x_stepped - x_new) / max(1, x_stepped))^2
 * in err_ws_d; d3p_adadp_finish_f32 then adds them in a fixed order, sets
 * lr *= min(max(sqrt(tol / err), 0.9), 1.1) and, if stability_check and err > tol, restores
 * params_d = x_prev_d (d3p/optimizers.py:72-99).  Even steps need only the first launch. */
size_t d3p_adadp_workspace_floats(uint32_t P);
int32_t d3p_adadp_finish_f32(const d3p_optim_desc* optim_h, uint32_t P, float* params_d, const float* x_prev_d,
                             void* stream);

/* ------------------------------------------------------------------------------------------
 * Whole-epoch driver (SURVEY.md section 8 row f2) — the `lax.fori_loop(0, num_batches, body)` of
 * examples/logistic_regression.py:149-160 with body = get_batch(i, batchifier_state) followed by
 * DPSVI.update (d3p/minibatch.py:103-131,217-237 + d3p/svi.py:395-434), for the mean-field
 * families.  Queues n_steps steps on `stream` without synchronising; the interpreter is not
 * involved between launches.  Same kernels and key derivations as the step-by-step calls, so the
 * trajectory is bit-identical to them.
 * ------------------------------------------------------------------------------------------ */
#define D3P_SAMPLER_POISSON 0   /* poisson_batchify_data: q, batch = max_batch_size, suppress */
#define D3P_SAMPLER_SUBSAMPLE 1 /* subsample_batchify_data(with_replacement=False): batch     */
#define D3P_SAMPLER_SPLIT 2     /* split_batchify_data (d3p/minibatch.py:242-312): step i takes records
                                   perm_d[i * batch, (i + 1) * batch) of the epoch's shuffle; no sampler kernel, the batch
                                   key is unused */
#define D3P_SAMPLER_SUBSAMPLE_REPLACE 3 /* subsample_batchify_data(with_replacement=True): batch indices drawn with
                                           d3p_chacha_randint(fold_in(batch_key, i), 32, 0, n_records) */

typedef struct {
  int32_t kind;          /* D3P_SAMPLER_*                                            */
  float q;               /* Poisson selection probability                            */
  uint32_t n_records;    /* N                                                        */
  uint32_t batch;        /* structural batch size B (Poisson: max_batch_size)        */
  int32_t suppress;      /* Poisson: handle_oversized_batch == 'suppress'            */
  const int32_t* perm_d; /* SPLIT: the state `init` returned = shuffled record indices [n_records] (device) */
} d3p_sampler_desc;

size_t d3p_dpsvi_epoch_workspace_bytes(const d3p_meanfield_desc* desc, const d3p_sampler_desc* sampler);
/* The epoch drivers run the index sampler of step i + 1 on a forked stream beside step i (and the VAE step forks its
 * independent GEMMs).  Those streams and their events live in a caller-owned context, created once per device on the
 * current device: creating a stream costs tens of microseconds, which a caller running many short epochs should not pay
 * per call.  Every d3p_dpsvi_run_epoch_* takes `ctx`; NULL = make a temporary one for this call.  One context serves
 * one epoch call at a time. */
int32_t d3p_epoch_ctx_create(d3p_epoch_ctx** ctx_out);
int32_t d3p_epoch_ctx_destroy(d3p_epoch_ctx* ctx); /* returns at once; resources go when the queued work has drained */
/* batch_key_h: the batchifier state (the key `init` returned); step i uses fold_in(batch_key, i),
 * i = first_step .. first_step + n_steps - 1.  rng_key_io_h: DPSVIState.rng_key, advanced in place.
 * leaves_h: leaf offsets / lengths (site states are derived per step).  optim_io_h->step is advanced.
 * params_d / m_d / v_d (and optim->lr_d for ADADP) are updated in place.  With `comm` (below) the
 * batch positions are split contiguously over the ranks and the sums meet over NVLink peer memory.
 * stats_out_d (may be NULL): [n_steps, 3] = { loss, n, f } of every step. */
int32_t d3p_dpsvi_run_epoch_meanfield(const d3p_meanfield_desc* desc, const d3p_sampler_desc* sampler,
                                      const float* x_d, size_t x_row_stride, const int32_t* y_d,
                                      const uint32_t batch_key_h[16], uint32_t rng_key_io_h[16],
                                      uint32_t first_step, uint32_t n_steps, float obs_scale, float C,
                                      float dp_scale, const d3p_leaf_table* leaves_h, d3p_optim_desc* optim_io_h,
                                      float* params_d, float* m_d, float* v_d, float* stats_out_d,
                                      d3p_comm* comm /* NULL = single GPU */, void* ws_d, size_t ws_bytes,
                                      d3p_epoch_ctx* ctx /* NULL = temporary */, void* stream);

/* partials_d is [n_partials, P + 2] (grad sum | loss sum | count).  With n = total count,
 * f = (n == 0 ? 0 : B / n):
 *   grad = ((sum / B) + dp_scale * (C / n) * xi) * obs_scale * f     (d3p/svi.py:342-375)
 *   loss = (loss_sum / B) * f                                          (d3p/svi.py:306,342)
 * xi ~ N(0, 1) from the ChaCha stream of the leaf's site state (counter from 0).
 * grad_out_d[P] (may be NULL) receives grad; if optim->kind != NONE, params_d / m_d / v_d are
 * updated in place (d3p/svi.py:379-393 with numpyro.optim.SGD / Adam / Momentum / Adagrad / RMSProp /
 * RMSPropMomentum / ClippedAdam or d3p's ADADP; m_d holds the first-moment / velocity / momentum state, v_d the
 * squared-gradient state, and a kind that keeps one of them needs its pointer).
 * stats_d[3] (may be NULL) = { loss, n, f }.
 * nf_override_h (may be NULL) = { n, f } supplied by the caller instead of the counts in the
 * partials — the stage-method form DPSVI._perturb_and_reassemble_gradients(state, key,
 * avg_clipped_grads, num_elements, batch_mask_scaling_factor) (d3p/svi.py:350-377), called with
 * partials = the averaged gradients, n_partials = 1, B = 1. */
int32_t d3p_perturb_finalize_f32(const float* partials_d, uint32_t n_partials, uint32_t P, uint32_t B,
                                 const d3p_leaf_table* leaves_h, float dp_scale, float C, float obs_scale,
                                 int32_t add_noise, float* grad_out_d, const d3p_optim_desc* optim_h,
                                 float* params_d, float* m_d, float* v_d, float* stats_d,
                                 const float* nf_override_h, void* stream);

/* ------------------------------------------------------------------------------------------
 * Sharded minibatch over the GPUs of one box (SURVEY.md section 8e) without NCCL in the step:
 * every rank owns a peer-mapped window (CUDA IPC over NVLink / NVSwitch) and the finalize kernel
 * itself exchanges the P + 2 clipped sums: each value is pushed into every peer's window as one
 * 8-byte word {value, epoch}; the reader polls its own memory for the current epoch's tag and adds
 * the G copies in rank order, so every replica computes bit-identical sums, noise and parameters.
 *   create  : allocate this rank's window (max_records > 0 also provisions the sharded Poisson
 *             sampler for data sets of up to that many records), return its 64-byte IPC handle
 *   connect : map the windows of all ranks (handles_h = world x 64 bytes, gathered by the caller,
 *             e.g. torch.distributed.all_gather_object)
 * All ranks must issue the same sequence of d3p_perturb_finalize_p2p_f32 /
 * d3p_poisson_sample_sharded calls.  A peer that never shows up makes the waiting kernel give up
 * after the time-out (default 10 s, d3p_comm_set_timeout_ms) instead of hanging the GPU.  A slot whose
 * tag never matched is never consumed: the kernel yields NaN for it, which poisons that step's
 * gradient, parameters and loss (and, through the next exchange, every replica), and the error is
 * STICKY: the time-out is counted in a host-mapped word, and every later call that takes the window
 * (d3p_perturb_finalize_p2p_f32, d3p_poisson_sample_sharded, d3p_dpsvi_run_epoch_*) returns
 * D3P_ERR_PEER_TIMEOUT.  d3p_comm_timeouts reads that word without synchronising the device (it
 * covers the work that has completed; synchronise the stream first for a definitive answer).
 * ------------------------------------------------------------------------------------------ */
int32_t d3p_comm_create(int32_t rank, int32_t world, uint32_t max_params, uint32_t max_records /* 0: no sharded
                        sampler */, d3p_comm** comm_out, uint8_t handle_out_h[64]);
int32_t d3p_comm_connect(d3p_comm* comm, const uint8_t* handles_h);
/* Same-process peers instead of CUDA IPC (one process driving several GPUs with peer access enabled, or
 * several logical ranks on one device, each on its own stream): windows_h[r] = d3p_comm_window of rank r. */
int32_t d3p_comm_window(d3p_comm* comm, void** window_out_h, size_t* bytes_out_h);
int32_t d3p_comm_connect_local(d3p_comm* comm, void* const* windows_h);
int32_t d3p_comm_timeouts(d3p_comm* comm, uint32_t* count_out_h);
int32_t d3p_comm_timeout_detail(d3p_comm* comm, uint32_t out_h[4]); /* [0] all, [1] clipped-sum exchange, [2] sampler counts */
int32_t d3p_comm_set_timeout_ms(d3p_comm* comm, uint32_t timeout_ms);
/* sharded sampler: tiles (4096 records) drawn redundantly on each side of a rank's slice (default 16; same on all ranks) */
int32_t d3p_comm_set_sampler_margin(d3p_comm* comm, uint32_t tiles);
int32_t d3p_comm_destroy(d3p_comm* comm);
/* d3p_poisson_sample with the selector draw (the expensive part: N / 16 ChaCha blocks) split over the
 * ranks: rank r draws its slice of the records, publishes 16-bit selection masks and per-tile counts in
 * its window, every rank scans all counts and compacts only the positions [pos_begin, pos_end) it owns.
 * counts_d / mask_d are complete on every rank; idx_d[p] is written for pos_begin <= p < min(pos_end,
 * counts_d[1]) only.  Bit-identical to d3p_poisson_sample on those positions. */
int32_t d3p_poisson_sample_sharded(d3p_comm* comm, const uint32_t state_h[16], float q, uint32_t n_records,
                                   uint32_t max_b, int32_t suppress, uint32_t pos_begin, uint32_t pos_end,
                                   int32_t* idx_d, int32_t* counts_d, uint8_t* mask_d, void* ws_d,
                                   size_t ws_bytes, void* stream);
/* d3p_perturb_finalize_f32 on this rank's partial rows + the peers' (comm may be NULL = local only). */
int32_t d3p_perturb_finalize_p2p_f32(const float* partials_d, uint32_t n_partials, uint32_t P, uint32_t B,
                                     const d3p_leaf_table* leaves_h, float dp_scale, float C, float obs_scale,
                                     int32_t add_noise, float* grad_out_d, const d3p_optim_desc* optim_h,
                                     float* params_d, float* m_d, float* v_d, float* stats_d,
                                     const float* nf_override_h, d3p_comm* comm, void* stream);

/* Multi-GPU (new; the reference is single-device): out_d[P + 2] = sum over the n_partials rows of
 * a step workspace, in a fixed order.  The caller all-reduces out_d over the ranks that share a
 * batch (ncclAllReduce, sum) and passes it to d3p_perturb_finalize_f32 with n_partials = 1; every
 * rank then draws the SAME noise from the replicated ChaCha state, so the mechanism is unchanged. */
int32_t d3p_reduce_partials_f32(const float* partials_d, uint32_t n_partials, uint32_t P, float* out_d,
                                void* stream);

/* ------------------------------------------------------------------------------------------
 * Tensor-core building blocks of the dense-layer (VAE) path — new; the reference leaves dense layers
 * to XLA's cuBLAS calls (examples/vae.py:80-103) and clips materialised [B, P] gradients
 * (d3p/svi.py:310-348).
 * ------------------------------------------------------------------------------------------ */

/* hi[i] = tf32_truncate(x[i] * s), lo[i] = x[i] * s - hi[i], s = row_scale_d ? row_scale_d[i / cols] : 1.
 * lo_d may be NULL. */
int32_t d3p_split_tf32(const float* x_d, const float* row_scale_d, uint32_t cols, float* hi_d, float* lo_d, size_t n,
                       void* stream);

/* out[split][m, n] = sum over the split's k range of A[m, k] * B[n, k] in 3xTF32 (fp32 accuracy) on
 * tcgen05 tensor cores fed by TMA.  A = a_hi + a_lo, B = b_hi + b_lo (d3p_split_tf32); a lo pointer
 * may be NULL when the operand is exact in TF32.  *_mn_major = 0: operand stored [M or N, K] with the
 * contraction index contiguous; 1: stored [K, M or N] (the clipped-sum case A^T diag(c) Delta, where
 * the contraction runs over the batch).  lda / ldb / ldc are row strides in floats (multiples of 4,
 * 16-byte aligned bases).  tile_n is 128 or 224.  The split_k partial results are written
 * split_stride floats apart (the caller reduces them in a fixed order); transpose_out stores
 * out[n * ldc + m]. */
int32_t d3p_gemm_tf32x3(const float* a_hi_d, const float* a_lo_d, int32_t a_mn_major, size_t lda, const float* b_hi_d,
                        const float* b_lo_d, int32_t b_mn_major, size_t ldb, uint32_t M, uint32_t N, uint32_t K,
                        uint32_t split_k, int32_t tile_n, float* out_d, size_t ldc, size_t split_stride,
                        int32_t transpose_out, void* stream);
/* The same product from UNSPLIT fp32 operands: every shared-memory stage is split into hi / lo by the kernel's
 * epilogue warps while the previous stages are being multiplied, which halves the operand bytes read per tile. */
int32_t d3p_gemm_f32x3(const float* a_d, int32_t a_mn_major, size_t lda, const float* b_d, int32_t b_mn_major, size_t ldb,
                       uint32_t M, uint32_t N, uint32_t K, uint32_t split_k, int32_t tile_n, float* out_d, size_t ldc,
                       size_t split_stride, int32_t transpose_out, void* stream);


/* ------------------------------------------------------------------------------------------
 * Fused per-example gradient + ghost-norm clip + clipped sum for the VAE of examples/vae.py:65-153
 * (encoder Dense(D->H) softplus -> {Dense(H->Z), exp(Dense(H->Z))}; decoder Dense(Z->H) softplus ->
 * Dense(H->D) sigmoid; Bernoulli(probs) likelihood; Normal(0, I) prior) — replaces d3p/svi.py:238-348.
 * Flat parameter vector = jax pytree order of {'decoder$params', 'encoder$params'}:
 * W4 [Z,H], b4 [H], W5 [H,D], b5 [D], W1 [D,H], b1 [H], W2 [H,Z], b2 [Z], W3 [H,Z], b3 [Z].
 * ------------------------------------------------------------------------------------------ */
typedef struct {
  uint32_t out_dim, hidden_dim, z_dim; /* D, H (multiples of 4; H <= 3156 on B200), 1 <= Z <= 32 */
  uint32_t n_params;
  uint32_t off_w4, off_b4, off_w5, off_b5, off_w1, off_b1, off_w2, off_b2, off_w3, off_b3;
  float site_scale; /* plate scale N / 1 times the scale handler's 1 / N (examples/vae.py:193-194) */
} d3p_vae_desc;

/* Workspace for batch_rows = pos_end - pos_begin examples; *n_partials_out = S, the number of partial
 * rows [S, P + 2] at the START of the workspace (input of d3p_perturb_finalize_f32). */
size_t d3p_vae_workspace_bytes(const d3p_vae_desc* desc, uint32_t batch_rows, uint32_t* n_partials_out);

/* Same contract as d3p_dpsvi_step_meanfield: x_d rows are [D] floats (x_row_stride floats apart), read
 * through idx_d when given; positions [pos_begin, pos_end) of a batch of B; per-example Threefry keys by
 * position.  ws_d must be 256-byte aligned.  px_norms_d[B] / px_loss_d[B] (may be NULL) receive the
 * pre-clip gradient norms and obs_scale * loss_p.  profile_events_h (may be NULL) = two events
 * (d3p_event_create) recorded immediately before and after the two tcgen05 clipped-sum GEMMs.
 * ctx (may be NULL): caller-owned side streams on which the four independent clipped-sum GEMMs and the small
 * preparation kernels run concurrently (forked from / joined to `stream`); NULL runs everything on `stream`.
 * One context serves one caller at a time (one per DPSVI object / per stream). */
int32_t d3p_vae_ctx_create(d3p_vae_ctx** ctx_out);
int32_t d3p_vae_ctx_destroy(d3p_vae_ctx* ctx); /* returns at once; resources go when the queued work has drained */
int32_t d3p_dpsvi_step_vae(const d3p_vae_desc* desc, const float* params_d, const float* x_d, size_t x_row_stride,
                           const int32_t* idx_d, const uint8_t* mask_d, const int32_t* num_valid_d, uint32_t B,
                           uint32_t pos_begin, uint32_t pos_end, const uint32_t threefry_key_h[2], float obs_scale,
                           float C, float* px_norms_d, float* px_loss_d, void* ws_d, size_t ws_bytes,
                           void* const* profile_events_h, d3p_vae_ctx* ctx, void* stream);

/* The same loop for the VAE family (examples/vae.py:216-233: lax.fori_loop over get_batch -> update for one epoch;
 * d3p/svi.py:395-434 per step).  `world` = number of ranks sharing the batch (1 without `comm`); ws_d must be
 * 256-byte aligned. */
size_t d3p_dpsvi_epoch_vae_workspace_bytes(const d3p_vae_desc* desc, const d3p_sampler_desc* sampler, int32_t world);
int32_t d3p_dpsvi_run_epoch_vae(const d3p_vae_desc* desc, const d3p_sampler_desc* sampler, const float* x_d,
                                size_t x_row_stride, const uint32_t batch_key_h[16], uint32_t rng_key_io_h[16],
                                uint32_t first_step, uint32_t n_steps, float obs_scale, float C, float dp_scale,
                                const d3p_leaf_table* leaves_h, d3p_optim_desc* optim_io_h, float* params_d,
                                float* m_d, float* v_d, float* stats_out_d, d3p_comm* comm /* NULL = single GPU */,
                                void* ws_d, size_t ws_bytes, d3p_epoch_ctx* ctx, void* stream);


/* ------------------------------------------------------------------------------------------
 * Fused per-example gradient + clip + sum for the Gaussian mixture model of
 * examples/gaussian_mixture_model.py:51-85 with the d3p.gmm.GaussianMixture likelihood
 * (d3p/gmm.py:71-86) — replaces d3p/svi.py:238-348.  Guide: pis ~ Dirichlet(exp(alpha_log)),
 * mus ~ Normal(mus_loc, 1), sigs ~ InverseGamma(1, 1), all drawn per example.
 * Flat parameter vector (pytree order): alpha_log [K], mus_loc [K, d].
 * ------------------------------------------------------------------------------------------ */
typedef struct {
  uint32_t K, d;        /* components, data columns */
  uint32_t n_params;    /* K + K * d */
  uint32_t alpha_off, mus_off;
  float num_obs_total;  /* plate size N */
} d3p_gmm_desc;

size_t d3p_gmm_workspace_bytes(const d3p_gmm_desc* desc, uint32_t* n_partials_out);

/* Same contract as d3p_dpsvi_step_meanfield (partial rows [n_partials, P + 2] at the start of ws_d). */
int32_t d3p_dpsvi_step_gmm(const d3p_gmm_desc* desc, const float* params_d, const float* x_d, size_t x_row_stride,
                           const int32_t* idx_d, const uint8_t* mask_d, const int32_t* num_valid_d, uint32_t B,
                           uint32_t pos_begin, uint32_t pos_end, const uint32_t threefry_key_h[2], float obs_scale,
                           float C, float* px_norms_d, float* px_grads_d, float* px_loss_d, void* ws_d, size_t ws_bytes,
                           void* stream);

/* d3p.gmm.GaussianMixture.log_prob (d3p/gmm.py:71-86) for a batch of rows: out[b] = logsumexp_k(log pis[k] +
 * sum_e log N(x[b, e]; locs[k, e], scales[k, e])); locs / scales are [K, E] (event dimensions flattened), pis [K]. */
int32_t d3p_gmm_log_prob_f32(const float* x_d, size_t x_row_stride, const float* locs_d, const float* scales_d,
                             const float* pis_d, uint32_t B, uint32_t K, uint32_t E, float* out_d, void* stream);

/* The same loop for the mixture model (examples/gaussian_mixture_model.py:205-218). */
size_t d3p_dpsvi_epoch_gmm_workspace_bytes(const d3p_gmm_desc* desc, const d3p_sampler_desc* sampler);
int32_t d3p_dpsvi_run_epoch_gmm(const d3p_gmm_desc* desc, const d3p_sampler_desc* sampler, const float* x_d,
                                size_t x_row_stride, const uint32_t batch_key_h[16], uint32_t rng_key_io_h[16],
                                uint32_t first_step, uint32_t n_steps, float obs_scale, float C, float dp_scale,
                                const d3p_leaf_table* leaves_h, d3p_optim_desc* optim_io_h, float* params_d,
                                float* m_d, float* v_d, float* stats_out_d, d3p_comm* comm /* NULL = single GPU */,
                                void* ws_d, size_t ws_bytes, d3p_epoch_ctx* ctx, void* stream);


/* ------------------------------------------------------------------------------------------
 * DPSVI.evaluate (d3p/svi.py:436-449 -> numpyro SVI.evaluate) for the mean-field families: the
 * non-private loss -(log p(theta) + (N / B) sum_i log p(x_i | theta) - log q(theta)) of a whole batch
 * with one guide sample drawn from threefry_key_h (= jax.random.split(jax_key)[1]).  loss_d[1].
 * ------------------------------------------------------------------------------------------ */
size_t d3p_elbo_evaluate_workspace_bytes(void);
int32_t d3p_elbo_evaluate_meanfield(const d3p_meanfield_desc* desc, const float* params_d, const float* x_d,
                                    size_t x_row_stride, const int32_t* y_d, const int32_t* idx_d, uint32_t B,
                                    const uint32_t threefry_key_h[2], float* loss_d, void* ws_d, size_t ws_bytes,
                                    void* stream);
/* The same for the VAE (examples/vae.py:236-247 evaluates the test loss every epoch): the forward half of the step on
 * the whole batch with ONE guide draw z [B, Z]; scale (N / B) * (1 / N).  Workspace: d3p_vae_workspace_bytes(desc, B). */
int32_t d3p_elbo_evaluate_vae(const d3p_vae_desc* desc, const float* params_d, const float* x_d, size_t x_row_stride,
                              const int32_t* idx_d, uint32_t B, const uint32_t threefry_key_h[2], float* loss_d,
                              void* ws_d, size_t ws_bytes, d3p_vae_ctx* ctx, void* stream);
/* ... and for the mixture: one guide draw (pis, mus, sigs), then the log-likelihood of every example under it. */
size_t d3p_elbo_evaluate_gmm_workspace_bytes(const d3p_gmm_desc* desc);
int32_t d3p_elbo_evaluate_gmm(const d3p_gmm_desc* desc, const float* params_d, const float* x_d, size_t x_row_stride,
                              const int32_t* idx_d, uint32_t B, const uint32_t threefry_key_h[2], float* loss_d,
                              void* ws_d, size_t ws_bytes, void* stream);

/* ------------------------------------------------------------------------------------------
 * jax.random with Threefry keys (2 words) on the device, for predictive sampling (d3p/modelling.py:39-223 runs numpyro
 * models under the `seed` handler, whose sites draw jax.random.normal / bernoulli / gamma ...): jax's legacy layout,
 * n variates from ceil(n / 2) Threefry-2x32-20 calls; gamma / loggamma with per-element keys split(key, n)
 * (alpha_n = 1: one shared concentration, else alpha_n = n).
 * ------------------------------------------------------------------------------------------ */
int32_t d3p_threefry_random_bits(const uint32_t key_h[2], uint32_t* out_d, size_t n_words, void* stream);
int32_t d3p_threefry_uniform_f32(const uint32_t key_h[2], float lo, float hi, float* out_d, size_t n, void* stream);
int32_t d3p_threefry_normal_f32(const uint32_t key_h[2], float* out_d, size_t n, void* stream);
int32_t d3p_threefry_gamma_f32(const uint32_t key_h[2], const float* alpha_d, uint32_t alpha_n, uint32_t n,
                               int32_t log_space, float* out_d, void* stream);

/* ------------------------------------------------------------------------------------------
 * Device-key forms (*_dk).  The reference runs get_batch + update as the body of a jitted lax.fori_loop with TRACED
 * keys (examples/logistic_regression.py:149-160; README.md:119-126; d3p/random/__init__.py:28-32): a key there is a
 * device value that no host code ever sees.  Every entry point above that takes a key as HOST words has a twin that
 * takes it as a DEVICE pointer (16 uint32 ChaCha state words, or 2 Threefry words), and the key plumbing itself
 * (split / fold_in / convert_to_jax_rng_key, the per-step keys of DPSVI.update) runs as one-block kernels on the
 * stream, so an XLA custom call bound to these needs no host synchronisation.  Same kernels, bit-identical results
 * (tests/test_gpu_device_keys.py).
 * ------------------------------------------------------------------------------------------ */
/* rng_suite.split (d3p/random/__init__.py:29): out_d = num x 16 words. */
int32_t d3p_chacha_split_dk(const uint32_t* in_d, int32_t num, uint32_t* out_d, void* stream);
/* rng_suite.fold_in(key, *data_d + data_imm) (d3p/random/__init__.py:30); data_d may be NULL (a loop index that
 * lives on the device, e.g. the `i` of fori_loop, or an immediate). */
int32_t d3p_chacha_fold_in_dk(const uint32_t* in_d, const uint32_t* data_d, uint32_t data_imm, uint32_t* out_d,
                              void* stream);
/* rng_suite.random_bits / uniform / normal with the key in device memory; random_bits with n_words = 2 is
 * convert_to_jax_rng_key (d3p/random/__init__.py:149-155). */
int32_t d3p_chacha_random_bits_dk(const uint32_t* state_d, uint64_t first_block, uint32_t* out_d, size_t n_words,
                                  void* stream);
int32_t d3p_chacha_uniform_f32_dk(const uint32_t* state_d, uint64_t first_block, float lo, float hi, float* out_d,
                                  size_t n, void* stream);
int32_t d3p_chacha_normal_f32_dk(const uint32_t* state_d, uint64_t first_block, float* out_d, size_t n, void* stream);
/* d3p_chacha_randint with the key in device memory. */
int32_t d3p_chacha_randint_dk(const uint32_t* key_d, uint32_t nbits, int64_t minval, int64_t maxval, void* out_d,
                              size_t n, void* stream);
/* The keys of one DPSVI.update (d3p/svi.py:208-211,413-414,490-491) from the state key, which is advanced in place:
 * (carry, k_grad, k_noise) = split(key, 3); key := carry; threefry_key_out_d[2] = convert_to_jax_rng_key(k_grad);
 * site_states_out_d[n_leaves][16] = split(k_noise, n_leaves). */
int32_t d3p_dpsvi_keys_dk(uint32_t* rng_key_io_d, uint32_t n_leaves, uint32_t* threefry_key_out_d,
                          uint32_t* site_states_out_d, void* stream);
/* d3p_autodiag_draw_f32 with the Threefry key (2 words) in device memory. */
int32_t d3p_autodiag_draw_f32_dk(const d3p_autodiag_desc* desc, const float* params_d,
                                 const uint32_t* threefry_key_d, uint32_t B, uint32_t pos_begin, uint32_t pos_end,
                                 float* theta_d, float* eps_d, size_t ld, void* stream);
/* Samplers.  rc_out_d / rc_d: 30 words (32 allocated is fine). */
int32_t d3p_feistel_round_constants_dk(const uint32_t* state_d, uint32_t* rc_out_d, void* stream);
int32_t d3p_feistel_sample_dk(const uint32_t* rc_d, uint32_t capacity, uint32_t first_pos, uint32_t n, int32_t* idx_d,
                              void* stream);
int32_t d3p_poisson_sample_dk(const uint32_t* state_d, float q, uint32_t n_records, uint32_t max_b, int32_t suppress,
                              int32_t* idx_d, int32_t* counts_d, uint8_t* mask_d, void* ws_d, size_t ws_bytes,
                              void* stream);
int32_t d3p_poisson_sample_sharded_dk(d3p_comm* comm, const uint32_t* state_d, float q, uint32_t n_records,
                                      uint32_t max_b, int32_t suppress, uint32_t pos_begin, uint32_t pos_end,
                                      int32_t* idx_d, int32_t* counts_d, uint8_t* mask_d, void* ws_d, size_t ws_bytes,
                                      void* stream);
/* Fused steps with the Threefry key (2 words) in device memory. */
int32_t d3p_dpsvi_step_meanfield_dk(const d3p_meanfield_desc* desc, const float* params_d, const float* x_d,
                                    size_t x_row_stride, const int32_t* y_d, const int32_t* idx_d,
                                    const uint8_t* mask_d, const int32_t* num_valid_d, uint32_t B,
                                    uint32_t pos_begin, uint32_t pos_end, const uint32_t* threefry_key_d,
                                    float obs_scale, float C, float* px_norms_d, float* px_grads_d, float* px_loss_d,
                                    void* ws_d, size_t ws_bytes, void* stream);
int32_t d3p_dpsvi_step_vae_dk(const d3p_vae_desc* desc, const float* params_d, const float* x_d, size_t x_row_stride,
                              const int32_t* idx_d, const uint8_t* mask_d, const int32_t* num_valid_d, uint32_t B,
                              uint32_t pos_begin, uint32_t pos_end, const uint32_t* threefry_key_d, float obs_scale,
                              float C, float* px_norms_d, float* px_loss_d, void* ws_d, size_t ws_bytes,
                              void* const* profile_events_h, d3p_vae_ctx* ctx, void* stream);
int32_t d3p_dpsvi_step_gmm_dk(const d3p_gmm_desc* desc, const float* params_d, const float* x_d, size_t x_row_stride,
                              const int32_t* idx_d, const uint8_t* mask_d, const int32_t* num_valid_d, uint32_t B,
                              uint32_t pos_begin, uint32_t pos_end, const uint32_t* threefry_key_d, float obs_scale,
                              float C, float* px_norms_d, float* px_grads_d, float* px_loss_d, void* ws_d,
                              size_t ws_bytes, void* stream);
/* d3p_perturb_finalize_p2p_f32 with the per-leaf noise keys in device memory (leaves_h: layout only). */
int32_t d3p_perturb_finalize_dk_f32(const float* partials_d, uint32_t n_partials, uint32_t P, uint32_t B,
                                    const d3p_leaf_table* leaves_h, const uint32_t* site_states_d, float dp_scale, float C,
                                    float obs_scale, float* grad_out_d, const d3p_optim_desc* optim_h, float* params_d,
                                    float* m_d, float* v_d, float* stats_d, d3p_comm* comm, void* stream);
/* The epoch loops with the batchifier key and the DPSVI state key in device memory (rng_key_io_d advanced in place). */
int32_t d3p_dpsvi_run_epoch_meanfield_dk(const d3p_meanfield_desc* desc, const d3p_sampler_desc* sampler,
                                         const float* x_d, size_t x_row_stride, const int32_t* y_d,
                                         const uint32_t* batch_key_d, uint32_t* rng_key_io_d, uint32_t first_step,
                                         uint32_t n_steps, float obs_scale, float C, float dp_scale,
                                         const d3p_leaf_table* leaves_h, d3p_optim_desc* optim_io_h, float* params_d,
                                         float* m_d, float* v_d, float* stats_out_d, d3p_comm* comm, void* ws_d,
                                         size_t ws_bytes, d3p_epoch_ctx* ctx, void* stream);
int32_t d3p_dpsvi_run_epoch_vae_dk(const d3p_vae_desc* desc, const d3p_sampler_desc* sampler, const float* x_d,
                                   size_t x_row_stride, const uint32_t* batch_key_d, uint32_t* rng_key_io_d,
                                   uint32_t first_step, uint32_t n_steps, float obs_scale, float C, float dp_scale,
                                   const d3p_leaf_table* leaves_h, d3p_optim_desc* optim_io_h, float* params_d,
                                   float* m_d, float* v_d, float* stats_out_d, d3p_comm* comm, void* ws_d,
                                   size_t ws_bytes, d3p_epoch_ctx* ctx, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* D3P_B200_H_ */
