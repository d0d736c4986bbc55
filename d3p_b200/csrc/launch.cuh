// Host-side launch helpers shared by the translation units of libd3p_b200.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/d3p_b200.h"

namespace d3p {

// Number of SMs of the current device (148 on B200); cached per device id.
inline int sm_count() {
  static int cached[64] = {0};
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return 148;
  if (cached[dev] == 0) {
    int n = 0;
    if (cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || n <= 0) n = 148;
    cached[dev] = n;
  }
  return cached[dev];
}

inline int32_t check_launch() { return cudaGetLastError() == cudaSuccess ? D3P_OK : D3P_ERR_CUDA; }

inline size_t align_up(size_t x, size_t a) { return (x + a - 1) / a * a; }

// Bodies of the public entry points that come as a host-key / device-key pair (d3p_x and d3p_x_dk): each takes its key
// as a (key_h, key_d) pair of which one is non-null, so a caller that serves both key modes (the epoch drivers) makes
// one call.  Arguments as in include/d3p_b200.h.
int32_t step_meanfield_impl(const d3p_meanfield_desc* desc, const float* params_d, const float* x_d, size_t x_row_stride,
                            const int32_t* y_d, const int32_t* idx_d, const uint8_t* mask_d, const int32_t* num_valid_d,
                            uint32_t B, uint32_t pos_begin, uint32_t pos_end, const uint32_t* threefry_key_h,
                            const uint32_t* threefry_key_d, float obs_scale, float C, float* px_norms_d,
                            float* px_grads_d, float* px_loss_d, void* ws_d, size_t ws_bytes, void* stream);
int32_t step_gmm_impl(const d3p_gmm_desc* desc, const float* params_d, const float* x_d, size_t x_row_stride,
                      const int32_t* idx_d, const uint8_t* mask_d, const int32_t* num_valid_d, uint32_t B,
                      uint32_t pos_begin, uint32_t pos_end, const uint32_t* threefry_key_h, const uint32_t* threefry_key_d,
                      float obs_scale, float C, float* px_norms_d, float* px_grads_d, float* px_loss_d, void* ws_d,
                      size_t ws_bytes, void* stream);
// eval_loss_d != nullptr: the forward half only, writing the evaluation loss (d3p_elbo_evaluate_vae)
int32_t step_vae_impl(const d3p_vae_desc* desc, const float* params_d, const float* x_d, size_t x_row_stride,
                      const int32_t* idx_d, const uint8_t* mask_d, const int32_t* num_valid_d, uint32_t B,
                      uint32_t pos_begin, uint32_t pos_end, const uint32_t* threefry_key_h, const uint32_t* threefry_key_d,
                      float obs_scale, float C, float* px_norms_d, float* px_loss_d, void* ws_d, size_t ws_bytes,
                      void* const* profile_events_h, d3p_vae_ctx* ctx, void* stream, float* eval_loss_d = nullptr);
int32_t feistel_sample_impl(const uint32_t* rc_h, const uint32_t* rc_d, uint32_t capacity, uint32_t first_pos, uint32_t n,
                            int32_t* idx_d, void* stream);
int32_t poisson_sample_impl(const uint32_t* state_h, const uint32_t* state_d, float q, uint32_t n_records, uint32_t max_b,
                            int32_t suppress, int32_t* idx_d, int32_t* counts_d, uint8_t* mask_d, void* ws_d,
                            size_t ws_bytes, void* stream);
int32_t poisson_sample_sharded_impl(d3p_comm* comm, const uint32_t* state_h, const uint32_t* state_d, float q,
                                    uint32_t n_records, uint32_t max_b, int32_t suppress, uint32_t pos_begin,
                                    uint32_t pos_end, int32_t* idx_d, int32_t* counts_d, uint8_t* mask_d, void* ws_d,
                                    size_t ws_bytes, void* stream);
// site_states_d == nullptr: the per-leaf ChaCha states are the site_state words of leaves_h
int32_t perturb_finalize_impl(const float* partials_d, uint32_t n_partials, uint32_t P, uint32_t B,
                              const d3p_leaf_table* leaves_h, const uint32_t* site_states_d, float dp_scale, float C,
                              float obs_scale, int32_t add_noise, float* grad_out_d, const d3p_optim_desc* optim_h,
                              float* params_d, float* m_d, float* v_d, float* stats_d, const float* nf_override_h,
                              d3p_comm* comm, void* stream);
// The optimizer checks of perturb_finalize_impl (descriptor as d3p_optim_step_size, plus the state buffers its kind
// needs), for callers that want to refuse a bad descriptor before they launch anything.
int32_t optim_check(const d3p_optim_desc* optim_h, const float* params_d, const float* m_d, const float* v_d);

}  // namespace d3p
