// K1: ChaCha20 keystream kernels (+ uniform / normal transforms, randint round) and the
// host-side key plumbing of the rng suite.  Replaces jax-chacha-prng behind
// d3p/random/__init__.py:28-155.
#include <math.h>

#include <type_traits>

#include "common.cuh"
#include "launch.cuh"

namespace d3p {

enum { kBits = 0, kUniform = 1, kNormal = 2 };

// One thread per 64-byte block; a warp writes 32 consecutive blocks.  Each lane owns 16
// consecutive words, stored as four 16-byte vectors (each lane writes a full 64 B line half).
template <int kMode>
__global__ void __launch_bounds__(256) chacha_stream_kernel(ChaChaArg key, uint32_t first_block, void* out,
                                                            size_t n_words, float lo, float hi) {
  ChaChaState st;
  load_chacha(key, st);
  size_t n_blocks = (n_words + 15) / 16;
  for (size_t b = (size_t)blockIdx.x * blockDim.x + threadIdx.x; b < n_blocks;
       b += (size_t)gridDim.x * blockDim.x) {
    uint32_t ks[16];
    chacha20_block(st.w, st.w[12] + first_block + (uint32_t)b, ks);
    uint32_t vals[16];
#pragma unroll
    for (int i = 0; i < 16; ++i) {
      if (kMode == kBits) vals[i] = ks[i];
      else if (kMode == kUniform) vals[i] = __float_as_uint(bits_to_uniform(ks[i], lo, hi));
      else vals[i] = __float_as_uint(bits_to_normal<false>(ks[i]));
    }
    size_t base = b * 16;
    uint32_t* o = reinterpret_cast<uint32_t*>(out);
    if (base + 16 <= n_words && ((reinterpret_cast<uintptr_t>(o) & 15) == 0)) {
      uint4* o4 = reinterpret_cast<uint4*>(o + base);
#pragma unroll
      for (int i = 0; i < 4; ++i) o4[i] = make_uint4(vals[4 * i], vals[4 * i + 1], vals[4 * i + 2], vals[4 * i + 3]);
    } else {
#pragma unroll
      for (int i = 0; i < 16; ++i)
        if (base + i < n_words) o[base + i] = vals[i];
    }
  }
}

// One rejection round of rng_suite.randint (d3p/random/__init__.py:127-142) for NBITS-wide draws: element e takes bit
// field e of the keystream (random_bits(key, NBITS, shape): the words viewed as little-endian NBITS-bit integers).
template <int NBITS>
__global__ void __launch_bounds__(256) randint_round_kernel(ChaChaArg key, uint32_t bitmask, uint32_t delta,
                                                            int first, uint32_t* vals, size_t n, int* pending) {
  constexpr int kPerWord = 32 / NBITS, kPerBlock = 16 * kPerWord;
  constexpr uint32_t kFieldMask = NBITS == 32 ? 0xFFFFFFFFu : ((1u << (NBITS & 31)) - 1u);
  ChaChaState st;
  load_chacha(key, st);
  size_t n_blocks = (n + kPerBlock - 1) / kPerBlock;
  int local = 0;
  for (size_t b = (size_t)blockIdx.x * blockDim.x + threadIdx.x; b < n_blocks;
       b += (size_t)gridDim.x * blockDim.x) {
    uint32_t ks[16];
    chacha20_block(st.w, st.w[12] + (uint32_t)b, ks);
#pragma unroll
    for (int i = 0; i < kPerBlock; ++i) {
      size_t e = b * kPerBlock + i;
      if (e < n) {
        uint32_t v = first ? 0xFFFFFFFFu : vals[e];
        if (first || v > delta) v = ((ks[i / kPerWord] >> ((i % kPerWord) * NBITS)) & kFieldMask) & bitmask;
        vals[e] = v;
        local += (v > delta);
      }
    }
  }
  local = __reduce_add_sync(0xffffffffu, local);
  if ((threadIdx.x & 31) == 0 && local) atomicAdd(pending, local);
}

// vals + minval in the arithmetic of the result type (wraps like vdtype(uvals) + minval, d3p/random/__init__.py:145)
template <typename T>
__global__ void randint_finish_kernel(const uint32_t* vals, int32_t minval, T* out, size_t n) {
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x)
    out[i] = (T)(uint32_t)(vals[i] + (uint32_t)minval);
}

// The whole rejection loop of rng_suite.randint (d3p/random/__init__.py:84-146) in one launch.  A thread owns one ChaCha
// block of outputs (kPerBlock elements) and walks the round-key chain (key, round_key) = split(key, 2) by itself,
// drawing bit field e of round_key_r's block b until every element of its block has been accepted: element e keeps the
// draw of the first round r with bits(round_key_r)[e] & bitmask <= delta, which is what the per-round loop keeps.
// There is no round cap.  Accepted fields are packed into `acc` exactly as the keystream packs them, so the block's
// 64 output bytes are written as four 16-byte vectors.
template <int NBITS>
__global__ void __launch_bounds__(256) randint_kernel(ChaChaArg key, uint32_t bitmask, uint32_t delta, uint32_t minval,
                                                      void* out, size_t n) {
  constexpr int kPerWord = 32 / NBITS, kPerBlock = 16 * kPerWord;
  constexpr uint32_t kFieldMask = NBITS == 32 ? 0xFFFFFFFFu : ((1u << (NBITS & 31)) - 1u);
  ChaChaState k0;
  load_chacha(key, k0);
  const size_t n_blocks = (n + kPerBlock - 1) / kPerBlock;
  for (size_t b = (size_t)blockIdx.x * blockDim.x + threadIdx.x; b < n_blocks;
       b += (size_t)gridDim.x * blockDim.x) {
    const size_t base = b * kPerBlock;
    const int valid = n - base < (size_t)kPerBlock ? (int)(n - base) : kPerBlock;
    using Mask = typename std::conditional<kPerBlock == 64, uint64_t, uint32_t>::type;
    // elements of this block not yet accepted (bit i = element i; kPerBlock may be narrower than Mask)
    Mask pending = valid == (int)(8 * sizeof(Mask)) ? ~(Mask)0 : (((Mask)1 << valid) - 1);
    uint32_t acc[16];
#pragma unroll
    for (int w = 0; w < 16; ++w) acc[w] = 0;
    uint32_t chain[16];
#pragma unroll
    for (int i = 0; i < 16; ++i) chain[i] = k0.w[i];
    while (pending) {
      uint32_t rk[16], next[16], ks[16];
      chacha_derive_key(chain, 1u, D3P_DERIVE_SPLIT, rk);
      chacha_derive_key(chain, 0u, D3P_DERIVE_SPLIT, next);
#pragma unroll
      for (int i = 0; i < 16; ++i) chain[i] = next[i];
      chacha20_block(rk, rk[12] + (uint32_t)b, ks);
#pragma unroll
      for (int i = 0; i < kPerBlock; ++i) {
        const int sh = (i % kPerWord) * NBITS;
        const uint32_t v = ((ks[i / kPerWord] >> sh) & kFieldMask) & bitmask;
        if (((pending >> i) & 1) && v <= delta) {
          acc[i / kPerWord] |= v << sh;
          pending &= ~((Mask)1 << i);
        }
      }
    }
    // + minval in the arithmetic of the result type (wraps like vdtype(uvals) + minval, d3p/random/__init__.py:145)
#pragma unroll
    for (int w = 0; w < 16; ++w) {
      uint32_t r = 0;
#pragma unroll
      for (int j = 0; j < kPerWord; ++j)
        r |= ((((acc[w] >> (j * NBITS)) & kFieldMask) + minval) & kFieldMask) << (j * NBITS);
      acc[w] = r;
    }
    uint8_t* o = static_cast<uint8_t*>(out) + base * (NBITS / 8);
    if (valid == kPerBlock && (reinterpret_cast<uintptr_t>(o) & 15) == 0) {
      uint4* o4 = reinterpret_cast<uint4*>(o);
#pragma unroll
      for (int i = 0; i < 4; ++i) o4[i] = make_uint4(acc[4 * i], acc[4 * i + 1], acc[4 * i + 2], acc[4 * i + 3]);
    } else {
#pragma unroll
      for (int i = 0; i < kPerBlock; ++i) {
        if (i < valid) {
          const uint32_t v = (acc[i / kPerWord] >> ((i % kPerWord) * NBITS)) & kFieldMask;
          if (NBITS == 8) o[i] = (uint8_t)v;
          else if (NBITS == 16) reinterpret_cast<uint16_t*>(o)[i] = (uint16_t)v;
          else reinterpret_cast<uint32_t*>(o)[i] = v;
        }
      }
    }
  }
}

// ---- device-resident keys (the *_dk entry points) -------------------------------------------------------------------
// The reference runs get_batch + update as the body of a jitted fori_loop with TRACED keys
// (examples/logistic_regression.py:149-160, d3p/random/__init__.py:28-32): a key there is a device value no host ever
// sees.  These one-block kernels are rng_suite.split / fold_in / convert_to_jax_rng_key and the per-step key plumbing
// of DPSVI.update (d3p/svi.py:208-211,413-414,490-491) on such keys.
__global__ void chacha_split_dk_kernel(const uint32_t* __restrict__ in, uint32_t num, uint32_t* __restrict__ out) {
  uint32_t parent[16];
#pragma unroll
  for (int i = 0; i < 16; ++i) parent[i] = in[i];
  for (uint32_t k = blockIdx.x * blockDim.x + threadIdx.x; k < num; k += gridDim.x * blockDim.x) {
    uint32_t child[16];
    chacha_derive_key(parent, k, D3P_DERIVE_SPLIT, child);
#pragma unroll
    for (int i = 0; i < 16; ++i) out[16 * (size_t)k + i] = child[i];
  }
}

__global__ void chacha_fold_in_dk_kernel(const uint32_t* __restrict__ in, const uint32_t* __restrict__ data_d,
                                         uint32_t data_imm, uint32_t* __restrict__ out) {
  if (threadIdx.x != 0 || blockIdx.x != 0) return;
  uint32_t parent[16], child[16];
#pragma unroll
  for (int i = 0; i < 16; ++i) parent[i] = in[i];
  chacha_derive_key(parent, (data_d ? *data_d : 0u) + data_imm, D3P_DERIVE_FOLD_IN, child);
#pragma unroll
  for (int i = 0; i < 16; ++i) out[i] = child[i];
}

// One DPSVI.update worth of keys from the state key, in place: (carry, k_grad, k_noise) = split(key, 3); key := carry;
// tf_key_out = convert_to_jax_rng_key(k_grad) = its first two keystream words; site_out = split(k_noise, n_leaves).
__global__ void dpsvi_keys_dk_kernel(uint32_t* __restrict__ key_io, uint32_t n_leaves, uint32_t* __restrict__ tf_key_out,
                                     uint32_t* __restrict__ site_out) {
  __shared__ uint32_t s_noise[16];
  uint32_t parent[16];
#pragma unroll
  for (int i = 0; i < 16; ++i) parent[i] = key_io[i];
  __syncthreads();                                   // everybody has read the old key before thread 0 replaces it
  if (threadIdx.x < 3) {
    uint32_t child[16];
    chacha_derive_key(parent, threadIdx.x, D3P_DERIVE_SPLIT, child);
    if (threadIdx.x == 0) {
#pragma unroll
      for (int i = 0; i < 16; ++i) key_io[i] = child[i];
    } else if (threadIdx.x == 1) {
      uint32_t ks[16];
      chacha20_block(child, child[12], ks);
      tf_key_out[0] = ks[0]; tf_key_out[1] = ks[1];
    } else {
#pragma unroll
      for (int i = 0; i < 16; ++i) s_noise[i] = child[i];
    }
  }
  __syncthreads();
  if (threadIdx.x < n_leaves) {
    uint32_t noise[16], child[16];
#pragma unroll
    for (int i = 0; i < 16; ++i) noise[i] = s_noise[i];
    chacha_derive_key(noise, threadIdx.x, D3P_DERIVE_SPLIT, child);
#pragma unroll
    for (int i = 0; i < 16; ++i) site_out[16 * threadIdx.x + i] = child[i];
  }
}

template <int kMode>
static int32_t launch_stream(const uint32_t* state_h, const uint32_t* state_d, uint64_t first_block, void* out_d, size_t n,
                             float lo, float hi, void* stream) {
  if ((!state_h && !state_d) || (!out_d && n)) return D3P_ERR_INVALID_ARGUMENT;
  if (n == 0) return D3P_OK;
  size_t n_blocks = (n + 15) / 16;
  if (first_block + n_blocks > 0x100000000ull) return D3P_ERR_INVALID_ARGUMENT;  // 32-bit block counter
  int threads = 256;
  size_t grid = (n_blocks + threads - 1) / threads;
  if (grid > (size_t)sm_count() * 16) grid = (size_t)sm_count() * 16;
  chacha_stream_kernel<kMode><<<(unsigned)grid, threads, 0, (cudaStream_t)stream>>>(
      chacha_arg(state_h, state_d), (uint32_t)first_block, out_d, n, lo, hi);
  return check_launch();
}

int32_t randint_impl(const uint32_t* key_h, const uint32_t* key_d, uint32_t nbits, int64_t minval, int64_t maxval,
                     void* out_d, size_t n, void* stream) {
  if (nbits != 8 && nbits != 16 && nbits != 32) return D3P_ERR_UNSUPPORTED;
  if (n == 0) return D3P_OK;
  if ((!key_h && !key_d) || !out_d) return D3P_ERR_INVALID_ARGUMENT;
  // delta = (maxval - 1 - minval) mod 2^nbits; the arithmetic is done unsigned so that it wraps without overflow
  const uint32_t full = nbits == 32 ? 0xFFFFFFFFu : (1u << nbits) - 1u;
  const uint32_t delta = (uint32_t)((uint64_t)maxval - 1u - (uint64_t)minval) & full;
  const uint32_t bitmask = d3p_randint_bitmask(nbits, delta);
  const size_t per_block = 512 / nbits;
  const size_t n_blocks = (n + per_block - 1) / per_block;
  size_t grid = (n_blocks + 255) / 256;
  if (grid > (size_t)sm_count() * 16) grid = (size_t)sm_count() * 16;
  const ChaChaArg key = chacha_arg(key_h, key_d);
  cudaStream_t s = (cudaStream_t)stream;
  if (nbits == 8)
    randint_kernel<8><<<(unsigned)grid, 256, 0, s>>>(key, bitmask, delta, (uint32_t)minval, out_d, n);
  else if (nbits == 16)
    randint_kernel<16><<<(unsigned)grid, 256, 0, s>>>(key, bitmask, delta, (uint32_t)minval, out_d, n);
  else
    randint_kernel<32><<<(unsigned)grid, 256, 0, s>>>(key, bitmask, delta, (uint32_t)minval, out_d, n);
  return check_launch();
}

}  // namespace d3p

using namespace d3p;

extern "C" {

int32_t d3p_abi_version(void) { return 3; }

// CUDA event helpers so that a host language without a CUDA binding can time kernels on the stream
// they are launched on (bench.py's roofline block).
int32_t d3p_event_create(void** event_out) {
  if (!event_out) return D3P_ERR_INVALID_ARGUMENT;
  cudaEvent_t e;
  if (cudaEventCreate(&e) != cudaSuccess) return D3P_ERR_CUDA;
  *event_out = e;
  return D3P_OK;
}
int32_t d3p_event_record(void* event, void* stream) {
  return cudaEventRecord((cudaEvent_t)event, (cudaStream_t)stream) == cudaSuccess ? D3P_OK : D3P_ERR_CUDA;
}
int32_t d3p_event_elapsed_ms(void* begin, void* end, float* ms_out) {
  if (!ms_out) return D3P_ERR_INVALID_ARGUMENT;
  if (cudaEventSynchronize((cudaEvent_t)end) != cudaSuccess) return D3P_ERR_CUDA;
  return cudaEventElapsedTime(ms_out, (cudaEvent_t)begin, (cudaEvent_t)end) == cudaSuccess ? D3P_OK : D3P_ERR_CUDA;
}
int32_t d3p_event_destroy(void* event) {
  return cudaEventDestroy((cudaEvent_t)event) == cudaSuccess ? D3P_OK : D3P_ERR_CUDA;
}

const char* d3p_error_string(int32_t code) {
  switch (code) {
    case D3P_OK: return "ok";
    case D3P_ERR_INVALID_ARGUMENT: return "invalid argument";
    case D3P_ERR_CUDA: return "CUDA error (kernel launch failed)";
    case D3P_ERR_UNSUPPORTED: return "unsupported configuration";
    case D3P_ERR_WORKSPACE: return "workspace too small";
    case D3P_ERR_PEER_TIMEOUT: return "a peer-memory exchange timed out earlier (sticky; the replicas have diverged)";
    default: return "unknown error";
  }
}

int32_t d3p_chacha_key_from_seed_h(const uint8_t* seed_h, size_t len, uint32_t out_h[16]) {
  if (!out_h || (!seed_h && len) || len > 32) return D3P_ERR_INVALID_ARGUMENT;
  uint8_t buf[32] = {0};
  for (size_t i = 0; i < len; ++i) buf[i] = seed_h[i];
  out_h[0] = 0x61707865u; out_h[1] = 0x3320646Eu; out_h[2] = 0x79622D32u; out_h[3] = 0x6B206574u;
  for (int i = 0; i < 8; ++i)
    out_h[4 + i] = (uint32_t)buf[4 * i] | ((uint32_t)buf[4 * i + 1] << 8) | ((uint32_t)buf[4 * i + 2] << 16) |
                   ((uint32_t)buf[4 * i + 3] << 24);
  out_h[12] = out_h[13] = out_h[14] = out_h[15] = 0;
  return D3P_OK;
}

int32_t d3p_chacha_fold_in_h(const uint32_t in_h[16], uint32_t data, uint32_t out_h[16]) {
  if (!in_h || !out_h) return D3P_ERR_INVALID_ARGUMENT;
  uint32_t tmp[16];
  uint32_t src[16];
  for (int i = 0; i < 16; ++i) src[i] = in_h[i];
  chacha_derive_key(src, data, D3P_DERIVE_FOLD_IN, tmp);
  for (int i = 0; i < 16; ++i) out_h[i] = tmp[i];
  return D3P_OK;
}

int32_t d3p_chacha_split_h(const uint32_t in_h[16], int32_t num, uint32_t* out_h) {
  if (!in_h || num < 0 || (!out_h && num)) return D3P_ERR_INVALID_ARGUMENT;
  uint32_t src[16];
  for (int i = 0; i < 16; ++i) src[i] = in_h[i];
  for (int32_t k = 0; k < num; ++k) {
    uint32_t child[16];
    chacha_derive_key(src, (uint32_t)k, D3P_DERIVE_SPLIT, child);
    for (int i = 0; i < 16; ++i) out_h[16 * (size_t)k + i] = child[i];
  }
  return D3P_OK;
}

int32_t d3p_chacha_random_bits_h(const uint32_t state_h[16], uint64_t first_block, uint32_t* out_h,
                                 size_t n_words) {
  if (!state_h || (!out_h && n_words)) return D3P_ERR_INVALID_ARGUMENT;
  uint32_t st[16], blk[16];
  for (int i = 0; i < 16; ++i) st[i] = state_h[i];
  for (size_t b = 0; b * 16 < n_words; ++b) {
    chacha20_block(st, st[12] + (uint32_t)first_block + (uint32_t)b, blk);
    for (int i = 0; i < 16 && b * 16 + i < n_words; ++i) out_h[b * 16 + i] = blk[i];
  }
  return D3P_OK;
}

int32_t d3p_chacha_random_bits(const uint32_t state_h[16], uint64_t first_block, uint32_t* out_d,
                               size_t n_words, void* stream) {
  return launch_stream<kBits>(state_h, nullptr, first_block, out_d, n_words, 0.f, 1.f, stream);
}

int32_t d3p_chacha_uniform_f32(const uint32_t state_h[16], uint64_t first_block, float lo, float hi,
                               float* out_d, size_t n, void* stream) {
  return launch_stream<kUniform>(state_h, nullptr, first_block, out_d, n, lo, hi, stream);
}

int32_t d3p_chacha_normal_f32(const uint32_t state_h[16], uint64_t first_block, float* out_d, size_t n,
                              void* stream) {
  return launch_stream<kNormal>(state_h, nullptr, first_block, out_d, n, 0.f, 1.f, stream);
}

int32_t d3p_chacha_randint_round(const uint32_t round_state_h[16], uint32_t nbits, uint32_t bitmask, uint32_t delta,
                                 int32_t first, uint32_t* vals_d, size_t n, int32_t* pending_d, void* stream) {
  if (!round_state_h || !pending_d || (!vals_d && n)) return D3P_ERR_INVALID_ARGUMENT;
  if (nbits != 8 && nbits != 16 && nbits != 32) return D3P_ERR_UNSUPPORTED;
  cudaMemsetAsync(pending_d, 0, sizeof(int32_t), (cudaStream_t)stream);
  if (n == 0) return check_launch();
  const size_t per_block = 512 / nbits;
  size_t n_blocks = (n + per_block - 1) / per_block;
  size_t grid = (n_blocks + 255) / 256;
  if (grid > (size_t)sm_count() * 16) grid = (size_t)sm_count() * 16;
  const ChaChaArg key = chacha_arg(round_state_h, nullptr);
  cudaStream_t s = (cudaStream_t)stream;
  if (nbits == 8)
    randint_round_kernel<8><<<(unsigned)grid, 256, 0, s>>>(key, bitmask, delta, first, vals_d, n, pending_d);
  else if (nbits == 16)
    randint_round_kernel<16><<<(unsigned)grid, 256, 0, s>>>(key, bitmask, delta, first, vals_d, n, pending_d);
  else
    randint_round_kernel<32><<<(unsigned)grid, 256, 0, s>>>(key, bitmask, delta, first, vals_d, n, pending_d);
  return check_launch();
}

int32_t d3p_chacha_randint_round_u32(const uint32_t round_state_h[16], uint32_t bitmask, uint32_t delta,
                                     int32_t first, uint32_t* vals_d, size_t n, int32_t* pending_d,
                                     void* stream) {
  return d3p_chacha_randint_round(round_state_h, 32, bitmask, delta, first, vals_d, n, pending_d, stream);
}

int32_t d3p_randint_finish(const uint32_t* vals_d, int32_t minval, uint32_t nbits, void* out_d, size_t n, void* stream) {
  if ((!vals_d || !out_d) && n) return D3P_ERR_INVALID_ARGUMENT;
  if (nbits != 8 && nbits != 16 && nbits != 32) return D3P_ERR_UNSUPPORTED;
  if (n == 0) return D3P_OK;
  size_t grid = (n + 255) / 256;
  if (grid > (size_t)sm_count() * 16) grid = (size_t)sm_count() * 16;
  cudaStream_t s = (cudaStream_t)stream;
  if (nbits == 8) randint_finish_kernel<int8_t><<<(unsigned)grid, 256, 0, s>>>(vals_d, minval, (int8_t*)out_d, n);
  else if (nbits == 16) randint_finish_kernel<int16_t><<<(unsigned)grid, 256, 0, s>>>(vals_d, minval, (int16_t*)out_d, n);
  else randint_finish_kernel<int32_t><<<(unsigned)grid, 256, 0, s>>>(vals_d, minval, (int32_t*)out_d, n);
  return check_launch();
}

int32_t d3p_randint_finish_i32(const uint32_t* vals_d, int32_t minval, int32_t* out_d, size_t n, void* stream) {
  return d3p_randint_finish(vals_d, minval, 32, out_d, n, stream);
}

// log_po2 = min(int(float32(log2(float32(delta))) + 1), nbits) of randint (d3p/random/__init__.py:84-146).  Rounding delta and
// its log2 to float32 widens the mask by one bit just below powers of two (delta = 2^25 - 1 rounds to 2^25, and
// log2(2^24 - 1) rounds to 24); the reference does this, so it is kept.  log2 is taken in double and rounded once to float32, i.e. a correctly rounded
// log2f: near an integer the float32 result is far from a rounding tie, so every faithful log2f agrees with it.
uint32_t d3p_randint_bitmask(uint32_t nbits, uint32_t delta) {
  if (nbits == 0) return 0;
  if (nbits > 32) nbits = 32;
  uint32_t log_po2 = 0;
  if (delta > 0) {
    const float l = (float)log2((double)(float)delta);
    log_po2 = (uint32_t)(l + 1.0f);
  }
  if (log_po2 > nbits) log_po2 = nbits;
  return log_po2 >= 32 ? 0xFFFFFFFFu : (1u << log_po2) - 1u;
}

int32_t d3p_chacha_randint(const uint32_t key_h[16], uint32_t nbits, int64_t minval, int64_t maxval, void* out_d,
                           size_t n, void* stream) {
  return randint_impl(key_h, nullptr, nbits, minval, maxval, out_d, n, stream);
}


// ---- device-key forms (keys never leave the device) ------------------------------------------------------------------
int32_t d3p_chacha_split_dk(const uint32_t* in_d, int32_t num, uint32_t* out_d, void* stream) {
  if (!in_d || num < 0 || (!out_d && num)) return D3P_ERR_INVALID_ARGUMENT;
  if (num == 0) return D3P_OK;
  const unsigned threads = 128, grid = ((unsigned)num + threads - 1) / threads;
  chacha_split_dk_kernel<<<grid > 1024 ? 1024 : grid, threads, 0, (cudaStream_t)stream>>>(in_d, (uint32_t)num, out_d);
  return check_launch();
}

int32_t d3p_chacha_fold_in_dk(const uint32_t* in_d, const uint32_t* data_d, uint32_t data_imm, uint32_t* out_d,
                              void* stream) {
  if (!in_d || !out_d) return D3P_ERR_INVALID_ARGUMENT;
  chacha_fold_in_dk_kernel<<<1, 32, 0, (cudaStream_t)stream>>>(in_d, data_d, data_imm, out_d);
  return check_launch();
}

int32_t d3p_chacha_random_bits_dk(const uint32_t* state_d, uint64_t first_block, uint32_t* out_d, size_t n_words,
                                  void* stream) {
  return launch_stream<kBits>(nullptr, state_d, first_block, out_d, n_words, 0.f, 1.f, stream);
}

int32_t d3p_chacha_uniform_f32_dk(const uint32_t* state_d, uint64_t first_block, float lo, float hi, float* out_d,
                                  size_t n, void* stream) {
  return launch_stream<kUniform>(nullptr, state_d, first_block, out_d, n, lo, hi, stream);
}

int32_t d3p_chacha_normal_f32_dk(const uint32_t* state_d, uint64_t first_block, float* out_d, size_t n, void* stream) {
  return launch_stream<kNormal>(nullptr, state_d, first_block, out_d, n, 0.f, 1.f, stream);
}

int32_t d3p_chacha_randint_dk(const uint32_t* key_d, uint32_t nbits, int64_t minval, int64_t maxval, void* out_d,
                              size_t n, void* stream) {
  return randint_impl(nullptr, key_d, nbits, minval, maxval, out_d, n, stream);
}

int32_t d3p_dpsvi_keys_dk(uint32_t* rng_key_io_d, uint32_t n_leaves, uint32_t* threefry_key_out_d,
                          uint32_t* site_states_out_d, void* stream) {
  if (!rng_key_io_d || !threefry_key_out_d || n_leaves > D3P_MAX_LEAVES || (n_leaves && !site_states_out_d))
    return D3P_ERR_INVALID_ARGUMENT;
  dpsvi_keys_dk_kernel<<<1, 32, 0, (cudaStream_t)stream>>>(rng_key_io_d, n_leaves, threefry_key_out_d, site_states_out_d);
  return check_launch();
}

}  // extern "C"
