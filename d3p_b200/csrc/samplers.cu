// K2 Feistel sampler, K3 Poisson select + ordered compaction, K4 masked row gather.
// Replace d3p/util.py:216-301 and d3p/minibatch.py:29-39,103-131,210,233,306.
#include <string.h>

#include "comm.cuh"
#include "common.cuh"
#include "launch.cuh"

namespace d3p {

// ---------------------------------------------------------------------------------------------
// K2: keyed Feistel bijection with cycle walking (d3p/util.py:249-299)
// ---------------------------------------------------------------------------------------------
struct FeistelParams {
  uint32_t rc[30];
  uint32_t capacity, bits_lower, bits_upper, mask_lower, mask_upper;
};

// round constants from device memory (d3p_feistel_sample_dk): 30 keystream words of the batch key, rc[3j] |= 1
__global__ void feistel_rc_dk_kernel(const uint32_t* __restrict__ state_d, uint32_t* __restrict__ rc_out) {
  if (threadIdx.x >= 2) return;
  uint32_t st[16], ks[16];
#pragma unroll
  for (int i = 0; i < 16; ++i) st[i] = state_d[i];
  chacha20_block(st, st[12] + threadIdx.x, ks);
#pragma unroll
  for (int i = 0; i < 16; ++i) {
    const uint32_t w = 16u * threadIdx.x + i;
    if (w < 30) rc_out[w] = (w % 3 == 0) ? (ks[i] | 1u) : ks[i];
  }
}

D3P_D uint32_t feistel_rounds(const FeistelParams& p, uint32_t x) {
#pragma unroll
  for (int j = 0; j < 10; ++j) {
    uint32_t xu = x >> p.bits_lower;
    uint32_t xl = x & p.mask_lower;
    uint32_t f = ((xu * p.rc[3 * j + 1]) >> p.bits_upper) ^ p.rc[3 * j + 2];
    uint32_t yu = (f & p.mask_lower) ^ xl;
    uint32_t yl = (xu * p.rc[3 * j]) & p.mask_upper;
    x = (yu << p.bits_upper) | yl;
  }
  return x;
}

__global__ void __launch_bounds__(256) feistel_kernel(FeistelParams p, const uint32_t* __restrict__ rc_d,
                                                      uint32_t first_pos, uint32_t n, int32_t* __restrict__ idx) {
  if (rc_d) {
#pragma unroll
    for (int j = 0; j < 30; ++j) p.rc[j] = __ldg(rc_d + j);
  }
  for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    uint32_t x = feistel_rounds(p, first_pos + i);
    while (x >= p.capacity) x = feistel_rounds(p, x);
    idx[i] = (int32_t)x;
  }
}

// ---------------------------------------------------------------------------------------------
// K3: Poisson sampling. One thread per ChaCha block (16 records), one CTA per tile of 4096 records.
//   pass A: selectors -> 16-bit masks + per-tile counts
//   pass B: one CTA scans tile counts from the HIGH end (output order is descending index)
//   pass C: ordered scatter of selected (and, for the padding slots, unselected) indices
// ---------------------------------------------------------------------------------------------
constexpr int kPoisThreads = 256;
constexpr uint32_t kTileRecords = kPoisThreads * 16;

// 16 selectors of ChaCha block `blk`: rng_suite.uniform(key, (N,), float32) <= q  (d3p/minibatch.py:34)
// The uniform of word w is u = k 2^-23 with k = w >> 9, exactly (jax.random._uniform: mantissa bits | 1.0f, minus 1, times
// (1 - 0) plus 0, max with 0: every step exact), so u <= q  <=>  k <= floor(q 2^23) for 0 <= q < 1 (q 2^23 is exact in
// float32); q >= 1 selects everything, q < 0 or NaN nothing.  One integer compare per record instead of the float path.
D3P_D int32_t poisson_threshold(float q) {
  return q >= 1.0f ? 0x7fffff : (q >= 0.0f ? (int32_t)floorf(q * 8388608.0f) : -1);
}
D3P_D uint32_t poisson_block_mask(const ChaChaState& st, float q, uint32_t n_records, uint32_t blk) {
  uint32_t ks[16];
  chacha20_block(st.w, st.w[12] + blk, ks);
  const int32_t kq = poisson_threshold(q);
  uint32_t m = 0;
#pragma unroll
  for (int i = 0; i < 16; ++i) m |= ((int32_t)(ks[i] >> 9) <= kq ? 1u : 0u) << i;
  const uint32_t first = blk * 16u;                          // records past the end of the data set (last block only)
  const uint32_t n_valid = n_records > first ? min(16u, n_records - first) : 0u;
  return m & ((1u << n_valid) - 1u);
}

D3P_D int tile_count(uint32_t m, int* warp_c) {      // CTA total of popc(m); valid in thread 0
  int c = __popc(m);
  c = __reduce_add_sync(0xffffffffu, c);
  if ((threadIdx.x & 31) == 0) warp_c[threadIdx.x >> 5] = c;
  __syncthreads();
  int t = 0;
  if (threadIdx.x == 0) {
#pragma unroll
    for (int w = 0; w < kPoisThreads / 32; ++w) t += warp_c[w];
  }
  return t;
}

__global__ void __launch_bounds__(kPoisThreads) poisson_select_kernel(ChaChaArg key, float q, uint32_t n_records,
                                                                      uint16_t* __restrict__ masks,
                                                                      int32_t* __restrict__ tile_counts, uint32_t* ready) {
  if (blockIdx.x == 0 && threadIdx.x == 0) *ready = 0u;      // the compaction kernel's "prefix published" flag
  ChaChaState st;
  load_chacha(key, st);
  uint32_t blk = blockIdx.x * kPoisThreads + threadIdx.x;
  uint32_t n_blocks = (n_records + 15) / 16;
  uint32_t m = 0;
  if (blk < n_blocks) {
    m = poisson_block_mask(st, q, n_records, blk);
    masks[blk] = (uint16_t)m;
  }
  __shared__ int warp_c[kPoisThreads / 32];
  const int t = tile_count(m, warp_c);
  if (threadIdx.x == 0) tile_counts[blockIdx.x] = t;
}

// ---- sharded variant (comm.cuh) -----------------------------------------------------------------------------
// This rank draws tiles [cov_lo, cov_lo + gridDim.x): the slice it owns, [own_lo, own_hi), plus a margin on
// both sides, so that the tiles its batch positions fall into are (with overwhelming probability) local and
// no selection mask ever crosses NVLink.  Only the owner pushes a tile's tagged count {count, epoch & 0xffff}
// into every window (posted stores: no fence and no flag, the tag validates the word).
__global__ void __launch_bounds__(kPoisThreads) poisson_select_sharded_kernel(ChaChaArg key, float q,
                                                                              uint32_t n_records, uint32_t cov_lo,
                                                                              uint32_t own_lo, uint32_t own_hi,
                                                                              uint16_t* __restrict__ masks, SampDev sd,
                                                                              uint32_t* ready) {
  if (blockIdx.x == 0 && threadIdx.x == 0) *ready = 0u;
  ChaChaState st;
  load_chacha(key, st);
  const uint32_t tile = cov_lo + blockIdx.x;
  const uint32_t blk = tile * kPoisThreads + threadIdx.x;
  const uint32_t n_blocks = (n_records + 15) / 16;
  uint32_t m = 0;
  if (blk < n_blocks) {
    m = poisson_block_mask(st, q, n_records, blk);
    masks[blk] = (uint16_t)m;
  }
  __shared__ int warp_c[kPoisThreads / 32];
  const int t = tile_count(m, warp_c);
  if (threadIdx.x == 0 && tile >= own_lo && tile < own_hi) {
    const uint32_t w = ((sd.epoch & 0xffffu) << 16) | (uint32_t)t;
    for (int r = 0; r < sd.world; ++r)
      asm volatile("st.relaxed.sys.global.u32 [%0], %1;" ::"l"(sd.counts_peer[r] + tile), "r"(w) : "memory");
  }
}


// Pass B (CTA 0 of the compaction kernel): the per-tile counts become "selected records in the tiles above" (exclusive
// prefix in DESCENDING tile order, the output order of d3p/minibatch.py:37) + the total, published to the other CTAs
// through a ready flag.  Sharded: the counts are the tagged words the tile owners pushed into this rank's window; only
// this CTA polls them.  (Round 1 had every compaction CTA add up all n_tiles counts itself: n_tiles^2 loads, 15.5 us at
// N = 10 M, paid in full by every rank of a sharded run.)  A separate scan launch would do the same, but it would put
// a kernel that waits for the peers in front of a dependent kernel of the same stream, and streams that share a
// hardware work queue would then block each other; this way the waiting kernel stays the last one of the sampler call.
template <bool kSharded>
D3P_D void scan_tiles(const int32_t* __restrict__ tile_counts, uint32_t n_tiles, uint32_t max_b, int suppress,
                      int32_t* __restrict__ tile_above, int32_t* __restrict__ counts, const SampDev& sd, int* warp_tot) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  // thread i owns a run of consecutive tiles, runs ordered from the HIGH end: thread 0 has the top tiles
  const uint32_t per = (n_tiles + kPoisThreads - 1) / kPoisThreads;
  const uint32_t hi = n_tiles > threadIdx.x * per ? n_tiles - threadIdx.x * per : 0;      // exclusive upper end
  const uint32_t lo = hi > per ? hi - per : 0;
  int mine = 0;
  for (uint32_t t = lo; t < hi; ++t) mine += kSharded ? (int)samp_wait_count(sd, t) : tile_counts[t];
  int incl = mine;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const int v = __shfl_up_sync(0xffffffffu, incl, o);
    if (lane >= o) incl += v;
  }
  if (lane == 31) warp_tot[warp] = incl;
  __syncthreads();
  int before = 0, total = 0;                                     // sums of the warps before mine / of all warps
#pragma unroll
  for (int w = 0; w < kPoisThreads / 32; ++w) { before += w < warp ? warp_tot[w] : 0; total += warp_tot[w]; }
  int above = incl - mine + before;                              // selected records in the runs of lower thread ids
  for (uint32_t t = hi; t-- > lo;) {                             // descending inside the run
    tile_above[t] = above;
    above += kSharded ? (int)samp_wait_count(sd, t) : tile_counts[t];
  }
  if (threadIdx.x == 0) {
    const uint32_t tot = (uint32_t)total;
    const uint32_t eff = suppress ? (tot <= max_b ? tot : 0u) : (tot < max_b ? tot : max_b);
    tile_above[n_tiles] = (int32_t)tot;
    counts[0] = (int32_t)tot; counts[1] = (int32_t)eff;
  }
}

// Pass C: one CTA per tile compacts it in DESCENDING record order: idx[s] for the selected records (s = number of
// selected records with a larger index = tile_above[tile] + those above it inside the tile), and the unselected ones
// behind them for the padding slots (d3p/minibatch.py:37).  CTAs whose tile cannot reach a wanted position leave at once.
// counts[0] = number selected, counts[1] = after truncate / suppress (:119-122), mask = arange(max_b) < counts[1].
// kSharded (comm.cuh): counts were pushed into the local window by the tile owners, masks are local (or
// re-drawn), only positions [pos_begin, pos_end) are written and padding slots are left alone.
constexpr int kCompactTiles = 1;               // tiles per CTA (8 measured slower: the per-tile barriers serialise)

template <bool kSharded>
__global__ void __launch_bounds__(kPoisThreads) poisson_compact_kernel(const uint16_t* __restrict__ masks,
                                                                       const int32_t* __restrict__ tile_counts,
                                                                       int32_t* tile_above_g, uint32_t* ready,
                                                                       uint32_t n_records, uint32_t n_tiles,
                                                                       uint32_t max_b, int suppress, uint32_t pos_begin,
                                                                       uint32_t pos_end, int32_t* __restrict__ idx,
                                                                       int32_t* __restrict__ counts,
                                                                       uint8_t* __restrict__ mask, SampDev sd,
                                                                       ChaChaArg key, float q, uint32_t cov_lo,
                                                                       uint32_t cov_hi) {
  const uint32_t t_first = blockIdx.x * kCompactTiles;                       // this CTA's tiles [t_first, t_end)
  const uint32_t t_end = min(n_tiles, t_first + kCompactTiles);
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  __shared__ int warp_tot[kPoisThreads / 32];
  static_assert(kCompactTiles == 1, "one tile per CTA");
  // CTA 0 (always dispatched first) scans the tile counts and raises `ready` (reset by the selector kernel, which
  // precedes this one on the stream); the others wait for it
  if (blockIdx.x == 0) {
    scan_tiles<kSharded>(tile_counts, n_tiles, max_b, suppress, tile_above_g, counts, sd, warp_tot);
    __threadfence();
    __syncthreads();
    if (threadIdx.x == 0) asm volatile("st.release.gpu.global.u32 [%0], %1;" ::"l"(ready), "r"(1u) : "memory");
  } else {
    if (threadIdx.x == 0) {
      uint32_t v;
      do { asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(ready) : "memory"); } while (v != 1u);
    }
    __syncthreads();
  }
  const uint32_t total = (uint32_t)__ldcg(tile_above_g + n_tiles);
  const int above = __ldcg(tile_above_g + t_first);
  // this tile's count = the next-lower tile's "above" minus ours (the lowest tile: total - above)
  const uint32_t own_count = (t_first > 0 ? (uint32_t)__ldcg(tile_above_g + t_first - 1) : total) - (uint32_t)above;
  const uint32_t eff = suppress ? (total <= max_b ? total : 0u) : (total < max_b ? total : max_b);
  if (mask) {                                  // this CTA's slice of the mask, 4 bytes per store when aligned
    const uint32_t words = (max_b + 3) / 4, per = (words + gridDim.x - 1) / gridDim.x;
    const bool aligned = (reinterpret_cast<uintptr_t>(mask) & 3) == 0;
    for (uint32_t wd = blockIdx.x * per + threadIdx.x; wd < min(words, (blockIdx.x + 1) * per); wd += kPoisThreads) {
      const uint32_t i = wd * 4;
      if (aligned && i + 4 <= max_b) {
        uint32_t v = 0;
#pragma unroll
        for (int k = 0; k < 4; ++k) v |= ((i + k < eff) ? 1u : 0u) << (8 * k);
        *reinterpret_cast<uint32_t*>(mask + i) = v;
      } else {
        for (uint32_t j = i; j < min(i + 4, max_b); ++j) mask[j] = j < eff ? 1 : 0;
      }
    }
  }
  const uint32_t lim = kSharded ? min(min(pos_end, max_b), eff) : max_b;
  const uint32_t n_blocks = (n_records + 15) / 16;
  uint32_t tile_above = (uint32_t)above;       // selected records in tiles above the current one
  for (uint32_t tile = t_end; tile-- > t_first;) {                           // descending: running offset
    const uint32_t cnt = own_count;
    const uint32_t base = tile_above;
    tile_above += cnt;
    // CTA-uniform early outs: nothing of this tile lands in the wanted positions
    if (kSharded && (base + cnt <= pos_begin || base >= lim)) continue;
    if (!kSharded && base >= max_b && total >= max_b) continue;
    const uint32_t blk = tile * kPoisThreads + threadIdx.x;
    uint32_t m = 0;
    if (blk < n_blocks) {
      // sharded: inside the locally drawn range the masks are in this rank's scratch; a tile outside it (a
      // position boundary further off than the margin: many standard deviations) is simply drawn again
      if (!kSharded || (tile >= cov_lo && tile < cov_hi)) {
        m = masks[blk];
      } else {
        ChaChaState st;
        load_chacha(key, st);
        m = poisson_block_mask(st, q, n_records, blk);
      }
    }
    const int c = __popc(m);
    int incl = c;                              // exclusive scan over threads in DESCENDING thread order
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      int t = __shfl_down_sync(0xffffffffu, incl, o);
      if (lane + o < 32) incl += t;
    }
    __syncthreads();                           // warp_tot of the previous tile has been consumed
    if (lane == 0) warp_tot[warp] = incl;
    __syncthreads();
    int higher = 0;
#pragma unroll
    for (int w = 0; w < kPoisThreads / 32; ++w)
      if (w > warp) higher += warp_tot[w];
    uint32_t s = base + (uint32_t)(higher + incl - c);   // selected records with a larger index
    if (blk >= n_blocks) continue;
    if (kSharded) {
      // walk the SET bits from the top (1 % of the records are selected: 2 - 3 iterations per warp instead of 16)
      for (uint32_t mm = m; mm;) {
        const int i = 31 - __clz(mm);
        mm &= ~(1u << i);
        if (s >= pos_begin && s < lim) idx[s] = (int32_t)(blk * 16u + i);
        ++s;
      }
      continue;
    }
    const uint32_t rec_hi = blk * 16u + 15u;
    // quick reject: nothing from this chacha block can land in [0, max_b)
    const bool any_sel = (m != 0) && (s < max_b);
    const bool any_unsel = total < max_b && ((n_records - 1u - min(rec_hi, n_records - 1u)) - s + total < max_b + 16u);
    if (!any_sel && !any_unsel) continue;
    if (!any_unsel) {
      // the common case (no padding slot can come from this block): walk the set bits from the top, 2 - 3
      // iterations per warp instead of the 16 of the general loop below
      for (uint32_t mm = m; mm;) {
        const int i = 31 - __clz(mm);
        mm &= ~(1u << i);
        const uint32_t rec = blk * 16u + i;
        if (rec >= n_records) continue;
        if (s < max_b) idx[s] = (int32_t)rec;
        ++s;
      }
      continue;
    }
#pragma unroll
    for (int i = 15; i >= 0; --i) {
      const uint32_t rec = blk * 16u + i;
      if (rec >= n_records) continue;
      if ((m >> i) & 1u) {
        if (s < max_b) idx[s] = (int32_t)rec;
        ++s;
      } else {
        const uint32_t pos = total + (n_records - 1u - rec) - s;
        if (pos < max_b) idx[pos] = (int32_t)rec;
      }
    }
  }
}

// ---------------------------------------------------------------------------------------------
// K4: masked row gather (d3p/minibatch.py:126-131): one warp per row, 16-byte vectors when aligned
// ---------------------------------------------------------------------------------------------
template <typename V>
__global__ void __launch_bounds__(256) gather_rows_kernel(const V* __restrict__ src, size_t row_vecs,
                                                          const int32_t* __restrict__ idx,
                                                          const int32_t* __restrict__ num_valid, uint32_t b,
                                                          V* __restrict__ dst) {
  const int lane = threadIdx.x & 31;
  const uint32_t warps_per_grid = gridDim.x * (blockDim.x >> 5);
  const uint32_t nv = num_valid ? (uint32_t)max(*num_valid, 0) : b;
  V zero;
  memset(&zero, 0, sizeof(V));
  for (uint32_t r = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5); r < b; r += warps_per_grid) {
    V* d = dst + (size_t)r * row_vecs;
    if (r < nv) {
      const V* s = src + (size_t)idx[r] * row_vecs;
      for (size_t v = lane; v < row_vecs; v += 32) d[v] = __ldg(s + v);
    } else {
      for (size_t v = lane; v < row_vecs; v += 32) d[v] = zero;
    }
  }
}

struct PoissonWs {
  uint16_t* masks;
  int32_t* tile_counts;
  int32_t* tile_off;
  uint32_t* ready;
  size_t bytes;
};

static PoissonWs carve_poisson_ws(void* ws, uint32_t n_records) {
  size_t n_blocks = ((size_t)n_records + 15) / 16;
  size_t n_tiles = (n_blocks + kPoisThreads - 1) / kPoisThreads;
  size_t o_masks = 0;
  size_t o_counts = align_up(n_blocks * sizeof(uint16_t), 256);
  size_t o_off = o_counts + align_up(n_tiles * sizeof(int32_t), 256);
  PoissonWs w;
  char* base = reinterpret_cast<char*>(ws);
  w.masks = reinterpret_cast<uint16_t*>(base + o_masks);
  w.tile_counts = reinterpret_cast<int32_t*>(base + o_counts);
  w.tile_off = reinterpret_cast<int32_t*>(base + o_off);
  size_t o_ready = o_off + align_up((n_tiles + 1) * sizeof(int32_t), 256);      // tile_off: n_tiles prefixes + the total
  w.ready = reinterpret_cast<uint32_t*>(base + o_ready);
  w.bytes = o_ready + 256;
  return w;
}

}  // namespace d3p

using namespace d3p;

extern "C" {

int32_t d3p_feistel_round_constants_h(const uint32_t state_h[16], uint32_t rc_h[30]) {
  if (!state_h || !rc_h) return D3P_ERR_INVALID_ARGUMENT;
  int32_t rc = d3p_chacha_random_bits_h(state_h, 0, rc_h, 30);
  if (rc != D3P_OK) return rc;
  for (int j = 0; j < 10; ++j) rc_h[3 * j] |= 1u;
  return D3P_OK;
}

}  // extern "C"

int32_t d3p::feistel_sample_impl(const uint32_t* rc_h, const uint32_t* rc_d, uint32_t capacity, uint32_t first_pos,
                                 uint32_t n, int32_t* idx_d, void* stream) {
  if ((!rc_h && !rc_d) || capacity == 0 || (!idx_d && n)) return D3P_ERR_INVALID_ARGUMENT;
  if ((uint64_t)first_pos + n > (uint64_t)capacity) return D3P_ERR_INVALID_ARGUMENT;
  if (n == 0) return D3P_OK;
  FeistelParams p;
  for (int i = 0; i < 30; ++i) p.rc[i] = rc_h ? rc_h[i] : 0u;
  uint32_t bits = 0;
  for (uint32_t c = capacity - 1; c; c >>= 1) ++bits;   // (capacity - 1).bit_length()
  p.capacity = capacity;
  p.bits_lower = bits >> 1;
  p.bits_upper = bits - p.bits_lower;
  p.mask_lower = (1u << p.bits_lower) - 1u;
  p.mask_upper = (1u << p.bits_upper) - 1u;
  unsigned grid = (n + 255) / 256;
  unsigned cap = (unsigned)sm_count() * 16;
  if (grid > cap) grid = cap;
  feistel_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(p, rc_d, first_pos, n, idx_d);
  return check_launch();
}

extern "C" {

int32_t d3p_feistel_sample(const uint32_t rc_h[30], uint32_t capacity, uint32_t first_pos, uint32_t n,
                           int32_t* idx_d, void* stream) {
  if (!rc_h) return D3P_ERR_INVALID_ARGUMENT;
  return feistel_sample_impl(rc_h, nullptr, capacity, first_pos, n, idx_d, stream);
}

// Device-key forms: the round constants are derived on the device from a key in device memory (rc_out_d: 30 words)
int32_t d3p_feistel_round_constants_dk(const uint32_t* state_d, uint32_t* rc_out_d, void* stream) {
  if (!state_d || !rc_out_d) return D3P_ERR_INVALID_ARGUMENT;
  feistel_rc_dk_kernel<<<1, 32, 0, (cudaStream_t)stream>>>(state_d, rc_out_d);
  return check_launch();
}

int32_t d3p_feistel_sample_dk(const uint32_t* rc_d, uint32_t capacity, uint32_t first_pos, uint32_t n, int32_t* idx_d,
                              void* stream) {
  if (!rc_d) return D3P_ERR_INVALID_ARGUMENT;
  return feistel_sample_impl(nullptr, rc_d, capacity, first_pos, n, idx_d, stream);
}

size_t d3p_poisson_workspace_bytes(uint32_t n_records) { return carve_poisson_ws(nullptr, n_records).bytes; }

}  // extern "C"

int32_t d3p::poisson_sample_impl(const uint32_t* state_h, const uint32_t* state_d, float q, uint32_t n_records,
                                 uint32_t max_b, int32_t suppress, int32_t* idx_d, int32_t* counts_d, uint8_t* mask_d,
                                 void* ws_d, size_t ws_bytes, void* stream) {
  if ((!state_h && !state_d) || !counts_d || !ws_d || (!idx_d && max_b) || n_records == 0 || max_b > n_records)
    return D3P_ERR_INVALID_ARGUMENT;
  const ChaChaArg key = chacha_arg(state_h, state_d);
  PoissonWs w = carve_poisson_ws(ws_d, n_records);
  if (ws_bytes < w.bytes) return D3P_ERR_WORKSPACE;
  uint32_t n_blocks = (n_records + 15) / 16;
  uint32_t n_tiles = (n_blocks + kPoisThreads - 1) / kPoisThreads;
  cudaStream_t s = (cudaStream_t)stream;
  poisson_select_kernel<<<n_tiles, kPoisThreads, 0, s>>>(key, q, n_records, w.masks, w.tile_counts, w.ready);
  SampDev none;
  memset(&none, 0, sizeof(none));
  poisson_compact_kernel<false><<<n_tiles, kPoisThreads, 0, s>>>(w.masks, w.tile_counts, w.tile_off, w.ready, n_records, n_tiles, max_b, suppress, 0,
                                                                 max_b, idx_d, counts_d, mask_d, none, key,
                                                                 q, 0, n_tiles);
  return check_launch();
}

extern "C" {

int32_t d3p_poisson_sample(const uint32_t state_h[16], float q, uint32_t n_records, uint32_t max_b,
                           int32_t suppress, int32_t* idx_d, int32_t* counts_d, uint8_t* mask_d, void* ws_d,
                           size_t ws_bytes, void* stream) {
  if (!state_h) return D3P_ERR_INVALID_ARGUMENT;
  return poisson_sample_impl(state_h, nullptr, q, n_records, max_b, suppress, idx_d, counts_d, mask_d, ws_d, ws_bytes, stream);
}

int32_t d3p_poisson_sample_dk(const uint32_t* state_d, float q, uint32_t n_records, uint32_t max_b, int32_t suppress,
                              int32_t* idx_d, int32_t* counts_d, uint8_t* mask_d, void* ws_d, size_t ws_bytes,
                              void* stream) {
  if (!state_d) return D3P_ERR_INVALID_ARGUMENT;
  return poisson_sample_impl(nullptr, state_d, q, n_records, max_b, suppress, idx_d, counts_d, mask_d, ws_d, ws_bytes, stream);
}

}  // extern "C"

int32_t d3p::poisson_sample_sharded_impl(d3p_comm* comm, const uint32_t* state_h, const uint32_t* state_d, float q,
                                         uint32_t n_records, uint32_t max_b, int32_t suppress, uint32_t pos_begin,
                                         uint32_t pos_end, int32_t* idx_d, int32_t* counts_d, uint8_t* mask_d,
                                         void* ws_d, size_t ws_bytes, void* stream) {
  const ChaChaArg key = chacha_arg(state_h, state_d);
  if (!comm || (!state_h && !state_d) || !counts_d || !ws_d || (!idx_d && max_b) || n_records == 0 || max_b > n_records ||
      pos_begin > pos_end || pos_end > max_b)
    return D3P_ERR_INVALID_ARGUMENT;
  PoissonWs w = carve_poisson_ws(ws_d, n_records);
  if (ws_bytes < w.bytes) return D3P_ERR_WORKSPACE;
  const uint32_t n_blocks = (n_records + 15) / 16;
  const uint32_t n_tiles = (n_blocks + kPoisThreads - 1) / kPoisThreads;
  // every rank must own at least one tile (the decision is the same on all ranks: nothing is signalled yet)
  const uint32_t tpr = (n_tiles + comm->world - 1) / comm->world;
  if (comm->world < 2 || (uint64_t)(comm->world - 1) * tpr >= n_tiles || comm->max_records < n_records)
    return D3P_ERR_UNSUPPORTED;
  SampDev sd;
  memset(&sd, 0, sizeof(sd));
  { const int32_t rc = samp_next(comm, n_records, n_tiles, &sd); if (rc != D3P_OK) return rc; }
  cudaStream_t s = (cudaStream_t)stream;
  // slices in DESCENDING record order: rank 0 draws the top tiles, whose records fill the first positions
  const uint32_t hi = n_tiles > (uint32_t)sd.rank * sd.tiles_per_rank ? n_tiles - (uint32_t)sd.rank * sd.tiles_per_rank : 0;
  const uint32_t lo = hi > sd.tiles_per_rank ? hi - sd.tiles_per_rank : 0;
  // tiles (4096 records each) drawn redundantly on each side of the owned slice (d3p_comm_set_sampler_margin; tests
  // use 0 to force the re-draw path of the compaction kernel)
  const uint32_t margin = comm->sampler_margin;
  const uint32_t cov_lo = lo > margin ? lo - margin : 0, cov_hi = hi + margin < n_tiles ? hi + margin : n_tiles;
  poisson_select_sharded_kernel<<<cov_hi - cov_lo, kPoisThreads, 0, s>>>(key, q, n_records, cov_lo, lo,
                                                                         hi, w.masks, sd, w.ready);
  poisson_compact_kernel<true><<<n_tiles, kPoisThreads, 0, s>>>(w.masks, nullptr, w.tile_off, w.ready, n_records, n_tiles, max_b, suppress,
                                                                pos_begin, pos_end, idx_d, counts_d, mask_d, sd,
                                                                key, q, cov_lo, cov_hi);
  return check_launch();
}

extern "C" {

int32_t d3p_poisson_sample_sharded(d3p_comm* comm, const uint32_t state_h[16], float q, uint32_t n_records,
                                   uint32_t max_b, int32_t suppress, uint32_t pos_begin, uint32_t pos_end,
                                   int32_t* idx_d, int32_t* counts_d, uint8_t* mask_d, void* ws_d, size_t ws_bytes,
                                   void* stream) {
  if (!state_h) return D3P_ERR_INVALID_ARGUMENT;
  return poisson_sample_sharded_impl(comm, state_h, nullptr, q, n_records, max_b, suppress, pos_begin, pos_end, idx_d,
                                     counts_d, mask_d, ws_d, ws_bytes, stream);
}

int32_t d3p_poisson_sample_sharded_dk(d3p_comm* comm, const uint32_t* state_d, float q, uint32_t n_records,
                                      uint32_t max_b, int32_t suppress, uint32_t pos_begin, uint32_t pos_end,
                                      int32_t* idx_d, int32_t* counts_d, uint8_t* mask_d, void* ws_d, size_t ws_bytes,
                                      void* stream) {
  if (!state_d) return D3P_ERR_INVALID_ARGUMENT;
  return poisson_sample_sharded_impl(comm, nullptr, state_d, q, n_records, max_b, suppress, pos_begin, pos_end, idx_d,
                                     counts_d, mask_d, ws_d, ws_bytes, stream);
}

int32_t d3p_gather_rows_masked(const void* src_d, size_t row_bytes, const int32_t* idx_d,
                               const int32_t* num_valid_d, uint32_t b, void* dst_d, void* stream) {
  if ((!src_d || !idx_d || !dst_d) && b) return D3P_ERR_INVALID_ARGUMENT;
  if (row_bytes == 0) return D3P_ERR_INVALID_ARGUMENT;
  if (b == 0) return D3P_OK;
  unsigned grid = (b + 7) / 8;
  unsigned cap = (unsigned)sm_count() * 8;
  if (grid > cap) grid = cap;
  cudaStream_t s = (cudaStream_t)stream;
  const uintptr_t both = reinterpret_cast<uintptr_t>(src_d) | reinterpret_cast<uintptr_t>(dst_d);
  bool vec16 = (row_bytes % 16 == 0) && (both % 16 == 0);
  if ((row_bytes & 3) || (both & 3))       // odd row sizes (int8 labels, 3-byte pixels, ...): byte granularity
    gather_rows_kernel<uint8_t><<<grid, 256, 0, s>>>(reinterpret_cast<const uint8_t*>(src_d), row_bytes, idx_d,
                                                     num_valid_d, b, reinterpret_cast<uint8_t*>(dst_d));
  else if (vec16)
    gather_rows_kernel<uint4><<<grid, 256, 0, s>>>(reinterpret_cast<const uint4*>(src_d), row_bytes / 16, idx_d,
                                                   num_valid_d, b, reinterpret_cast<uint4*>(dst_d));
  else
    gather_rows_kernel<uint32_t><<<grid, 256, 0, s>>>(reinterpret_cast<const uint32_t*>(src_d), row_bytes / 4, idx_d,
                                                      num_valid_d, b, reinterpret_cast<uint32_t*>(dst_d));
  return check_launch();
}

}  // extern "C"
