// Device-wide primitives written for this library (no CUB/Thrust): exclusive scan,
// order-preserving stream compaction, stable LSD radix sort of (key, index) pairs.
#pragma once
#include <stdlib.h>

#include <type_traits>

#include "common.cuh"

namespace tgp {

// ------------------------------------------------------------------------------------------
// Exclusive scan of int32 (n < 2^31): one block for small inputs, a single pass over 4096-item tiles otherwise.
// ------------------------------------------------------------------------------------------
constexpr int kScanThreads = 256;
constexpr int kScanItems = 16;
constexpr int kScanTile = kScanThreads * kScanItems;

__device__ __forceinline__ int block_exclusive_scan_i(int v, int* smem /* >= 33 ints */, int* block_total) {
  int lane = threadIdx.x & 31, w = threadIdx.x >> 5, nw = blockDim.x >> 5;
  int inc = v;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    int t = __shfl_up_sync(kFull, inc, o);
    if (lane >= o) inc += t;
  }
  __syncthreads();
  if (lane == 31) smem[w] = inc;
  __syncthreads();
  if (w == 0) {
    int s = lane < nw ? smem[lane] : 0;
    int si = s;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      int t = __shfl_up_sync(kFull, si, o);
      if (lane >= o) si += t;
    }
    smem[lane] = si - s;  // exclusive warp base
    if (lane == 31) smem[32] = si;
  }
  __syncthreads();
  int base = smem[w];
  if (block_total) *block_total = smem[32];
  return base + inc - v;
}

// Single block: exclusive scan of tile_sums[nt] in place; optional totals.
static __global__ void k_scan_spine(int* __restrict__ tile_sums, int nt, int* __restrict__ total32,
                                    int64_t* __restrict__ total64) {
  __shared__ int red[33];
  int carry = 0;
  for (int start = 0; start < nt; start += blockDim.x) {
    int i = start + threadIdx.x;
    int v = i < nt ? tile_sums[i] : 0;
    int tot;
    int ex = block_exclusive_scan_i(v, red, &tot);
    if (i < nt) tile_sums[i] = carry + ex;
    carry += tot;
    __syncthreads();
  }
  if (threadIdx.x == 0) {
    if (total32) *total32 = carry;
    if (total64) *total64 = carry;
  }
}

// Small inputs (n <= kScanSmall): ONE block scans the whole array with a running carry -- one launch and no memset.
// (The TopK step on 128 small graphs, BASELINE config 1, is a chain of ~20 launches of a few microseconds each.)
// Integer sums: the result is identical to the tiled path.
constexpr int kScanSmall = 32768;
constexpr int kScanSmallItems = 8;
static __global__ void __launch_bounds__(1024) k_scan_small(const int* __restrict__ in, int* __restrict__ out, int n,
                                                            int* __restrict__ total32, int64_t* __restrict__ total64) {
  __shared__ int red[33];
  int carry = 0;
  for (int start = 0; start < n; start += 1024 * kScanSmallItems) {
    const int base = start + (int)threadIdx.x * kScanSmallItems;
    int v[kScanSmallItems];
    int s = 0;
#pragma unroll
    for (int j = 0; j < kScanSmallItems; ++j) {
      v[j] = base + j < n ? in[base + j] : 0;
      s += v[j];
    }
    int tot;
    int ex = carry + block_exclusive_scan_i(s, red, &tot);
#pragma unroll
    for (int j = 0; j < kScanSmallItems; ++j) {
      if (base + j < n) out[base + j] = ex;
      ex += v[j];
    }
    carry += tot;
    __syncthreads();
  }
  if (threadIdx.x == 0) {
    if (total32) *total32 = carry;
    if (total64) *total64 = carry;
  }
}

// Large inputs: single-pass scan with decoupled look-back -- the input is read ONCE and there is one kernel (plus the
// memset of the tile states).  Tiles take a ticket, publish (flag, tile sum) packed in 64 bits and walk
// back over the published aggregates until they meet an inclusive prefix (same protocol as k_compact_onepass).
// tile_state ([tiles] uint64) and ticket (int) must be zero before the launch.  Sums are < 2^31 (contract of this scan).
static __global__ void __launch_bounds__(kScanThreads)
    k_scan_onepass(const int* __restrict__ in, int* __restrict__ out, int64_t n, unsigned long long* __restrict__ tile_state,
                   int* __restrict__ ticket, int num_tiles, int* __restrict__ total32, int64_t* __restrict__ total64) {
  __shared__ int red[33];
  __shared__ int s_tile, s_excl;
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  if (threadIdx.x == 0) s_tile = atomicAdd(ticket, 1);
  __syncthreads();
  const int tile = s_tile;
  const int64_t base = (int64_t)tile * kScanTile + (int64_t)threadIdx.x * kScanItems;
  int v[kScanItems];
  int s = 0;
  if (base + kScanItems <= n && (reinterpret_cast<uintptr_t>(in) & 15) == 0) {
#pragma unroll
    for (int j = 0; j < kScanItems; j += 4) {
      const int4 q = *reinterpret_cast<const int4*>(in + base + j);
      v[j] = q.x, v[j + 1] = q.y, v[j + 2] = q.z, v[j + 3] = q.w;
    }
  } else {
#pragma unroll
    for (int j = 0; j < kScanItems; ++j) v[j] = base + j < n ? in[base + j] : 0;
  }
#pragma unroll
  for (int j = 0; j < kScanItems; ++j) s += v[j];
  int total;
  int ex = block_exclusive_scan_i(s, red, &total);
  if (w == 0) {
    unsigned long long excl = 0;
    if (tile == 0) {
      if (lane == 0) atomicExch(&tile_state[0], (2ull << 32) | (unsigned)total);
    } else {
      if (lane == 0) atomicExch(&tile_state[tile], (1ull << 32) | (unsigned)total);
      int t = tile - 1;
      while (true) {
        const int idx = t - lane;
        unsigned long long st = 2ull << 32;  // before tile 0: an inclusive prefix of 0
        if (idx >= 0) {
          long long spins = 0;
          while (((st = *(volatile unsigned long long*)&tile_state[idx]) >> 32) == 0) {
            if (++spins > (1ll << 26)) __trap();
          }
        }
        const unsigned done = __ballot_sync(kFull, (st >> 32) == 2);
        const int first = done ? __ffs(done) - 1 : 31;  // lanes up to the nearest inclusive prefix contribute
        unsigned val = lane <= first ? (unsigned)(st & 0xffffffffull) : 0u;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) val += __shfl_xor_sync(kFull, val, o);
        excl += val;
        if (done) break;
        t -= 32;
      }
      if (lane == 0) {
        __threadfence();
        atomicExch(&tile_state[tile], (2ull << 32) | (unsigned)(excl + (unsigned)total));
      }
    }
    if (lane == 0) {
      s_excl = (int)excl;
      if (tile == num_tiles - 1) {
        if (total32) *total32 = (int)excl + total;
        if (total64) *total64 = (int64_t)excl + total;
      }
    }
  }
  __syncthreads();
  ex += s_excl;
  if (base + kScanItems <= n && (reinterpret_cast<uintptr_t>(out) & 15) == 0) {
#pragma unroll
    for (int j = 0; j < kScanItems; j += 4) {
      int4 q;
      q.x = ex, q.y = ex + v[j], q.z = q.y + v[j + 1], q.w = q.z + v[j + 2];
      ex = q.w + v[j + 3];
      *reinterpret_cast<int4*>(out + base + j) = q;
    }
  } else {
#pragma unroll
    for (int j = 0; j < kScanItems; ++j) {
      if (base + j < n) out[base + j] = ex;
      ex += v[j];
    }
  }
}

// workspace: tile states + ticket of the one-pass path
inline size_t scan_workspace_bytes(int64_t n) {
  return align_up(((size_t)ceil_div(n > 0 ? n : 1, kScanTile) + 2) * sizeof(unsigned long long));
}

// out may alias in.  total32/total64 (device) receive the grand total when non-null.
inline int exclusive_scan_i32(const int* in, int* out, int64_t n, int* total32, int64_t* total64, Workspace& ws,
                              cudaStream_t stream) {
  int nt = (int)ceil_div(n > 0 ? n : 1, kScanTile);
  unsigned long long* state = ws.take<unsigned long long>((size_t)nt + 2);
  if (!ws.ok) return TGPB200_ERR_WORKSPACE;
  if (n <= kScanSmall) {
    launch("k_scan_small", k_scan_small, 1, 1024, 0, stream, in, out, (int)n, total32, total64);
    return launch_status();
  }
  cudaMemsetAsync(state, 0, ((size_t)nt + 2) * sizeof(unsigned long long), stream);
  launch("k_scan_onepass", k_scan_onepass, nt, kScanThreads, 0, stream, in, out, n, state,
         reinterpret_cast<int*>(state + nt), nt, total32, total64);
  return launch_status();
}

// ------------------------------------------------------------------------------------------
// Order-preserving stream compaction.
//   Pred:  __device__ bool operator()(int64_t i, Payload& p)   -- may cache loaded data in p
//   Emit:  __device__ void operator()(int64_t i, int pos, const Payload& p)
// Pass 1 counts survivors per tile, the spine scan turns counts into offsets (+ total),
// pass 2 re-evaluates the predicate and writes survivors at offset + in-tile rank.
// ------------------------------------------------------------------------------------------
constexpr int kCompactThreads = 256;
constexpr int kCompactItems = 8;
constexpr int kCompactTile = kCompactThreads * kCompactItems;

template <typename Pred>
static __global__ void k_compact_count(Pred pred, int64_t n, int* __restrict__ tile_counts) {
  __shared__ int red[33];
  int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  int64_t base = (int64_t)blockIdx.x * kCompactTile + (int64_t)w * (32 * kCompactItems);
  int c = 0;
#pragma unroll
  for (int j = 0; j < kCompactItems; ++j) {
    int64_t i = base + j * 32 + lane;
    typename Pred::Payload p;
    if (i < n && pred(i, p)) ++c;
  }
  int tot;
  block_exclusive_scan_i(c, red, &tot);
  if (threadIdx.x == 0) tile_counts[blockIdx.x] = tot;
}

template <typename Pred, typename Emit>
static __global__ void k_compact_emit(Pred pred, Emit emit, int64_t n, const int* __restrict__ tile_offsets) {
  __shared__ int warp_tot[kCompactThreads / 32];
  int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  int64_t base = (int64_t)blockIdx.x * kCompactTile + (int64_t)w * (32 * kCompactItems);
  typename Pred::Payload pay[kCompactItems];
  unsigned ball[kCompactItems];
  int cnt = 0;
#pragma unroll
  for (int j = 0; j < kCompactItems; ++j) {
    int64_t i = base + j * 32 + lane;
    bool f = (i < n) && pred(i, pay[j]);
    ball[j] = __ballot_sync(kFull, f);
    cnt += __popc(ball[j]);
  }
  if (lane == 0) warp_tot[w] = cnt;
  __syncthreads();
  int run = tile_offsets[blockIdx.x];
  for (int k = 0; k < w; ++k) run += warp_tot[k];
  unsigned lt = (1u << lane) - 1u;
#pragma unroll
  for (int j = 0; j < kCompactItems; ++j) {
    if (ball[j] >> lane & 1u) emit(base + j * 32 + lane, run + __popc(ball[j] & lt), pay[j]);
    run += __popc(ball[j]);
  }
}

inline size_t compact_workspace_bytes(int64_t n) {
  return align_up((size_t)ceil_div(n > 0 ? n : 1, kCompactTile) * sizeof(int));
}

// Phase 1: per-tile survivor counts -> exclusive tile offsets in `counts`, grand total to total32/total64.
template <typename Pred>
inline int compact_count(Pred pred, int64_t n, int* counts, int* total32, int64_t* total64, cudaStream_t stream) {
  int nt = (int)ceil_div(n > 0 ? n : 1, kCompactTile);
  launch("k_compact_count", k_compact_count<Pred>, nt, kCompactThreads, 0, stream, pred, n, counts);
  launch("k_scan_spine", k_scan_spine, 1, 1024, 0, stream, counts, nt, total32, total64);
  return launch_status();
}
// Phase 2: write survivors (counts must hold the offsets produced by compact_count on the same input).
template <typename Pred, typename Emit>
inline int compact_emit(Pred pred, Emit emit, int64_t n, const int* counts, cudaStream_t stream) {
  int nt = (int)ceil_div(n > 0 ? n : 1, kCompactTile);
  if (n > 0) launch("k_compact_emit", k_compact_emit<Pred, Emit>, nt, kCompactThreads, 0, stream, pred, emit, n, counts);
  return launch_status();
}

// ------------------------------------------------------------------------------------------
// Single-pass order-preserving compaction (decoupled look-back): the input is read ONCE.  Outputs must have
// capacity n (the survivor count is only known at the end).  Tiles take a ticket (so a tile's predecessors are
// always running or done), publish their survivor count as (flag, value) packed in 64 bits, and resolve their
// exclusive offset by walking back over the published aggregates until they meet an inclusive prefix.
// tile_state ([tiles] uint64) and ticket (int) must be zero before the launch.  Spins are bounded (trap).
// ------------------------------------------------------------------------------------------
// A predicate may split itself into stage0 (independent streaming loads) / stage1 / stage2 (dependent lookups) and
// declare `static constexpr bool kStaged = true`.
template <typename P, typename = void>
struct pred_is_staged : std::false_type {};
template <typename P>
struct pred_is_staged<P, std::void_t<decltype(P::kStaged)>> : std::integral_constant<bool, P::kStaged> {};

template <typename Pred, typename Emit>
static __global__ void __launch_bounds__(kCompactThreads)
    k_compact_onepass(Pred pred, Emit emit, int64_t n, unsigned long long* __restrict__ tile_state,
                      int* __restrict__ ticket, int num_tiles, int64_t* __restrict__ count_out) {
  __shared__ int warp_tot[kCompactThreads / 32];
  __shared__ int s_tile, s_excl;
  int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  if (threadIdx.x == 0) s_tile = atomicAdd(ticket, 1);
  __syncthreads();
  const int tile = s_tile;
  int64_t base = (int64_t)tile * kCompactTile + (int64_t)w * (32 * kCompactItems);
  typename Pred::Payload pay[kCompactItems];
  unsigned ball[kCompactItems];
  int cnt = 0;
  if constexpr (pred_is_staged<Pred>::value) {
    // staged predicate: every stage is a separate fully unrolled loop, so the loads of all items of a stage are in
    // flight together (a one-call predicate with early exits serialises row -> col -> mask -> table per item)
    bool ok[kCompactItems];
#pragma unroll
    for (int j = 0; j < kCompactItems; ++j) {
      int64_t i = base + j * 32 + lane;
      ok[j] = i < n;
      if (ok[j]) pred.stage0(i, pay[j]);
    }
#pragma unroll
    for (int j = 0; j < kCompactItems; ++j) ok[j] = ok[j] && pred.stage1(pay[j]);
#pragma unroll
    for (int j = 0; j < kCompactItems; ++j) ok[j] = ok[j] && pred.stage2(pay[j]);
#pragma unroll
    for (int j = 0; j < kCompactItems; ++j) {
      ball[j] = __ballot_sync(kFull, ok[j]);
      cnt += __popc(ball[j]);
    }
  } else {
#pragma unroll
    for (int j = 0; j < kCompactItems; ++j) {
      int64_t i = base + j * 32 + lane;
      bool f = (i < n) && pred(i, pay[j]);
      ball[j] = __ballot_sync(kFull, f);
      cnt += __popc(ball[j]);
    }
  }
  if (lane == 0) warp_tot[w] = cnt;
  __syncthreads();
  if (w == 0) {
    // warp 0 resolves the tile's exclusive offset: 32 predecessors per look-back step
    int total = 0;
    for (int k = 0; k < kCompactThreads / 32; ++k) total += warp_tot[k];
    unsigned long long excl = 0;
    if (tile == 0) {
      if (lane == 0) atomicExch(&tile_state[0], (2ull << 32) | (unsigned)total);
    } else {
      if (lane == 0) atomicExch(&tile_state[tile], (1ull << 32) | (unsigned)total);
      int t = tile - 1;
      while (true) {
        const int idx = t - lane;
        unsigned long long v = 2ull << 32;  // before tile 0: an inclusive prefix of 0
        if (idx >= 0) {
          long long spins = 0;
          while (((v = *(volatile unsigned long long*)&tile_state[idx]) >> 32) == 0) {
            if (++spins > (1ll << 26)) __trap();
          }
        }
        const unsigned done = __ballot_sync(kFull, (v >> 32) == 2);
        // lanes up to (and including) the nearest inclusive prefix contribute
        const int first = done ? __ffs(done) - 1 : 31;
        unsigned val = lane <= first ? (unsigned)(v & 0xffffffffull) : 0u;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) val += __shfl_xor_sync(kFull, val, o);
        excl += val;
        if (done) break;
        t -= 32;
      }
      if (lane == 0) {
        __threadfence();
        atomicExch(&tile_state[tile], (2ull << 32) | (unsigned)(excl + total));
      }
    }
    if (lane == 0) {
      s_excl = (int)excl;
      if (tile == num_tiles - 1 && count_out) *count_out = (int64_t)excl + total;
    }
  }
  __syncthreads();
  int run = s_excl;
  for (int k = 0; k < w; ++k) run += warp_tot[k];
  unsigned lt = (1u << lane) - 1u;
#pragma unroll
  for (int j = 0; j < kCompactItems; ++j) {
    if (ball[j] >> lane & 1u) emit(base + j * 32 + lane, run + __popc(ball[j] & lt), pay[j]);
    run += __popc(ball[j]);
  }
}

inline size_t compact_onepass_workspace_bytes(int64_t n) {
  return align_up(((size_t)ceil_div(n > 0 ? n : 1, kCompactTile) + 2) * sizeof(unsigned long long));
}

inline size_t compact_onepass_state_words(int64_t n) { return (size_t)ceil_div(n > 0 ? n : 1, kCompactTile) + 2; }

// `state` = compact_onepass_state_words(n) 64-bit words; the caller zeroes them when state_is_zero is set (small
// inputs fold that into a kernel they launch anyway: one graph node less).
template <typename Pred, typename Emit>
static int compact_onepass_on(Pred pred, Emit emit, int64_t n, int64_t* count_out, unsigned long long* state,
                              bool state_is_zero, cudaStream_t stream) {
  int nt = (int)ceil_div(n > 0 ? n : 1, kCompactTile);
  if (!state_is_zero) cudaMemsetAsync(state, 0, ((size_t)nt + 2) * sizeof(unsigned long long), stream);
  int* ticket = reinterpret_cast<int*>(state + nt);
  if (n <= 0) {
    if (count_out) cudaMemsetAsync(count_out, 0, sizeof(int64_t), stream);
    return launch_status();
  }
  launch("k_compact_onepass", k_compact_onepass<Pred, Emit>, nt, kCompactThreads, 0, stream, pred, emit, n, state, ticket,
         nt, count_out);
  return launch_status();
}

template <typename Pred, typename Emit>
static int compact_onepass(Pred pred, Emit emit, int64_t n, int64_t* count_out, Workspace& ws, cudaStream_t stream) {
  unsigned long long* state = ws.take<unsigned long long>(compact_onepass_state_words(n));
  if (!ws.ok) return TGPB200_ERR_WORKSPACE;
  return compact_onepass_on(pred, emit, n, count_out, state, false, stream);
}

// ------------------------------------------------------------------------------------------
// Stable LSD radix sort of (key, uint32 payload) pairs, 8 bits per pass.
// Pass = tile histogram -> scan of [bins][tiles] -> stable scatter (warp match ranking, smem-staged stores).
// ------------------------------------------------------------------------------------------
constexpr int kSortThreads = 256;
#ifndef TGPB200_SORT_ITEMS
#define TGPB200_SORT_ITEMS 8  // measured on C4 (ms/step): 8: 3.32, 12: 3.35, 16: 3.50, 24: 3.85, 32: 4.11 (occupancy wins)
#endif
constexpr int kSortItems = TGPB200_SORT_ITEMS;
constexpr int kSortTile = kSortThreads * kSortItems;
constexpr int kSortMaxBins = 2048;  // histogram rows reserved per tile in the workspace (a pass uses kRadixBins)

// Measured on B200 (20 M 39-bit keys): a 10-bit pass costs 1.55x an 8-bit pass (2 KB x 8 warp counters and the staging
// buffer halve the occupancy), so 4 x 10-bit passes lose to 5 x 8-bit passes.
constexpr int kRadixBits = 8;
constexpr int kRadixBins = 1 << kRadixBits;
inline int radix_passes(int key_bits) { return key_bits < 1 ? 1 : (key_bits + kRadixBits - 1) / kRadixBits; }

template <typename KeyT>
static __global__ void k_radix_hist(const KeyT* __restrict__ keys, int64_t n, const int64_t* __restrict__ n_dev,
                                    int shift, int* __restrict__ tile_hist, int nt) {
  constexpr int BINS = kRadixBins;
  __shared__ int h[BINS];
  if (n_dev) n = min(n, *n_dev);  // device-side count (capacity launch): tiles past it publish empty histograms
  for (int d = threadIdx.x; d < BINS; d += kSortThreads) h[d] = 0;
  __syncthreads();
  int64_t base = (int64_t)blockIdx.x * kSortTile;
#pragma unroll
  for (int j = 0; j < kSortItems; ++j) {
    int64_t i = base + j * kSortThreads + threadIdx.x;
    if (i < n) atomicAdd(&h[(int)((keys[i] >> shift) & (BINS - 1))], 1);
  }
  __syncthreads();
  for (int d = threadIdx.x; d < BINS; d += kSortThreads) tile_hist[(size_t)d * nt + blockIdx.x] = h[d];
}

// Stable scatter of one tile.  Ranking: every warp owns 512 consecutive items and ranks them round by round with
// __match_any_sync (stable inside the warp); per-digit counts are then prefixed over warps and digits.  The items
// are first placed in shared memory in tile-local sorted order, so that the final global writes of a digit run are
// consecutive (full-sector stores) instead of one scattered 8/12-byte write per item.
template <typename KeyT, bool kIota>
static __global__ void __launch_bounds__(kSortThreads)
    k_radix_scatter(const KeyT* __restrict__ keys_in, const uint32_t* __restrict__ vals_in,
                    KeyT* __restrict__ keys_out, uint32_t* __restrict__ vals_out, int64_t n,
                    const int64_t* __restrict__ n_dev, int shift, const int* __restrict__ tile_off, int nt) {
  constexpr int NW = kSortThreads / 32;
  if (n_dev) n = min(n, *n_dev);
  if ((int64_t)blockIdx.x * kSortTile >= n) return;
  constexpr int BINS = kRadixBins;
  constexpr int DPT = BINS / kSortThreads;  // digits owned by one thread (consecutive)
  extern __shared__ __align__(16) unsigned char radix_smem[];
  KeyT* s_keys = reinterpret_cast<KeyT*>(radix_smem);                                     // [kSortTile]
  uint32_t* s_vals = reinterpret_cast<uint32_t*>(radix_smem + sizeof(KeyT) * kSortTile);  // [kSortTile]
  int(*warp_cnt)[BINS] = reinterpret_cast<int(*)[BINS]>(s_vals + kSortTile);              // [NW][bins]
  int* dig_base = &warp_cnt[0][0] + NW * BINS;                                            // [bins] tile-local start
  int* g_base = dig_base + BINS;                                                          // [bins] global start
  __shared__ int scan_tmp[33];
  int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  for (int i = threadIdx.x; i < NW * BINS; i += kSortThreads) (&warp_cnt[0][0])[i] = 0;
  __syncthreads();

  const int64_t tile0 = (int64_t)blockIdx.x * kSortTile;
  const int64_t base = tile0 + (int64_t)w * (32 * kSortItems);
  KeyT key[kSortItems];
  uint32_t val[kSortItems];
  int rank[kSortItems];
  // all loads of the tile first (the ranking rounds below are separated by warp-synchronous operations, which keep
  // the compiler from hoisting a load above the previous round: one exposed memory latency per round)
#pragma unroll
  for (int j = 0; j < kSortItems; ++j) {
    int64_t i = base + j * 32 + lane;
    key[j] = i < n ? keys_in[i] : (KeyT)0;
    val[j] = kIota ? (uint32_t)i : (i < n ? vals_in[i] : 0u);
  }
#pragma unroll
  for (int j = 0; j < kSortItems; ++j) {
    int64_t i = base + j * 32 + lane;
    bool valid = i < n;
    unsigned vmask = __ballot_sync(kFull, valid);
    rank[j] = 0;
    if (valid) {
      // (issuing the match of every round before the counter chain measured slower: 2.97 vs 2.81 ms on C4)
      int d = (int)((key[j] >> shift) & (BINS - 1));
      unsigned peers = __match_any_sync(vmask, d);
      int leader = __ffs(peers) - 1;
      int old = 0;
      if (lane == leader) {
        old = warp_cnt[w][d];
        warp_cnt[w][d] = old + __popc(peers);
      }
      old = __shfl_sync(vmask, old, leader);
      rank[j] = old + __popc(peers & ((1u << lane) - 1u));
    }
    __syncwarp();
  }
  __syncthreads();
  int tot;
  {
    // thread t owns digits [t*DPT, (t+1)*DPT): exclusive prefix over warps per digit, then over digits
    int dsum[DPT];
    int tsum = 0;
#pragma unroll
    for (int q = 0; q < DPT; ++q) {
      int d = threadIdx.x * DPT + q;
      int run = 0;
#pragma unroll
      for (int k = 0; k < NW; ++k) {
        int c = warp_cnt[k][d];
        warp_cnt[k][d] = run;
        run += c;
      }
      dsum[q] = run;
      tsum += run;
      g_base[d] = tile_off ? tile_off[(size_t)d * nt + blockIdx.x] : 0;
    }
    int ex = block_exclusive_scan_i(tsum, scan_tmp, &tot);
#pragma unroll
    for (int q = 0; q < DPT; ++q) {
      dig_base[threadIdx.x * DPT + q] = ex;
      ex += dsum[q];
    }
  }
  __syncthreads();
#pragma unroll
  for (int j = 0; j < kSortItems; ++j) {
    int64_t i = base + j * 32 + lane;
    if (i < n) {
      int d = (int)((key[j] >> shift) & (BINS - 1));
      int lp = dig_base[d] + warp_cnt[w][d] + rank[j];
      s_keys[lp] = key[j];
      s_vals[lp] = val[j];
    }
  }
  __syncthreads();
  for (int lp = threadIdx.x; lp < tot; lp += kSortThreads) {
    KeyT k = s_keys[lp];
    int d = (int)((k >> shift) & (BINS - 1));
    // a single tile (tile_off == nullptr: no histogram / scan launches) is globally sorted once it is tile-sorted
    int64_t pos = tile_off ? (int64_t)g_base[d] + (lp - dig_base[d]) : (int64_t)lp;
    keys_out[pos] = k;
    vals_out[pos] = s_vals[lp];
  }
}

template <typename KeyT>
constexpr size_t radix_scatter_smem() {
  return (sizeof(KeyT) + 4) * kSortTile + sizeof(int) * (kSortThreads / 32 + 2) * kRadixBins;
}

inline size_t radix_sort_workspace_bytes(int64_t n) {
  int64_t nt = ceil_div(n > 0 ? n : 1, kSortTile);
  return align_up((size_t)nt * kSortMaxBins * sizeof(int)) + scan_workspace_bytes(nt * kSortMaxBins);
}

// NOTE: internal linkage on purpose.  The kernels above are `static` (one copy per translation unit), so the
// "attribute already set" flag below must be per translation unit too; an `inline` function would share one flag
// across units and leave the other units' kernel copies without the > 48 KB shared-memory opt-in.
template <typename KeyT>
static int radix_pass(const KeyT* kin, const uint32_t* vin, KeyT* kout, uint32_t* vout, int64_t n,
                      const int64_t* n_dev, int shift, int* hist, int nt, Workspace& ws, cudaStream_t stream) {
  static bool smem_attr_set = false;  // per instantiation: > 48 KB dynamic shared memory needs the opt-in
  if (!smem_attr_set) {
    smem_attr_set = true;
    cudaFuncSetAttribute(k_radix_scatter<KeyT, true>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                         (int)radix_scatter_smem<KeyT>());
    cudaFuncSetAttribute(k_radix_scatter<KeyT, false>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                         (int)radix_scatter_smem<KeyT>());
  }
  if (nt == 1) {
    // one tile: the scatter kernel's own digit prefix is the global one -- one launch per pass instead of three
    hist = nullptr;
  } else {
    launch("k_radix_hist", k_radix_hist<KeyT>, nt, kSortThreads, 0, stream, kin, n, n_dev, shift, hist, nt);
    int rc = exclusive_scan_i32(hist, hist, (int64_t)nt * kRadixBins, nullptr, nullptr, ws, stream);
    if (rc != TGPB200_OK) return rc;
  }
  if (vin == nullptr)
    launch("k_radix_scatter", k_radix_scatter<KeyT, true>, nt, kSortThreads, radix_scatter_smem<KeyT>(),
           stream, kin, (const uint32_t*)nullptr, kout, vout, n, n_dev, shift, hist, nt);
  else
    launch("k_radix_scatter", k_radix_scatter<KeyT, false>, nt, kSortThreads, radix_scatter_smem<KeyT>(),
           stream, kin, vin, kout, vout, n, n_dev, shift, hist, nt);
  return TGPB200_OK;
}

// Sorts n pairs by the low `key_bits` bits of the key (n_dev, when given, is a device-side count <= n: the launch
// covers the capacity n and tiles past the count do nothing).  The first pass takes the payload as
// iota when vals0 == nullptr.  Buffers (keys0, vals0) and (keys1, vals1) ping-pong; returns
// (via *result_in_1) which pair holds the result.  keys0 is overwritten.
template <typename KeyT>
static int radix_sort_pairs(KeyT* keys0, uint32_t* vals0_or_null, uint32_t* vals0_buf, KeyT* keys1, uint32_t* vals1,
                            int64_t n, int key_bits, bool* result_in_1, Workspace& ws, cudaStream_t stream,
                            const int64_t* n_dev = nullptr) {
  int nt = (int)ceil_div(n > 0 ? n : 1, kSortTile);
  const int passes = radix_passes(key_bits);
  int* hist = ws.take<int>((size_t)nt * kRadixBins);
  if (!ws.ok) return TGPB200_ERR_WORKSPACE;
  size_t mark2 = ws.off;
  KeyT* kin = keys0;
  KeyT* kout = keys1;
  const uint32_t* vin = vals0_or_null;
  uint32_t* vout = vals1;
  bool in1 = false;
  for (int p = 0; p < passes; ++p) {
    ws.off = mark2;
    int rc = radix_pass<KeyT>(kin, vin, kout, vout, n, n_dev, kRadixBits * p, hist, nt, ws, stream);
    if (rc != TGPB200_OK) return rc;
    in1 = !in1;
    KeyT* tk = kin;
    kin = kout;
    kout = tk;
    vin = vout;
    vout = (vout == vals1) ? vals0_buf : vals1;
  }
  *result_in_1 = in1;
  return launch_status();
}

}  // namespace tgp
