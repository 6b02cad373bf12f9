// Sparse Connect: kept-node filter + relabel, cluster remap + coalesce, edge-weight normalisations.
// Reference: tgp/connect/base_conn.py:57-112, tgp/utils/ops.py:338-419 (and the PyG subgraph /
// coalesce / remove_self_loops semantics restated in oracle/pyg_shim.py).
#include <limits.h>

#include "prims.cuh"

namespace tgp {

// ------------------------------------------------------------------------------------------
// kept-node branch
// ------------------------------------------------------------------------------------------
// table[v] = position of v in node_index (-1 if not kept) and a 1-bit-per-node membership mask.  The mask (N/8
// bytes) stays cache resident, so the two random table reads are only paid by the edges that survive.
static __global__ void k_build_table(const int64_t* __restrict__ node_index, int64_t kept, int64_t N,
                                     int32_t* __restrict__ table, uint32_t* __restrict__ bits) {
  int64_t j = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= kept) return;
  int64_t v = node_index[j];
  if (v >= 0 && v < N) {
    table[v] = (int32_t)j;
    atomicOr(&bits[v >> 5], 1u << (v & 31));
  }
}

// Small graphs (one block): the -1 / 0 fills of the table, of the mask and of the compaction state and the table
// build itself as ONE launch instead of three memsets and a kernel (a mini-batch step is launch-bound).
constexpr int kSmallNodes = 32768;
constexpr int kSmallThreads = 1024;

static __global__ void __launch_bounds__(kSmallThreads)
    k_kept_init_small(const int64_t* __restrict__ node_index, int kept, int N, int32_t* __restrict__ table,
                      uint32_t* __restrict__ bits, unsigned long long* __restrict__ state, int state_words) {
  const int t = threadIdx.x;
  for (int v = t; v < N; v += kSmallThreads) table[v] = -1;
  for (int j = t; j < N / 32 + 1; j += kSmallThreads) bits[j] = 0u;
  for (int j = t; j < state_words; j += kSmallThreads) state[j] = 0ull;
  __syncthreads();
  for (int j = t; j < kept; j += kSmallThreads) {
    const int64_t v = node_index[j];
    if (v >= 0 && v < N) {
      table[v] = j;
      atomicOr(&bits[v >> 5], 1u << (v & 31));
    }
  }
}

struct KeptPred {
  static constexpr bool kStaged = true;
  struct Payload {
    int64_t r64, c64;
    int32_t r, c;
    float w;
  };
  const int64_t* row;
  const int64_t* col;
  const float* w;
  const int32_t* table;
  const uint32_t* bits;
  int64_t N;
  bool rsl;
  float eps;
  // stage 0: the three streaming loads of the edge (touched once: evict-first keeps the mask / table lines in L2)
  __device__ void stage0(int64_t i, Payload& p) const {
    p.r64 = __ldcs(row + i);
    p.c64 = __ldcs(col + i);
    p.w = w ? __ldcs(w + i) : 1.f;
  }
  // stage 1: range / self-loop / tiny-weight tests and the two membership bits
  __device__ bool stage1(Payload& p) const {
    const int64_t r = p.r64, c = p.c64;
    if (r < 0 || r >= N || c < 0 || c >= N) return false;
    if (rsl && r == c) return false;
    if (w && !(fabsf(p.w) > eps)) return false;
    return ((__ldg(bits + (r >> 5)) >> (r & 31)) & 1u) && ((__ldg(bits + (c >> 5)) >> (c & 31)) & 1u);
  }
  // stage 2: relabel (only the surviving edges touch the table)
  __device__ bool stage2(Payload& p) const {
    p.r = __ldg(table + p.r64);
    p.c = __ldg(table + p.c64);
    return true;
  }
  __device__ bool operator()(int64_t i, Payload& p) const {
    stage0(i, p);
    return stage1(p) && stage2(p);
  }
};
struct KeptEmit {
  int64_t* out_row;
  int64_t* out_col;
  float* out_w;
  int32_t* src;
  __device__ void operator()(int64_t i, int pos, const KeptPred::Payload& p) const {
    __stcs(out_row + pos, (int64_t)p.r);
    __stcs(out_col + pos, (int64_t)p.c);
    if (out_w) __stcs(out_w + pos, p.w);
    if (src) __stcs(src + pos, (int32_t)i);
  }
};

// ------------------------------------------------------------------------------------------
// cluster branch
// ------------------------------------------------------------------------------------------
template <typename KeyT>
static __global__ void k_remap_keys(const int64_t* __restrict__ row, const int64_t* __restrict__ col,
                                    const int64_t* __restrict__ cluster, int64_t E, int64_t N, int64_t K, int cb,
                                    KeyT* __restrict__ keys) {
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= E) return;
  int64_t r = row[i], c = col[i];
  int64_t cr = (r >= 0 && r < N) ? cluster[r] : 0;
  int64_t cc = (c >= 0 && c < N) ? cluster[c] : 0;
  if (cr < 0 || cr >= K) cr = 0;
  if (cc < 0 || cc >= K) cc = 0;
  // (row << cb) | col sorts exactly like row * K + col (cb = bits of K - 1) and decomposes without a 64-bit division
  keys[i] = (KeyT)(((uint64_t)cr << cb) | (uint64_t)cc);
}






static int key_bits_for_u64(uint64_t max_value) {
  int b = 0;
  while (max_value) {
    ++b;
    max_value >>= 1;
  }
  return b < 1 ? 1 : b;
}

static int coarse_col_bits(int64_t K) { return key_bits_for_u64(K > 1 ? (uint64_t)K - 1 : 1); }

// Fused run handling on the sorted keys: a run head (first position of a key) walks its run, combining the member
// weights in sorted (= original, the sort is stable) order; the same pass decides whether the coarse edge survives
// the self-loop / tiny-weight filters.  The count phase stores the combined weight at the head position so that
// the emit phase does not repeat the random gathers.
template <typename KeyT>
struct RunCountPred {
  struct Payload {};
  const KeyT* ks;
  const uint32_t* perm;
  const float* w;  // null when unweighted
  float* comb;     // [E] combined weight at head positions
  int64_t E;
  int cb;          // column bits of the key
  int op;
  bool rsl;
  float eps;
  __device__ bool operator()(int64_t i, Payload&) const {
    const KeyT key = ks[i];
    if (i > 0 && ks[i - 1] == key) return false;
    const uint64_t k64 = (uint64_t)key;
    const bool self = (k64 >> cb) == (k64 & ((1ull << cb) - 1ull));
    if (w == nullptr) return !(rsl && self);
    float acc = w[perm[i]];
    int64_t j = i + 1;
    for (; j < E && ks[j] == key; ++j) {
      const float v = w[perm[j]];
      if (op == TGPB200_SUM || op == TGPB200_MEAN) acc = __fadd_rn(acc, v);
      else if (op == TGPB200_MAX) acc = fmaxf(acc, v);
      else if (op == TGPB200_MIN) acc = fminf(acc, v);
      else acc = __fmul_rn(acc, v);
    }
    if (op == TGPB200_MEAN) acc = __fdiv_rn(acc, (float)(j - i));
    comb[i] = acc;
    if (rsl && self) return false;
    return fabsf(acc) > eps;
  }
};
template <typename KeyT>
struct RunEmitPred {
  struct Payload {
    int64_t cr, cc;
    float w;
  };
  const KeyT* ks;
  const float* comb;  // null when unweighted
  int cb;
  bool rsl;
  float eps;
  __device__ bool operator()(int64_t i, Payload& p) const {
    const KeyT key = ks[i];
    if (i > 0 && ks[i - 1] == key) return false;
    const uint64_t k64 = (uint64_t)key;
    p.cr = (int64_t)(k64 >> cb);
    p.cc = (int64_t)(k64 & ((1ull << cb) - 1ull));
    if (rsl && p.cr == p.cc) return false;
    if (comb) {
      p.w = comb[i];
      if (!(fabsf(p.w) > eps)) return false;
    }
    return true;
  }
};
template <typename KeyT>
struct RunEmit2 {
  const KeyT* ks;
  const uint32_t* perm;
  int64_t E;
  int64_t* out_row;
  int64_t* out_col;
  float* out_w;
  int32_t* run_len;
  int32_t* edge_slot;  // pre-filled with -1
  __device__ void operator()(int64_t i, int pos, const typename RunEmitPred<KeyT>::Payload& p) const {
    out_row[pos] = p.cr;
    out_col[pos] = p.cc;
    if (out_w) out_w[pos] = p.w;
    if (run_len || edge_slot) {
      const KeyT key = ks[i];
      int64_t j = i;
      for (; j < E && ks[j] == key; ++j)
        if (edge_slot) edge_slot[perm[j]] = pos;
      if (run_len) run_len[pos] = (int32_t)(j - i);
    }
  }
};

// Workspace layout shared by the count and emit phases (carved identically in both calls).
template <typename KeyT>
struct CoalescePlan {
  KeyT *keys0, *keys1;
  uint32_t *vals0, *vals1;
  float* comb;
  Workspace sort, tiles;
  CoalescePlan(Workspace& ws, int64_t E) {
    size_t n = (size_t)(E > 0 ? E : 1);
    keys0 = ws.take<KeyT>(n);
    keys1 = ws.take<KeyT>(n);
    vals0 = ws.take<uint32_t>(n);
    vals1 = ws.take<uint32_t>(n);
    comb = ws.take<float>(n);
    sort = ws.sub(radix_sort_workspace_bytes(E));
    tiles = ws.sub(compact_workspace_bytes(E));
  }
};

template <typename KeyT>
static int remap_coalesce_count_impl(const int64_t* row, const int64_t* col, const float* w, int64_t E,
                                     const int64_t* cluster, int64_t N, int64_t K, int op, uint32_t flags, float eps,
                                     int64_t* count_out, Workspace& ws, cudaStream_t st) {
  CoalescePlan<KeyT> pl(ws, E);
  if (!ws.ok) return TGPB200_ERR_WORKSPACE;
  unsigned grid = (unsigned)ceil_div(E, 256);
  const int cb = coarse_col_bits(K);
  launch("k_remap_keys", k_remap_keys<KeyT>, grid, 256, 0, st, row, col, cluster, E, N, K, cb, pl.keys0);
  int bits = 2 * cb;
  bool in1 = false;
  int rc = radix_sort_pairs<KeyT>(pl.keys0, nullptr, pl.vals0, pl.keys1, pl.vals1, E, bits, &in1, pl.sort, st);
  if (rc != TGPB200_OK) return rc;
  RunCountPred<KeyT> pred{in1 ? pl.keys1 : pl.keys0, in1 ? pl.vals1 : pl.vals0, w, pl.comb, E, cb, op,
                          (flags & TGPB200_REMOVE_SELF_LOOPS) != 0, eps};
  return compact_count(pred, E, pl.tiles, nullptr, count_out, st);
}

template <typename KeyT>
static int remap_coalesce_emit_impl(int64_t E, int64_t K, bool weighted, uint32_t flags, float eps, int64_t* out_row,
                                    int64_t* out_col, float* out_w, int32_t* edge_slot, int32_t* run_len,
                                    Workspace& ws, cudaStream_t st) {
  CoalescePlan<KeyT> pl(ws, E);
  if (!ws.ok) return TGPB200_ERR_WORKSPACE;
  const int cb = coarse_col_bits(K);
  int bits = 2 * cb;
  bool in1 = (radix_passes(bits) & 1) != 0;
  const KeyT* ks = in1 ? pl.keys1 : pl.keys0;
  const uint32_t* perm = in1 ? pl.vals1 : pl.vals0;
  if (edge_slot) cudaMemsetAsync(edge_slot, 0xff, (size_t)E * sizeof(int32_t), st);
  RunEmitPred<KeyT> pred{ks, weighted ? pl.comb : nullptr, cb, (flags & TGPB200_REMOVE_SELF_LOOPS) != 0, eps};
  RunEmit2<KeyT> emit{ks, perm, E, out_row, out_col, weighted ? out_w : nullptr, run_len, edge_slot};
  return compact_emit(pred, emit, E, pl.tiles, st);
}

// ------------------------------------------------------------------------------------------
// coalesce backward
// ------------------------------------------------------------------------------------------
static __global__ void k_coalesce_ties(const float* __restrict__ w, const float* __restrict__ out_w,
                                       const int32_t* __restrict__ slot, int64_t E, int* __restrict__ ties) {
  int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= E) return;
  int s = slot[e];
  if (s >= 0 && w[e] == out_w[s]) atomicAdd(&ties[s], 1);
}
// sum / mean: four edges per thread (128-bit slot read and gradient write, the gathers of the four in flight together)
static __global__ void k_coalesce_bwd4(const float* __restrict__ gout, const int32_t* __restrict__ slot,
                                       const int32_t* __restrict__ run_len, int64_t E4, int mean,
                                       float* __restrict__ gin) {
  const int64_t q = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (q >= E4) return;
  const int4 s = reinterpret_cast<const int4*>(slot)[q];
  const int ss[4] = {s.x, s.y, s.z, s.w};
  float g[4];
#pragma unroll
  for (int j = 0; j < 4; ++j) g[j] = ss[j] >= 0 ? __ldg(gout + ss[j]) : 0.f;
  if (mean) {
    int len[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) len[j] = ss[j] >= 0 ? __ldg(run_len + ss[j]) : 1;
#pragma unroll
    for (int j = 0; j < 4; ++j) g[j] = g[j] / (float)len[j];
  }
  reinterpret_cast<float4*>(gin)[q] = make_float4(g[0], g[1], g[2], g[3]);
}

static __global__ void k_coalesce_bwd(const float* __restrict__ w, const float* __restrict__ out_w,
                                      const float* __restrict__ gout, const int32_t* __restrict__ slot,
                                      const int32_t* __restrict__ run_len, const float* __restrict__ run_aux,
                                      const int* __restrict__ ties, int64_t E, int op, float* __restrict__ gin) {
  int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= E) return;
  int s = slot[e];
  float g = 0.f;
  if (s >= 0) {
    g = gout[s];
    if (op == TGPB200_MEAN) g = g / (float)run_len[s];
    else if (op == TGPB200_MAX || op == TGPB200_MIN) g = (w[e] == out_w[s]) ? g / (float)ties[s] : 0.f;
    else if (op == TGPB200_MUL) {
      if (run_aux) {  // run_len = zero members of the run, run_aux = product of the others: exact product rule
        const int z = run_len[s];
        g = z == 0 ? g * out_w[s] / w[e] : ((z == 1 && w[e] == 0.f) ? g * run_aux[s] : 0.f);
      } else {
        g = (w[e] != 0.f) ? g * out_w[s] / w[e] : 0.f;
      }
    }
  }
  gin[e] = g;
}

// ------------------------------------------------------------------------------------------
// Deterministic segmented sums (degree / normalisation partials): no floating-point atomics.
//   out[k] = sum of val(i) over the positions i with key(i) == k, k in [0, K)
// For a non-decreasing key sequence (coarse edge lists are row-sorted: the cluster path sorts them, the kept-node
// path keeps the order of a row-sorted input) a key's positions form one run, and a SEGMENTED scan in double
// precision sums every run on its own: a position starts a segment where its key differs from the one before, and
// the running sum restarts there.  Fixed reduce-then-scan structure (tile summaries -> sequential spine -> tile
// down-sweep): bitwise reproducible, perfectly load-balanced whatever the run lengths (a power-law hub row is just a
// long run), and every partial sum holds values of one run only, so the error of out[k] is bounded by its own
// sum of |values| (|err| <= ~n_k 2^-53 sum|values| before the final rounding to fp32), whatever precedes it in the
// sequence.  Other key sequences are first grouped with the stable radix sort.
// `n_dev`, when given, is the device-side element count (<= the launch capacity n).
//
// (flag, value) pairs combine as  a . b = (a.f | b.f, b.f ? b.v : a.v + b.v): the flag says that a segment starts
// inside the span, the value is the sum from the span's last segment start (or from its beginning) to its end.
// ------------------------------------------------------------------------------------------
constexpr int kDsThreads = 256;
constexpr int kDsItems = 8;
constexpr int kDsTile = kDsThreads * kDsItems;
constexpr int kDsWarps = kDsThreads / 32;

struct KeyOfArray64 {
  const int64_t* k;
  __device__ int64_t operator()(int64_t i) const { return k[i]; }
};
struct KeyOfArray32 {
  const uint32_t* k;
  __device__ int64_t operator()(int64_t i) const { return (int64_t)k[i]; }
};

// key at position i, -1 when i is past the end or the key is outside [0, K)
template <typename KeyF>
__device__ __forceinline__ int64_t dsum_key(KeyF key, int64_t i, int64_t n, int64_t K) {
  if (i < 0 || i >= n) return -1;
  const int64_t k = key(i);
  return (k < 0 || k >= K) ? -1 : k;
}

// Tile layout of all passes: warp w of the block owns the 256 consecutive positions [tile + 256 w, +256) and reads
// them in 8 rounds of 32 (round r, lane l -> position 256 w + 32 r + l): every load is a full coalesced line.
// Segmented inclusive scan over the warp's positions, round after round.  k: keys (-1 = none), v: values (0 where
// k = -1), k_before: key of the position before the window (lane 0; -1 if none).  inc[r] is the sum from the latest
// segment start in the window at or before the position (from the window's start if there is none, fl[r] = false);
// any / tail: the window's summary.  The segment starts of a round are one ballot: lane l adds the partial of lane
// l - o unless a segment starts in lanes (l - o, l].
__device__ __forceinline__ void dsum_warp_scan(const int64_t (&k)[kDsItems], const double (&v)[kDsItems],
                                               int64_t k_before, double (&inc)[kDsItems], bool (&fl)[kDsItems],
                                               bool& any, double& tail) {
  const int lane = threadIdx.x & 31;
  any = false;
  tail = 0.0;
#pragma unroll
  for (int r = 0; r < kDsItems; ++r) {
    int64_t prev = __shfl_up_sync(kFull, k[r], 1);
    const int64_t last_prev = __shfl_sync(kFull, r > 0 ? k[r > 0 ? r - 1 : 0] : k_before, r > 0 ? 31 : 0);
    if (lane == 0) prev = last_prev;
    const unsigned heads = __ballot_sync(kFull, k[r] >= 0 && k[r] != prev);
    double x = v[r];
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const double t = __shfl_up_sync(kFull, x, o);
      if (lane >= o && ((heads >> (lane - o + 1)) & ((1u << o) - 1u)) == 0u) x = t + x;
    }
    const bool f = (heads & ((2u << lane) - 1u)) != 0u;  // a segment starts in lanes [0, lane]
    inc[r] = f ? x : tail + x;
    fl[r] = f || any;
    const double x31 = __shfl_sync(kFull, x, 31);
    tail = heads ? x31 : tail + x31;
    any = any || heads != 0u;
  }
}

// Summary of one tile (keys / values in the tile layout, k_before = key before the warp's window): per warp, whether
// a segment starts in its window and the sum of the values from the last such start (from the window's start if
// none); the warps folded in warp order.  Shared by every producer of tile summaries, so they agree bit for bit.
__device__ __forceinline__ void dsum_tile_summary(const int64_t (&k)[kDsItems], const double (&v)[kDsItems],
                                                  int64_t k_before, double* __restrict__ tile_sums,
                                                  uint32_t* __restrict__ tile_flags) {
  __shared__ double s_tail[kDsWarps];
  __shared__ int s_any[kDsWarps];
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  unsigned last = 0;  // 1 + window position of the thread's last segment start, 0 if none
#pragma unroll
  for (int r = 0; r < kDsItems; ++r) {
    int64_t prev = __shfl_up_sync(kFull, k[r], 1);
    const int64_t last_prev = __shfl_sync(kFull, r > 0 ? k[r > 0 ? r - 1 : 0] : k_before, r > 0 ? 31 : 0);
    if (lane == 0) prev = last_prev;
    if (k[r] >= 0 && k[r] != prev) last = (unsigned)(r * 32 + lane) + 1u;
  }
  const unsigned head = __reduce_max_sync(kFull, last);
  double s = 0.0;
#pragma unroll
  for (int r = 0; r < kDsItems; ++r)
    if ((unsigned)(r * 32 + lane) + 1u >= head) s += v[r];
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(kFull, s, o);
  if (lane == 0) {
    s_tail[w] = s;
    s_any[w] = head != 0u;
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    bool a = false;
    double t = 0.0;
    for (int q = 0; q < kDsWarps; ++q) {
      t = s_any[q] ? s_tail[q] : t + s_tail[q];
      a = a || s_any[q];
    }
    tile_sums[blockIdx.x] = t;
    tile_flags[blockIdx.x] = a ? 1u : 0u;
  }
}

template <typename KeyF, typename ValF>
static __global__ void __launch_bounds__(kDsThreads)
    k_dsum_reduce(KeyF key, ValF val, int64_t n, const int64_t* __restrict__ n_dev, int64_t K,
                  double* __restrict__ tile_sums, uint32_t* __restrict__ tile_flags) {
  if (n_dev) n = min(n, *n_dev);
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  const int64_t wbase = (int64_t)blockIdx.x * kDsTile + (int64_t)w * (32 * kDsItems);
  int64_t k[kDsItems];
  double v[kDsItems];
#pragma unroll
  for (int r = 0; r < kDsItems; ++r) {
    const int64_t i = wbase + r * 32 + lane;
    k[r] = dsum_key(key, i, n, K);
    v[r] = k[r] >= 0 ? (double)val(i) : 0.0;
  }
  const int64_t k_before = lane == 0 ? dsum_key(key, wbase - 1, n, K) : -1;
  dsum_tile_summary(k, v, k_before, tile_sums, tile_flags);
}

// one block: segmented exclusive scan of the tile summaries in place (tile_sums[t] becomes the running sum of the
// segment open at the start of tile t), 1024 tiles per round, rounds in order with the carry between them
static __global__ void __launch_bounds__(1024) k_dsum_spine(double* __restrict__ tile_sums,
                                                            const uint32_t* __restrict__ tile_flags, int nt) {
  __shared__ double s_tail[32], s_in[32];
  __shared__ int s_any[32];
  __shared__ double s_carry;
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  double carry = 0.0;
  for (int start = 0; start < nt; start += blockDim.x) {
    const int i = start + threadIdx.x;
    double x = i < nt ? tile_sums[i] : 0.0;
    const unsigned heads = __ballot_sync(kFull, i < nt && tile_flags[i] != 0u);
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const double t = __shfl_up_sync(kFull, x, o);
      if (lane >= o && ((heads >> (lane - o + 1)) & ((1u << o) - 1u)) == 0u) x = t + x;
    }
    const bool f = (heads & ((2u << lane) - 1u)) != 0u;
    if (lane == 31) {
      s_tail[w] = x;
      s_any[w] = heads != 0u;
    }
    __syncthreads();
    if (w == 0) {  // running sum entering every warp: the round's carry, then the warps before it in order
      double y = s_tail[lane];
      const unsigned wh = __ballot_sync(kFull, s_any[lane] != 0);
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        const double t = __shfl_up_sync(kFull, y, o);
        if (lane >= o && ((wh >> (lane - o + 1)) & ((1u << o) - 1u)) == 0u) y = t + y;
      }
      const double ye = __shfl_up_sync(kFull, y, 1);
      const bool fe = (wh & ((1u << lane) - 1u)) != 0u;  // a segment starts in the warps before this one
      s_in[lane] = lane == 0 ? carry : (fe ? ye : carry + ye);
      if (lane == 31) s_carry = wh ? y : carry + y;
    }
    __syncthreads();
    const double c = s_in[w];
    const double incl = f ? x : c + x;
    const double before = __shfl_up_sync(kFull, incl, 1);
    if (i < nt) tile_sums[i] = lane == 0 ? c : before;
    carry = s_carry;
    __syncthreads();
  }
}

// down-sweep: segmented running sum at every position; the last position of a key's run writes the run's sum
template <typename KeyF, typename ValF>
static __global__ void __launch_bounds__(kDsThreads)
    k_dsum_down(KeyF key, ValF val, int64_t n, const int64_t* __restrict__ n_dev, int64_t K,
                const double* __restrict__ tile_off, float* __restrict__ out) {
  __shared__ double s_tail[kDsWarps];
  __shared__ int s_any[kDsWarps];
  if (n_dev) n = min(n, *n_dev);
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  const int64_t wbase = (int64_t)blockIdx.x * kDsTile + (int64_t)w * (32 * kDsItems);
  int64_t k[kDsItems];
  double v[kDsItems], inc[kDsItems];
  bool fl[kDsItems];
#pragma unroll
  for (int r = 0; r < kDsItems; ++r) {
    const int64_t i = wbase + r * 32 + lane;
    k[r] = dsum_key(key, i, n, K);
    v[r] = k[r] >= 0 ? (double)val(i) : 0.0;
  }
  // keys just outside the warp's window
  const int64_t k_before = lane == 0 ? dsum_key(key, wbase - 1, n, K) : -1;
  const int64_t k_after = lane == 31 ? dsum_key(key, wbase + 32 * kDsItems, n, K) : -1;
  bool any;
  double tail;
  dsum_warp_scan(k, v, k_before, inc, fl, any, tail);
  if (lane == 0) {
    s_tail[w] = tail;
    s_any[w] = any;
  }
  __syncthreads();
  double c = tile_off[blockIdx.x];  // running sum entering the warp's window
  for (int q = 0; q < w; ++q) c = s_any[q] ? s_tail[q] : c + s_tail[q];
#pragma unroll
  for (int r = 0; r < kDsItems; ++r) {
    int64_t next = __shfl_down_sync(kFull, k[r], 1);
    const int64_t first_next =
        __shfl_sync(kFull, r + 1 < kDsItems ? k[r + 1 < kDsItems ? r + 1 : r] : k_after, r + 1 < kDsItems ? 0 : 31);
    if (lane == 31) next = first_next;
    const int64_t kk = k[r];
    if (kk >= 0 && next != kk) out[kk] = (float)(fl[r] ? inc[r] : c + inc[r]);
  }
}

template <typename KeyF>
static __global__ void k_fill_keys32(KeyF key, int64_t n, const int64_t* __restrict__ n_dev, int64_t K,
                                     uint32_t* __restrict__ keys) {
  if (n_dev) n = min(n, *n_dev);
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const int64_t k = key(i);
  keys[i] = (k < 0 || k >= K) ? (uint32_t)K : (uint32_t)k;  // out-of-range keys sort last and match no run
}

// grouped (unsorted-key) path: the values are evaluated once in position order (coalesced operand reads) and carried
// into key order as the payload of the stable sort; the scan passes read them linearly
template <typename ValF>
static __global__ void k_eval_vals(ValF val, int64_t n, const int64_t* __restrict__ n_dev, float* __restrict__ out) {
  if (n_dev) n = min(n, *n_dev);
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) out[i] = val(i);
}
struct ValOfArray {
  const float* a;
  __device__ float operator()(int64_t i) const { return a[i]; }
};

// Scratch of one det_segment_sum of n values: the tile summaries of the scan passes, and for unsorted keys the 32-bit
// keys, the values in position order and the stable sort that groups them.  Nothing in it is per segment: the sums
// go straight to `out`.
struct DetSumScratch {
  double* tiles;
  uint32_t* tile_flags;
  uint32_t *keys0, *keys1, *vals0, *vals1;
  float* ev;
  Workspace sort;
  DetSumScratch(Workspace& ws, int64_t n) {
    const size_t m = (size_t)(n > 0 ? n : 1);
    tiles = ws.take<double>(m / kDsTile + 2);
    tile_flags = ws.take<uint32_t>(m / kDsTile + 2);
    keys0 = ws.take<uint32_t>(m);
    keys1 = ws.take<uint32_t>(m);
    vals0 = ws.take<uint32_t>(m);
    vals1 = ws.take<uint32_t>(m);
    ev = ws.take<float>(m);
    sort = ws.sub(radix_sort_workspace_bytes(n));
  }
};

// tiles_ready: `tiles` / `tile_flags` already hold the tile summaries (a producer kernel with the tile layout of
// k_dsum_reduce that calls dsum_tile_summary)
template <typename KeyF, typename ValF>
static void segmented_run_sums(KeyF key, ValF val, int64_t n, const int64_t* n_dev, int64_t K, double* tiles,
                               uint32_t* tile_flags, float* out, cudaStream_t st, bool tiles_ready = false) {
  const int nt = (int)ceil_div(n, kDsTile);
  cudaMemsetAsync(out, 0, (size_t)K * sizeof(float), st);  // keys without a run sum to 0
  if (!tiles_ready)
    launch("k_dsum_reduce", k_dsum_reduce<KeyF, ValF>, nt, kDsThreads, 0, st, key, val, n, n_dev, K, tiles,
           tile_flags);
  launch("k_dsum_spine", k_dsum_spine, 1, 1024, 0, st, tiles, tile_flags, nt);
  launch("k_dsum_down", k_dsum_down<KeyF, ValF>, nt, kDsThreads, 0, st, key, val, n, n_dev, K, tiles, out);
}

// A value functor that gathers (`static constexpr bool kCostly = true`) is evaluated ONCE into a float array and the
// two scan passes read the array: the degree backward's dependent gather deg[other[e]] otherwise runs in both the
// tile-sum and the down-sweep pass (ncu: down-sweep 1.37 ms against 0.45 ms for the plain-array form on 100 M edges).
template <typename V, typename = void>
struct val_is_costly : std::false_type {};
template <typename V>
struct val_is_costly<V, std::void_t<decltype(V::kCostly)>> : std::integral_constant<bool, V::kCostly> {};

// s.keys0 (32-bit, invalid keys = K) and s.ev (values in position order) are ready: group by key, then run sums.
// The values themselves ride through the stable sort as its 32-bit payload: no index payload, no gather afterwards
// (a random 4-byte gather over 100 M values cost 1.5 ms, as much as two sort passes).  s.keys0 is overwritten.
static int grouped_sums_of(const DetSumScratch& s, int64_t n, const int64_t* n_dev, int64_t K, float* out,
                           cudaStream_t st) {
  bool in1 = false;
  int rc = radix_sort_pairs<uint32_t>(s.keys0, reinterpret_cast<uint32_t*>(s.ev), s.vals0, s.keys1, s.vals1, n,
                                      key_bits_for_u64((uint64_t)K), &in1, s.sort, st, n_dev);
  if (rc != TGPB200_OK) return rc;
  const float* sv = reinterpret_cast<const float*>(in1 ? s.vals1 : s.vals0);
  segmented_run_sums(KeyOfArray32{in1 ? s.keys1 : s.keys0}, ValOfArray{sv}, n, n_dev, K, s.tiles, s.tile_flags, out,
                     st);
  return launch_status();
}

// s: carved for at least n values.
template <typename KeyF, typename ValF>
static int det_segment_sum(KeyF key, ValF val, int64_t n, const int64_t* n_dev, int64_t K, bool keys_sorted, float* out,
                           const DetSumScratch& s, cudaStream_t st) {
  if (K <= 0) return TGPB200_OK;
  if (n <= 0) {
    cudaMemsetAsync(out, 0, (size_t)K * sizeof(float), st);
    return launch_status();
  }
  if (keys_sorted) {
    if constexpr (val_is_costly<ValF>::value) {
      launch("k_eval_vals", k_eval_vals<ValF>, (unsigned)ceil_div(n, 256), 256, 0, st, val, n, n_dev, s.ev);
      segmented_run_sums(key, ValOfArray{s.ev}, n, n_dev, K, s.tiles, s.tile_flags, out, st);
    } else {
      segmented_run_sums(key, val, n, n_dev, K, s.tiles, s.tile_flags, out, st);
    }
    return launch_status();
  }
  const unsigned grid = (unsigned)ceil_div(n, 256);
  launch("k_fill_keys32", k_fill_keys32<KeyF>, grid, 256, 0, st, key, n, n_dev, K, s.keys0);
  launch("k_eval_vals", k_eval_vals<ValF>, grid, 256, 0, st, val, n, n_dev, s.ev);
  return grouped_sums_of(s, n, n_dev, K, out, st);
}

static __global__ void k_rows_sorted(const int64_t* __restrict__ row, int64_t E, int32_t* __restrict__ sorted_out) {
  int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (e + 1 < E && row[e + 1] < row[e]) *sorted_out = 0;
}

// ------------------------------------------------------------------------------------------
// degree / max-weight normalisation
// ------------------------------------------------------------------------------------------
__device__ __forceinline__ float dinv_of(float deg, float eps) { return 1.0f / sqrtf(fmaxf(deg, eps)); }

struct DegVal {
  const float* w;
  __device__ float operator()(int64_t e) const { return w ? w[e] : 1.f; }
};
// gradient w.r.t. dinv: row side sum_{e: row = v} g w dinv[col], column side sum_{e: col = v} g w dinv[row]
struct DegBwdVal {
  static constexpr bool kCostly = true;  // dependent gather: evaluated once into an array (det_segment_sum)
  const int64_t* other;  // the opposite endpoint of the key
  const float* w;
  const float* deg;
  const float* gout;
  int64_t K;
  float eps;
  __device__ float operator()(int64_t e) const {
    const int64_t o = other[e];
    if (o < 0 || o >= K) return 0.f;
    return gout[e] * (w ? w[e] : 1.f) * dinv_of(deg[o], eps);
  }
};
struct ProdVal {
  const float* a;
  const float* b;
  __device__ float operator()(int64_t e) const { return a[e] * b[e]; }
};
struct ArrVal {
  const float* a;
  __device__ float operator()(int64_t i) const { return a[i]; }
};

// Both sides of the degree backward from ONE pass over the edges (row-sorted input): the row-side values
// g w dinv[col], the column-side values g w dinv[row] and the 32-bit column keys of the grouped sum.  Same products in
// the same order as DegBwdVal, so the sums are bit-identical to the two-functor form (3 kernels, each edge read 3 x).
// It also leaves the row-side tile summaries behind (one k_dsum_reduce pass less).
static __global__ void __launch_bounds__(kDsThreads)
    k_deg_bwd_prepare(const int64_t* __restrict__ row, const int64_t* __restrict__ col, const float* __restrict__ w,
                      const float* __restrict__ deg, const float* __restrict__ gout, int64_t E,
                      const int64_t* __restrict__ E_dev, int64_t K, float eps, float* __restrict__ ev_row,
                      float* __restrict__ ev_col, uint32_t* __restrict__ keys_col, double* __restrict__ tile_sums,
                      uint32_t* __restrict__ tile_flags) {
  // tile layout, keys and values of k_dsum_reduce over (row, ev_row), so the summaries agree with it bit for bit
  if (E_dev) E = min(E, *E_dev);
  const int lane = threadIdx.x & 31, wp = threadIdx.x >> 5;
  const int64_t wbase = (int64_t)blockIdx.x * kDsTile + (int64_t)wp * (32 * kDsItems);
  int64_t r[kDsItems], c[kDsItems];
  float g[kDsItems];
#pragma unroll
  for (int k = 0; k < kDsItems; ++k) {
    const int64_t e = wbase + k * 32 + lane;
    r[k] = e < E ? row[e] : -1;
    c[k] = e < E ? col[e] : -1;
    g[k] = e < E ? gout[e] * (w ? w[e] : 1.f) : 0.f;
  }
  float dr[kDsItems], dc[kDsItems];
#pragma unroll
  for (int k = 0; k < kDsItems; ++k) {
    dr[k] = (r[k] >= 0 && r[k] < K) ? __ldg(deg + r[k]) : 0.f;
    dc[k] = (c[k] >= 0 && c[k] < K) ? __ldg(deg + c[k]) : 0.f;
  }
  int64_t kr[kDsItems];
  double vr[kDsItems];
#pragma unroll
  for (int k = 0; k < kDsItems; ++k) {
    const int64_t e = wbase + k * 32 + lane;
    const bool okr = r[k] >= 0 && r[k] < K, okc = c[k] >= 0 && c[k] < K;
    kr[k] = okr ? r[k] : -1;
    vr[k] = 0.0;
    if (e >= E) continue;
    const float v = okc ? g[k] * dinv_of(dc[k], eps) : 0.f;  // keyed by row, opposite endpoint = col
    ev_row[e] = v;
    ev_col[e] = okr ? g[k] * dinv_of(dr[k], eps) : 0.f;      // keyed by col, opposite endpoint = row
    keys_col[e] = okc ? (uint32_t)c[k] : (uint32_t)K;
    if (okr) vr[k] = (double)v;
  }
  const int64_t k_before = lane == 0 ? dsum_key(KeyOfArray64{row}, wbase - 1, E, K) : -1;
  dsum_tile_summary(kr, vr, k_before, tile_sums, tile_flags);
}

static __global__ void k_deg_apply(const int64_t* __restrict__ row, const int64_t* __restrict__ col,
                                   const float* __restrict__ w, const float* __restrict__ deg, int64_t E,
                                   const int64_t* __restrict__ E_dev, int64_t K, float eps, float* __restrict__ w_out) {
  if (E_dev) E = min(E, *E_dev);
  int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= E) return;
  int64_t r = row[e], c = col[e];
  if (r < 0 || r >= K || c < 0 || c >= K) { w_out[e] = 0.f; return; }
  float v = w ? w[e] : 1.f;
  w_out[e] = __fmul_rn(__fmul_rn(v, dinv_of(deg[r], eps)), dinv_of(deg[c], eps));
}
static __global__ void k_add_vec(const float* __restrict__ a, const float* __restrict__ b, int64_t n,
                                 float* __restrict__ out) {
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) out[i] = __fadd_rn(a[i], b[i]);
}
static __global__ void k_deg_bwd_apply(const int64_t* __restrict__ row, const int64_t* __restrict__ col,
                                       const float* __restrict__ deg, const float* __restrict__ gout,
                                       const float* __restrict__ gdinv, int64_t E, const int64_t* __restrict__ E_dev,
                                       int64_t K, float eps, float* __restrict__ gw) {
  if (E_dev) E = min(E, *E_dev);
  int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= E) return;
  int64_t r = row[e], c = col[e];
  if (r < 0 || r >= K || c < 0 || c >= K) { gw[e] = 0.f; return; }
  float dr = dinv_of(deg[r], eps), dc = dinv_of(deg[c], eps);
  float gdeg = (deg[r] >= eps) ? -0.5f * gdinv[r] * dr * dr * dr : 0.f;
  gw[e] = gout[e] * dr * dc + gdeg;
}

// Workspace shared by the edge-normalisation entry points (tgpb200_edge_norm_workspace_bytes(E, K)): the two sides
// of the degree backward, the sums over the E edges by row and by column, and the weight-norm backward's sum of the
// per-node values by graph (its K is max(pooled nodes, graphs)).
struct EdgeNormLayout {
  float *part_row, *part_col;  // [K]
  DetSumScratch row, col;      // E values each
  DetSumScratch nodes;         // K values
  EdgeNormLayout(Workspace& ws, int64_t E, int64_t K)
      : part_row(ws.take<float>((size_t)(K > 0 ? K : 1))),
        part_col(ws.take<float>((size_t)(K > 0 ? K : 1))),
        row(ws, E),
        col(ws, E),
        nodes(ws, K) {}
};

static __global__ void k_wn_max(const int64_t* __restrict__ row, const float* __restrict__ w,
                                const int64_t* __restrict__ batch, int64_t E, const int64_t* __restrict__ E_dev,
                                int64_t G, float* __restrict__ mx) {
  if (E_dev) E = min(E, *E_dev);
  int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= E) return;
  int64_t g = batch[row[e]];
  if (g < 0 || g >= G) return;
  float a = fabsf(w[e]);
  if (a == a) atomicMax(reinterpret_cast<int*>(&mx[g]), __float_as_int(a));  // |w| >= 0: int order == float order
}
static __global__ void k_wn_apply(const int64_t* __restrict__ row, const float* __restrict__ w,
                                  const int64_t* __restrict__ batch, const float* __restrict__ mx, int64_t E,
                                  const int64_t* __restrict__ E_dev, int64_t G, int32_t* __restrict__ arg,
                                  float* __restrict__ w_out) {
  if (E_dev) E = min(E, *E_dev);
  int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= E) return;
  int64_t g = batch[row[e]];
  if (g < 0 || g >= G) { w_out[e] = w[e]; return; }
  float m = mx[g];
  if (arg && fabsf(w[e]) == m) atomicMin(&arg[g], (int)e);
  w_out[e] = __fdiv_rn(w[e], m == 0.f ? 1.f : m);
}
static __global__ void k_wn_bwd_apply(const int64_t* __restrict__ row, const float* __restrict__ w,
                                      const int64_t* __restrict__ batch, const float* __restrict__ mx,
                                      const int32_t* __restrict__ arg, const float* __restrict__ gout,
                                      const float* __restrict__ acc, int64_t E, const int64_t* __restrict__ E_dev,
                                      int64_t G, float* __restrict__ gw) {
  if (E_dev) E = min(E, *E_dev);
  int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= E) return;
  int64_t g = batch[row[e]];
  if (g < 0 || g >= G) { gw[e] = gout[e]; return; }
  float m = mx[g];
  float v = gout[e] / (m == 0.f ? 1.f : m);
  if (m != 0.f && arg[g] == (int)e) v += (w[e] < 0.f ? -1.f : 1.f) * (-acc[g] / (m * m));
  gw[e] = v;
}

}  // namespace tgp

using namespace tgp;

extern "C" {

size_t tgpb200_remap_coalesce_workspace_bytes(int64_t E, int64_t K) {
  if (2 * coarse_col_bits(K) <= 32) return layout_bytes<CoalescePlan<uint32_t>>(E);
  return layout_bytes<CoalescePlan<uint64_t>>(E);
}

int tgpb200_remap_coalesce_count(const int64_t* row, const int64_t* col, const float* edge_weight, int64_t E,
                                 const int64_t* cluster_index, int64_t N, int64_t K, int op, uint32_t flags, float eps,
                                 int64_t* count_out, void* workspace, size_t workspace_bytes,
                                 tgpb200_stream_t stream) {
  if (E < 0 || N < 0 || K < 0 || E >= INT32_MAX || K >= INT32_MAX || !count_out) return TGPB200_ERR_INVALID;
  if (op < TGPB200_SUM || op > TGPB200_MUL) return TGPB200_ERR_INVALID;
  cudaStream_t st = (cudaStream_t)stream;
  if (E == 0) {
    cudaMemsetAsync(count_out, 0, sizeof(int64_t), st);
    return launch_status();
  }
  if (!row || !col || !cluster_index || K == 0) return TGPB200_ERR_INVALID;
  Workspace ws(workspace, workspace_bytes);
  if (2 * coarse_col_bits(K) <= 32)
    return remap_coalesce_count_impl<uint32_t>(row, col, edge_weight, E, cluster_index, N, K, op, flags, eps,
                                               count_out, ws, st);
  return remap_coalesce_count_impl<uint64_t>(row, col, edge_weight, E, cluster_index, N, K, op, flags, eps, count_out,
                                             ws, st);
}

int tgpb200_remap_coalesce_emit(int64_t E, int64_t K, int weighted, uint32_t flags, float eps, int64_t* out_row,
                                int64_t* out_col, float* out_weight, int32_t* edge_slot, int32_t* run_len,
                                void* workspace, size_t workspace_bytes, tgpb200_stream_t stream) {
  if (E < 0 || K < 0 || E >= INT32_MAX || K >= INT32_MAX) return TGPB200_ERR_INVALID;
  if (E == 0) return TGPB200_OK;
  if (!out_row || !out_col || K == 0 || (weighted && !out_weight)) return TGPB200_ERR_INVALID;
  Workspace ws(workspace, workspace_bytes);
  cudaStream_t st = (cudaStream_t)stream;
  if (2 * coarse_col_bits(K) <= 32)
    return remap_coalesce_emit_impl<uint32_t>(E, K, weighted != 0, flags, eps, out_row, out_col, out_weight,
                                              edge_slot, run_len, ws, st);
  return remap_coalesce_emit_impl<uint64_t>(E, K, weighted != 0, flags, eps, out_row, out_col, out_weight, edge_slot,
                                            run_len, ws, st);
}

// Workspace of tgpb200_filter_relabel_onepass: the relabel table, the kept-node bits and the compaction's tile states.
struct KeptLayout {
  int32_t* table;
  uint32_t* bits;
  unsigned long long* state;
  KeptLayout(Workspace& ws, int64_t E, int64_t N) {
    table = ws.take<int32_t>((size_t)(N > 0 ? N : 1));
    bits = ws.take<uint32_t>((size_t)(N / 32 + 1));
    state = ws.take<unsigned long long>(compact_onepass_state_words(E));
  }
};

size_t tgpb200_filter_relabel_onepass_workspace_bytes(int64_t E, int64_t N) { return layout_bytes<KeptLayout>(E, N); }

// Single-pass form: the edge list is read once; outputs have capacity E and *count_out gets the survivor count.
int tgpb200_filter_relabel_onepass(const int64_t* row, const int64_t* col, const float* edge_weight, int64_t E,
                                   const int64_t* node_index, int64_t kept, int64_t N, uint32_t flags, float eps,
                                   int64_t* out_row, int64_t* out_col, float* out_weight, int32_t* src_edge,
                                   int64_t* count_out, void* workspace, size_t workspace_bytes,
                                   tgpb200_stream_t stream) {
  if (E < 0 || kept < 0 || N < 0 || E >= INT32_MAX || N >= INT32_MAX || !count_out) return TGPB200_ERR_INVALID;
  if (E > 0 && (!row || !col || !out_row || !out_col)) return TGPB200_ERR_INVALID;
  if (edge_weight && E > 0 && !out_weight) return TGPB200_ERR_INVALID;
  if (kept > 0 && !node_index) return TGPB200_ERR_INVALID;
  cudaStream_t st = (cudaStream_t)stream;
  Workspace ws(workspace, workspace_bytes);
  const KeptLayout l(ws, E, N);
  if (!ws.ok) return TGPB200_ERR_WORKSPACE;
  int32_t* table = l.table;
  uint32_t* bits = l.bits;
  unsigned long long* state = l.state;
  const size_t state_words = compact_onepass_state_words(E);
  const bool small = N <= kSmallNodes && kept <= kSmallNodes && state_words <= 4096;
  if (small) {
    launch("k_kept_init_small", k_kept_init_small, 1, kSmallThreads, 0, st, node_index, (int)kept, (int)N, table, bits, state,
           (int)state_words);
  } else {
    cudaMemsetAsync(table, 0xff, (size_t)(N > 0 ? N : 1) * sizeof(int32_t), st);
    cudaMemsetAsync(bits, 0, (size_t)(N / 32 + 1) * sizeof(uint32_t), st);
    if (kept > 0)
      launch("k_build_table", k_build_table, (unsigned)ceil_div(kept, 256), 256, 0, st, node_index, kept, N, table, bits);
  }
  KeptPred pred{row, col, edge_weight, table, bits, N, (flags & TGPB200_REMOVE_SELF_LOOPS) != 0, eps};
  KeptEmit emit{out_row, out_col, edge_weight ? out_weight : nullptr, src_edge};
  return compact_onepass_on(pred, emit, E, count_out, state, small, st);
}

// grad_in[e] = grad_out[j] for the surviving edges (src_edge[j] == e), 0 elsewhere.
static __global__ void k_unfilter(const float* __restrict__ gout, const int32_t* __restrict__ src, int64_t cnt,
                                  const int64_t* __restrict__ cnt_dev, float* __restrict__ gin) {
  if (cnt_dev) cnt = min(cnt, *cnt_dev);
  int64_t j = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (j < cnt) gin[src[j]] = gout[j];
}

static __global__ void __launch_bounds__(kSmallThreads)
    k_unfilter_small(const float* __restrict__ gout, const int32_t* __restrict__ src, int cnt,
                     const int64_t* __restrict__ cnt_dev, int E, float* __restrict__ gin) {
  if (cnt_dev) cnt = (int)min((int64_t)cnt, *cnt_dev);
  for (int e = threadIdx.x; e < E; e += kSmallThreads) gin[e] = 0.f;
  __syncthreads();
  for (int j = threadIdx.x; j < cnt; j += kSmallThreads) gin[src[j]] = gout[j];
}

int tgpb200_filter_relabel_bwd(const float* grad_out, const int32_t* src_edge, int64_t num_out,
                               const int64_t* num_out_dev, int64_t E, float* grad_in, tgpb200_stream_t stream) {
  if (num_out < 0 || E < 0) return TGPB200_ERR_INVALID;
  if (E == 0) return TGPB200_OK;
  if (!grad_in || (num_out > 0 && (!grad_out || !src_edge))) return TGPB200_ERR_INVALID;
  cudaStream_t st = (cudaStream_t)stream;
  if (E <= kSmallNodes && num_out <= kSmallNodes) {  // zero fill + scatter as one launch
    launch("k_unfilter_small", k_unfilter_small, 1, kSmallThreads, 0, st, grad_out, src_edge, (int)num_out, num_out_dev, (int)E,
           grad_in);
    return launch_status();
  }
  cudaMemsetAsync(grad_in, 0, (size_t)E * sizeof(float), st);
  if (num_out > 0) launch("k_unfilter", k_unfilter, (unsigned)ceil_div(num_out, 256), 256, 0, st, grad_out, src_edge, num_out, num_out_dev, grad_in);
  return launch_status();
}

// Workspace of tgpb200_coalesce_bwd: the tie counts of MAX / MIN runs (the other ops need none).
struct CoalesceBwdLayout {
  int* ties;
  CoalesceBwdLayout(Workspace& ws, int64_t num_out, int op) {
    ties = (op == TGPB200_MAX || op == TGPB200_MIN) ? ws.take<int>((size_t)(num_out > 0 ? num_out : 1)) : nullptr;
  }
};

size_t tgpb200_coalesce_bwd_workspace_bytes(int64_t E, int64_t num_out, int op) {
  (void)E;
  return layout_bytes<CoalesceBwdLayout>(num_out, op);
}

int tgpb200_coalesce_bwd(const float* edge_weight, const float* out_weight, const float* grad_out,
                         const int32_t* edge_slot, const int32_t* run_len, const float* run_aux, int64_t E,
                         int64_t num_out, int op, float* grad_in, void* workspace, size_t workspace_bytes,
                         tgpb200_stream_t stream) {
  if (E < 0 || num_out < 0 || op < TGPB200_SUM || op > TGPB200_MUL) return TGPB200_ERR_INVALID;
  if (E == 0) return TGPB200_OK;
  if (!edge_slot || !grad_in || (num_out > 0 && !grad_out)) return TGPB200_ERR_INVALID;
  if (op == TGPB200_MEAN && !run_len) return TGPB200_ERR_INVALID;
  if (op >= TGPB200_MAX && (!edge_weight || !out_weight)) return TGPB200_ERR_INVALID;
  cudaStream_t st = (cudaStream_t)stream;
  Workspace ws(workspace, workspace_bytes);
  const CoalesceBwdLayout l(ws, num_out, op);
  if (!ws.ok) return TGPB200_ERR_WORKSPACE;
  int* ties = l.ties;
  unsigned grid = (unsigned)ceil_div(E, 256);
  if (ties) {
    cudaMemsetAsync(ties, 0, (size_t)(num_out > 0 ? num_out : 1) * sizeof(int), st);
    launch("k_coalesce_ties", k_coalesce_ties, grid, 256, 0, st, edge_weight, out_weight, edge_slot, E, ties);
  }
  if ((op == TGPB200_SUM || op == TGPB200_MEAN) && E >= 4 &&
      ((reinterpret_cast<uintptr_t>(edge_slot) | reinterpret_cast<uintptr_t>(grad_in)) & 15) == 0) {
    const int64_t E4 = E / 4;
    launch("k_coalesce_bwd", k_coalesce_bwd4, (unsigned)ceil_div(E4, 256), 256, 0, st, grad_out, edge_slot, run_len, E4,
           op == TGPB200_MEAN ? 1 : 0, grad_in);
    if (E % 4)  // tail through the general kernel
      launch("k_coalesce_bwd", k_coalesce_bwd, 1, 256, 0, st, edge_weight ? edge_weight + E4 * 4 : nullptr, out_weight, grad_out, edge_slot + E4 * 4,
             run_len, run_aux, ties, E - E4 * 4, op, grad_in + E4 * 4);
    return launch_status();
  }
  launch("k_coalesce_bwd", k_coalesce_bwd, grid, 256, 0, st, edge_weight, out_weight, grad_out, edge_slot, run_len, run_aux, ties, E, op, grad_in);
  return launch_status();
}

size_t tgpb200_edge_norm_workspace_bytes(int64_t E, int64_t K) { return layout_bytes<EdgeNormLayout>(E, K); }

int tgpb200_rows_sorted(const int64_t* row, int64_t E, int32_t* sorted_out, tgpb200_stream_t stream) {
  if (E < 0 || !sorted_out) return TGPB200_ERR_INVALID;
  cudaStream_t st = (cudaStream_t)stream;
  const int32_t one = 1;
  cudaMemcpyAsync(sorted_out, &one, sizeof(one), cudaMemcpyHostToDevice, st);
  if (E > 1) {
    if (!row) return TGPB200_ERR_INVALID;
    launch("k_rows_sorted", k_rows_sorted, (unsigned)ceil_div(E, 256), 256, 0, st, row, E, sorted_out);
  }
  return launch_status();
}

int tgpb200_degree_accumulate(const int64_t* row, const float* w, int64_t E, const int64_t* E_dev, int64_t K,
                              int rows_sorted, float* deg, void* workspace, size_t workspace_bytes,
                              tgpb200_stream_t stream) {
  if (E < 0 || K < 0 || E >= INT32_MAX) return TGPB200_ERR_INVALID;
  if (K == 0) return TGPB200_OK;
  if (!deg || (E > 0 && !row)) return TGPB200_ERR_INVALID;
  Workspace ws(workspace, workspace_bytes);
  const EdgeNormLayout l(ws, E, K);
  if (!ws.ok) return TGPB200_ERR_WORKSPACE;
  return det_segment_sum(KeyOfArray64{row}, DegVal{w}, E, E_dev, K, rows_sorted != 0, deg, l.row, (cudaStream_t)stream);
}

int tgpb200_degree_apply(const int64_t* row, const int64_t* col, const float* w, const float* deg, int64_t E,
                         const int64_t* E_dev, int64_t K, float eps, float* w_out, tgpb200_stream_t stream) {
  if (E < 0 || K < 0) return TGPB200_ERR_INVALID;
  if (E == 0) return TGPB200_OK;
  if (!row || !col || !deg || !w_out) return TGPB200_ERR_INVALID;
  launch("k_deg_apply", k_deg_apply, (unsigned)ceil_div(E, 256), 256, 0, (cudaStream_t)stream, row, col, w, deg, E, E_dev,
         K, eps, w_out);
  return launch_status();
}

int tgpb200_degree_norm_fwd(const int64_t* row, const int64_t* col, const float* w, int64_t E, const int64_t* E_dev,
                            int64_t K, float eps, int rows_sorted, float* deg_out, float* w_out, void* workspace,
                            size_t workspace_bytes, tgpb200_stream_t stream) {
  int rc = tgpb200_degree_accumulate(row, w, E, E_dev, K, rows_sorted, deg_out, workspace, workspace_bytes, stream);
  if (rc != TGPB200_OK) return rc;
  return tgpb200_degree_apply(row, col, w, deg_out, E, E_dev, K, eps, w_out, stream);
}

int tgpb200_degree_bwd_accumulate(const int64_t* row, const int64_t* col, const float* w, const float* deg,
                                  const float* grad_out, int64_t E, const int64_t* E_dev, int64_t K, float eps,
                                  int rows_sorted, float* grad_dinv, void* workspace, size_t workspace_bytes,
                                  tgpb200_stream_t stream) {
  if (E < 0 || K < 0 || E >= INT32_MAX) return TGPB200_ERR_INVALID;
  if (K == 0) return TGPB200_OK;
  if (!grad_dinv || (E > 0 && (!row || !col || !deg || !grad_out))) return TGPB200_ERR_INVALID;
  cudaStream_t st = (cudaStream_t)stream;
  Workspace ws(workspace, workspace_bytes);
  const EdgeNormLayout l(ws, E, K);
  if (!ws.ok) return TGPB200_ERR_WORKSPACE;
  int rc;
  if (rows_sorted && E > 0) {
    launch("k_deg_bwd_prepare", k_deg_bwd_prepare, (unsigned)ceil_div(E, kDsTile), kDsThreads, 0, st, row, col, w, deg,
           grad_out, E, E_dev, K, eps, l.row.ev, l.col.ev, l.col.keys0, l.row.tiles, l.row.tile_flags);
    segmented_run_sums(KeyOfArray64{row}, ValOfArray{l.row.ev}, E, E_dev, K, l.row.tiles, l.row.tile_flags,
                       l.part_row, st, true);
    // the column side is a scatter by `col`: grouped through the stable sort
    rc = grouped_sums_of(l.col, E, E_dev, K, l.part_col, st);
    if (rc != TGPB200_OK) return rc;
  } else {
    rc = det_segment_sum(KeyOfArray64{row}, DegBwdVal{col, w, deg, grad_out, K, eps}, E, E_dev, K, rows_sorted != 0,
                         l.part_row, l.row, st);
    if (rc != TGPB200_OK) return rc;
    // the column side is a scatter by `col`: always grouped through the stable sort
    rc = det_segment_sum(KeyOfArray64{col}, DegBwdVal{row, w, deg, grad_out, K, eps}, E, E_dev, K, false, l.part_col,
                         l.col, st);
    if (rc != TGPB200_OK) return rc;
  }
  launch("k_add_vec", k_add_vec, (unsigned)ceil_div(K, 256), 256, 0, st, l.part_row, l.part_col, K, grad_dinv);
  return launch_status();
}

int tgpb200_degree_bwd_apply(const int64_t* row, const int64_t* col, const float* deg, const float* grad_out,
                             const float* grad_dinv, int64_t E, const int64_t* E_dev, int64_t K, float eps,
                             float* grad_w, tgpb200_stream_t stream) {
  if (E < 0 || K < 0) return TGPB200_ERR_INVALID;
  if (E == 0) return TGPB200_OK;
  if (!row || !col || !deg || !grad_out || !grad_dinv || !grad_w) return TGPB200_ERR_INVALID;
  launch("k_deg_bwd_apply", k_deg_bwd_apply, (unsigned)ceil_div(E, 256), 256, 0, (cudaStream_t)stream, row, col, deg,
         grad_out, grad_dinv, E, E_dev, K, eps, grad_w);
  return launch_status();
}

int tgpb200_degree_norm_bwd(const int64_t* row, const int64_t* col, const float* w, const float* deg,
                            const float* grad_out, int64_t E, const int64_t* E_dev, int64_t K, float eps,
                            int rows_sorted, float* grad_dinv, float* grad_w, void* workspace, size_t workspace_bytes,
                            tgpb200_stream_t stream) {
  if (E == 0) return TGPB200_OK;
  int rc = tgpb200_degree_bwd_accumulate(row, col, w, deg, grad_out, E, E_dev, K, eps, rows_sorted, grad_dinv, workspace,
                                         workspace_bytes, stream);
  if (rc != TGPB200_OK) return rc;
  return tgpb200_degree_bwd_apply(row, col, deg, grad_out, grad_dinv, E, E_dev, K, eps, grad_w, stream);
}

int tgpb200_weight_max_accumulate(const int64_t* row, const float* w, const int64_t* batch_pooled, int64_t E,
                                  const int64_t* E_dev, int64_t G, float* max_out, tgpb200_stream_t stream) {
  if (E < 0 || G < 0) return TGPB200_ERR_INVALID;
  cudaStream_t st = (cudaStream_t)stream;
  if (G > 0) {
    if (!max_out) return TGPB200_ERR_INVALID;
    cudaMemsetAsync(max_out, 0, (size_t)G * sizeof(float), st);
  }
  if (E > 0) {
    if (!row || !w || !batch_pooled) return TGPB200_ERR_INVALID;
    launch("k_wn_max", k_wn_max, (unsigned)ceil_div(E, 256), 256, 0, st, row, w, batch_pooled, E, E_dev, G, max_out);
  }
  return launch_status();
}

int tgpb200_weight_max_apply(const int64_t* row, const float* w, const int64_t* batch_pooled, const float* max_in,
                             int64_t E, const int64_t* E_dev, int64_t G, float* w_out, tgpb200_stream_t stream) {
  if (E < 0 || G < 0) return TGPB200_ERR_INVALID;
  if (E == 0) return TGPB200_OK;
  if (!row || !w || !batch_pooled || !max_in || !w_out) return TGPB200_ERR_INVALID;
  launch("k_wn_apply", k_wn_apply, (unsigned)ceil_div(E, 256), 256, 0, (cudaStream_t)stream, row, w, batch_pooled, max_in,
         E, E_dev, G, (int32_t*)nullptr, w_out);
  return launch_status();
}

int tgpb200_weight_norm_fwd(const int64_t* row, const float* w, const int64_t* batch_pooled, int64_t E,
                            const int64_t* E_dev, int64_t G, float* max_out, int32_t* arg_out, float* w_out,
                            tgpb200_stream_t stream) {
  if (E < 0 || G < 0) return TGPB200_ERR_INVALID;
  cudaStream_t st = (cudaStream_t)stream;
  if (G > 0) {
    if (!max_out) return TGPB200_ERR_INVALID;
    cudaMemsetAsync(max_out, 0, (size_t)G * sizeof(float), st);
    if (arg_out) cudaMemsetAsync(arg_out, 0x7f, (size_t)G * sizeof(int32_t), st);
  }
  if (E == 0) return launch_status();
  if (!row || !w || !batch_pooled || !w_out) return TGPB200_ERR_INVALID;
  unsigned grid = (unsigned)ceil_div(E, 256);
  launch("k_wn_max", k_wn_max, grid, 256, 0, st, row, w, batch_pooled, E, E_dev, G, max_out);
  launch("k_wn_apply", k_wn_apply, grid, 256, 0, st, row, w, batch_pooled, max_out, E, E_dev, G, arg_out, w_out);
  return launch_status();
}

// graph_acc[g] = sum over the graph's edges of grad_out * w, deterministically: per pooled node first (segmented by
// row), then per graph (pooled nodes grouped by batch_pooled with the stable sort).
int tgpb200_weight_norm_bwd(const int64_t* row, const float* w, const int64_t* batch_pooled, const float* max_in,
                            const int32_t* arg_in, const float* grad_out, int64_t E, const int64_t* E_dev, int64_t K,
                            int64_t G, int rows_sorted, float* graph_acc, float* grad_w, void* workspace,
                            size_t workspace_bytes, tgpb200_stream_t stream) {
  if (E < 0 || G < 0 || K < 0 || E >= INT32_MAX) return TGPB200_ERR_INVALID;
  if (E == 0) return TGPB200_OK;
  if (!row || !w || !batch_pooled || !max_in || !arg_in || !grad_out || !graph_acc || !grad_w)
    return TGPB200_ERR_INVALID;
  cudaStream_t st = (cudaStream_t)stream;
  Workspace ws(workspace, workspace_bytes);
  const EdgeNormLayout l(ws, E, K > G ? K : G);  // the query's K covers both the pooled nodes and the graphs
  if (!ws.ok) return TGPB200_ERR_WORKSPACE;
  float* node_acc = l.part_row;
  int rc = det_segment_sum(KeyOfArray64{row}, ProdVal{grad_out, w}, E, E_dev, K, rows_sorted != 0, node_acc, l.row, st);
  if (rc != TGPB200_OK) return rc;
  rc = det_segment_sum(KeyOfArray64{batch_pooled}, ArrVal{node_acc}, K, nullptr, G, false, graph_acc, l.nodes, st);
  if (rc != TGPB200_OK) return rc;
  launch("k_wn_bwd_apply", k_wn_bwd_apply, (unsigned)ceil_div(E, 256), 256, 0, st, row, w, batch_pooled, max_in, arg_in,
         grad_out, graph_acc, E, E_dev, G, grad_w);
  return launch_status();
}

}  // extern "C"
