// Sparse Reduce: CSR-by-cluster build, segment reduce forward/backward, reduce_batch.
// Reference: tgp/reduce/base_reduce.py:15-53,141-155; tgp/reduce/aggr_reduce.py:13-29,99-105.
#include "prims.cuh"

namespace tgp {

// ------------------------------------------------------------------------------------------
// CSR build
// ------------------------------------------------------------------------------------------
static __global__ void k_cluster_keys_count(const int64_t* __restrict__ cluster, int64_t nnz, int64_t K,
                                            uint32_t* __restrict__ keys, int* __restrict__ counts) {
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= nnz) return;
  int64_t c = cluster[i];
  if (c < 0 || c >= K) c = K - 1 > 0 ? K - 1 : 0;  // out-of-range ids are clamped (never dereferenced OOB)
  keys[i] = (uint32_t)c;
  atomicAdd(&counts[c], 1);
}

// Small inputs (a mini-batch of small graphs: a few thousand kept nodes) are launch-bound: the generic build is a
// memset + key / count kernel + one launch per radix pass + a scan.  ONE block does the same stable counting sort in
// shared memory: per-cluster counts, exclusive scan (= ptr), then the members are placed in ascending entry order --
// chunks of blockDim entries in order, the warps of a chunk in order, the lanes of a warp ranked with
// __match_any_sync -- so `order` and `ptr` are bit-identical to the radix path.
constexpr int kCsrSmallNnz = 8192;
constexpr int kCsrSmallK = 8192;
constexpr int kCsrSmallThreads = 1024;

static __global__ void __launch_bounds__(kCsrSmallThreads)
    k_build_csr_small(const int64_t* __restrict__ cluster, int nnz, int K, int32_t* __restrict__ order,
                      int32_t* __restrict__ ptr) {
  __shared__ int s_off[kCsrSmallK + 1];  // counts -> exclusive offsets -> next free position of every cluster
  __shared__ int s_scan[33];
  const int t = threadIdx.x, lane = t & 31, w = t >> 5;
  auto cluster_of = [&](int i) {
    const int64_t c = cluster[i];
    return (int)((c < 0 || c >= K) ? (K - 1 > 0 ? K - 1 : 0) : c);  // same clamp as k_cluster_keys_count
  };
  for (int c = t; c <= K; c += kCsrSmallThreads) s_off[c] = 0;
  __syncthreads();
  for (int i = t; i < nnz; i += kCsrSmallThreads) atomicAdd(&s_off[cluster_of(i)], 1);
  __syncthreads();
  {  // exclusive scan over the K + 1 counters (the last one is zero and becomes the total)
    const int per = (K + kCsrSmallThreads) / kCsrSmallThreads;  // ceil((K + 1) / threads)
    const int lo = min(t * per, K + 1), hi = min(lo + per, K + 1);
    int sum = 0;
    for (int j = lo; j < hi; ++j) sum += s_off[j];
    int base = block_exclusive_scan_i(sum, s_scan, nullptr);
    for (int j = lo; j < hi; ++j) {
      const int n = s_off[j];
      s_off[j] = base;
      ptr[j] = base;
      base += n;
    }
  }
  __syncthreads();
  for (int i0 = 0; i0 < nnz; i0 += kCsrSmallThreads) {
    const int i = i0 + t;
    const bool on = i < nnz;
    const int c = on ? cluster_of(i) : -1;
    const unsigned peers = __match_any_sync(kFull, c);
    const int rank = __popc(peers & ((1u << lane) - 1u));
    const bool last = lane == 31 - __clz((int)peers);  // the highest lane of the group advances the counter
    const int warps = min(32, (nnz - i0 + 31) >> 5);
    for (int ww = 0; ww < warps; ++ww) {
      if (w == ww) {
        const int p = on ? s_off[c] + rank : 0;
        __syncwarp();
        if (on && last) s_off[c] += __popc(peers);
        if (on) order[p] = i;
      }
      __syncthreads();
    }
  }
}

static int key_bits_for(int64_t max_value) {
  int b = 0;
  while (b < 63 && ((int64_t)1 << b) <= max_value) ++b;
  return b < 1 ? 1 : b;
}

// ------------------------------------------------------------------------------------------
// Vector row access: 16-byte chunks of VEC elements
// ------------------------------------------------------------------------------------------
template <typename T>
struct Vec;
template <>
struct Vec<float> {
  static constexpr int N = 4;
  __device__ static void load(const float* p, float (&v)[4]) {
    float4 t = __ldg(reinterpret_cast<const float4*>(p));
    v[0] = t.x, v[1] = t.y, v[2] = t.z, v[3] = t.w;
  }
  __device__ static void store(float* p, const float (&v)[4]) {
    *reinterpret_cast<float4*>(p) = make_float4(v[0], v[1], v[2], v[3]);
  }
};
template <>
struct Vec<__nv_bfloat16> {
  static constexpr int N = 8;
  __device__ static void load(const __nv_bfloat16* p, float (&v)[8]) {
    uint4 t = __ldg(reinterpret_cast<const uint4*>(p));
    const __nv_bfloat162* h = reinterpret_cast<const __nv_bfloat162*>(&t);
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      float2 f = __bfloat1622float2(h[k]);
      v[2 * k] = f.x, v[2 * k + 1] = f.y;
    }
  }
  __device__ static void store(__nv_bfloat16* p, const float (&v)[8]) {
    uint4 t;
    __nv_bfloat162* h = reinterpret_cast<__nv_bfloat162*>(&t);
#pragma unroll
    for (int k = 0; k < 4; ++k) h[k] = __floats2bfloat162_rn(v[2 * k], v[2 * k + 1]);
    *reinterpret_cast<uint4*>(p) = t;
  }
};

// generic chunk access honouring a scalar fallback (F not a multiple of the vector width)
template <typename T, int W, bool kVec>
__device__ __forceinline__ void load_chunk(const T* row, int64_t f, int64_t F, float (&v)[W]) {
  if (kVec) {
    Vec<T>::load(row + f, reinterpret_cast<float(&)[Vec<T>::N]>(v));
  } else {
#pragma unroll
    for (int k = 0; k < W; ++k) v[k] = (f + k < F) ? to_f32<T>(row[f + k]) : 0.f;
  }
}
template <typename T, int W, bool kVec>
__device__ __forceinline__ void store_chunk(T* row, int64_t f, int64_t F, const float (&v)[W]) {
  if (kVec) {
    Vec<T>::store(row + f, reinterpret_cast<const float(&)[Vec<T>::N]>(v));
  } else {
#pragma unroll
    for (int k = 0; k < W; ++k)
      if (f + k < F) row[f + k] = from_f32<T>(v[k]);
  }
}

__device__ __forceinline__ float combine(int op, float acc, float p, bool first) {
  if (op == TGPB200_SUM || op == TGPB200_MEAN) return __fadd_rn(acc, p);
  if (first) return p;
  return op == TGPB200_MAX ? fmaxf(acc, p) : fminf(acc, p);
}

// ------------------------------------------------------------------------------------------
// Forward: one lane-group per cluster, lanes over 16-byte feature chunks, members in CSR order.
// Products are rounded before the add (no FMA contraction) so fp32 sums are bit-identical
// to the reference's sequential CPU scatter_add_.
// ------------------------------------------------------------------------------------------
template <typename XT, typename OT, bool kVec>
static __global__ void __launch_bounds__(256)
    k_segment_reduce_fwd(const XT* __restrict__ x, const int64_t* __restrict__ node_index,
                         const float* __restrict__ weight, const int32_t* __restrict__ order,
                         const int32_t* __restrict__ ptr, int64_t N, int64_t K, int64_t F, int op, int lpr,
                         OT* __restrict__ out) {
  constexpr int W = Vec<XT>::N;
  int64_t gid = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) / lpr;
  int sub = threadIdx.x % lpr;
  if (gid >= K) return;
  int beg = ptr[gid], end = ptr[gid + 1];
  for (int64_t f = (int64_t)sub * W; f < F; f += (int64_t)lpr * W) {
    float acc[W];
#pragma unroll
    for (int k = 0; k < W; ++k) acc[k] = 0.f;
    int m = beg;
    for (; m + 1 < end; m += 2) {  // two members in flight
      int i0 = order[m], i1 = order[m + 1];
      int64_t n0 = node_index[i0], n1 = node_index[i1];
      float w0 = weight ? weight[i0] : 1.f, w1 = weight ? weight[i1] : 1.f;
      float v0[W], v1[W];
      bool ok0 = n0 >= 0 && n0 < N, ok1 = n1 >= 0 && n1 < N;
      if (ok0) load_chunk<XT, W, kVec>(x + n0 * F, f, F, v0);
      if (ok1) load_chunk<XT, W, kVec>(x + n1 * F, f, F, v1);
#pragma unroll
      for (int k = 0; k < W; ++k) {
        float p0 = ok0 ? __fmul_rn(v0[k], w0) : 0.f;
        float p1 = ok1 ? __fmul_rn(v1[k], w1) : 0.f;
        acc[k] = combine(op, acc[k], p0, m == beg);
        acc[k] = combine(op, acc[k], p1, false);
      }
    }
    if (m < end) {
      int i0 = order[m];
      int64_t n0 = node_index[i0];
      float w0 = weight ? weight[i0] : 1.f;
      float v0[W];
      bool ok0 = n0 >= 0 && n0 < N;
      if (ok0) load_chunk<XT, W, kVec>(x + n0 * F, f, F, v0);
#pragma unroll
      for (int k = 0; k < W; ++k) acc[k] = combine(op, acc[k], ok0 ? __fmul_rn(v0[k], w0) : 0.f, m == beg);
    }
    if (op == TGPB200_MEAN) {
      float cnt = (float)(end - beg > 1 ? end - beg : 1);
#pragma unroll
      for (int k = 0; k < W; ++k) acc[k] = __fdiv_rn(acc[k], cnt);
    }
    store_chunk<OT, W, kVec>(out + gid * F, f, F, acc);
  }
}

// Vector-row fast path of the forward: a warp takes NPW clusters at once.  Lanes 0..MPL*NPW-1 resolve the first MPL
// members of each cluster side by side (ptr -> order -> node_index / weight are dependent loads), then all lanes
// gather up to MPL*NPW member rows with every load in flight; later members follow in the generic two-at-a-time
// loop.  Members are combined in CSR order exactly as in k_segment_reduce_fwd (bit-identical sums).  (NPW, MPL) =
// (4, 2) for clusters of about two members, (8, 1) when almost every cluster has one (TopK: nnz == K) -- eight rows
// in flight per warp either way; node ids travel as 32-bit (the launcher checks N < 2^31).
template <typename XT, typename OT, int NPW, int MPL>
static __global__ void __launch_bounds__(256)
    k_segment_reduce_fwd_rows(const XT* __restrict__ x, const int64_t* __restrict__ node_index,
                              const float* __restrict__ weight, const int32_t* __restrict__ order,
                              const int32_t* __restrict__ ptr, int64_t N, int64_t K, int64_t F, int op,
                              OT* __restrict__ out) {
  constexpr int W = Vec<XT>::N;
  const int lane = threadIdx.x & 31;
  const int64_t c0 = (((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5) * NPW;
  if (c0 >= K) return;
  int beg = 0, end = 0;
  int64_t node = -1;
  float wt = 0.f;
  if (lane < MPL * NPW && c0 + lane / MPL < K) {
    const int64_t c = c0 + lane / MPL;
    beg = ptr[c], end = ptr[c + 1];
    const int m = beg + lane % MPL;
    if (m < end) {
      const int i = order[m];
      node = node_index[i];
      wt = weight ? weight[i] : 1.f;
      if (node < 0 || node >= N) node = -1;
    }
  }
  int beg_j[NPW], end_j[NPW];
  int n_j[NPW][MPL];
  float w_j[NPW][MPL];
#pragma unroll
  for (int j = 0; j < NPW; ++j) {
    beg_j[j] = __shfl_sync(kFull, beg, MPL * j), end_j[j] = __shfl_sync(kFull, end, MPL * j);
#pragma unroll
    for (int k = 0; k < MPL; ++k) {
      n_j[j][k] = __shfl_sync(kFull, (int)node, MPL * j + k);
      w_j[j][k] = __shfl_sync(kFull, wt, MPL * j + k);
    }
  }
  for (int64_t f = (int64_t)lane * W; f < F; f += 32 * W) {
    float v[NPW][MPL][W];
#pragma unroll
    for (int j = 0; j < NPW; ++j)
#pragma unroll
      for (int k = 0; k < MPL; ++k)
        if (n_j[j][k] >= 0) load_chunk<XT, W, true>(x + (int64_t)n_j[j][k] * F, f, F, v[j][k]);
#pragma unroll
    for (int j = 0; j < NPW; ++j) {
      const int64_t c = c0 + j;
      if (c >= K) break;
      const int b = beg_j[j], e = end_j[j];
      float acc[W];
#pragma unroll
      for (int k = 0; k < W; ++k) acc[k] = 0.f;
#pragma unroll
      for (int k = 0; k < MPL; ++k) {
        if (b + k < e) {
#pragma unroll
          for (int q = 0; q < W; ++q)
            acc[q] = combine(op, acc[q], n_j[j][k] >= 0 ? __fmul_rn(v[j][k][q], w_j[j][k]) : 0.f, k == 0);
        }
      }
      int m = b + MPL;
      for (; m + 1 < e; m += 2) {  // larger clusters: two members in flight
        int i0 = order[m], i1 = order[m + 1];
        int64_t n0 = node_index[i0], n1 = node_index[i1];
        float w0 = weight ? weight[i0] : 1.f, w1 = weight ? weight[i1] : 1.f;
        float v0[W], v1[W];
        bool ok0 = n0 >= 0 && n0 < N, ok1 = n1 >= 0 && n1 < N;
        if (ok0) load_chunk<XT, W, true>(x + n0 * F, f, F, v0);
        if (ok1) load_chunk<XT, W, true>(x + n1 * F, f, F, v1);
#pragma unroll
        for (int q = 0; q < W; ++q) {
          acc[q] = combine(op, acc[q], ok0 ? __fmul_rn(v0[q], w0) : 0.f, false);
          acc[q] = combine(op, acc[q], ok1 ? __fmul_rn(v1[q], w1) : 0.f, false);
        }
      }
      if (m < e) {
        int i0 = order[m];
        int64_t n0 = node_index[i0];
        float w0 = weight ? weight[i0] : 1.f;
        float v0[W];
        bool ok0 = n0 >= 0 && n0 < N;
        if (ok0) load_chunk<XT, W, true>(x + n0 * F, f, F, v0);
#pragma unroll
        for (int q = 0; q < W; ++q) acc[q] = combine(op, acc[q], ok0 ? __fmul_rn(v0[q], w0) : 0.f, false);
      }
      if (op == TGPB200_MEAN) {
        float cnt = (float)(e - b > 1 ? e - b : 1);
#pragma unroll
        for (int q = 0; q < W; ++q) acc[q] = __fdiv_rn(acc[q], cnt);
      }
      store_chunk<OT, W, true>(out + c * F, f, F, acc);
    }
  }
}

// ------------------------------------------------------------------------------------------
// MAX / MIN backward pre-pass: inv_ties[c, f] = 1 / #members whose product equals x_pool[c, f].
// ------------------------------------------------------------------------------------------
template <typename XT, typename OT>
static __global__ void k_count_ties(const XT* __restrict__ x, const int64_t* __restrict__ node_index,
                                    const float* __restrict__ weight, const int32_t* __restrict__ order,
                                    const int32_t* __restrict__ ptr, const OT* __restrict__ pool, int64_t N, int64_t K,
                                    int64_t F, float* __restrict__ inv_ties) {
  int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= K * F) return;
  int64_t c = t / F, f = t % F;
  float target = to_f32<OT>(pool[t]);
  int cnt = 0;
  for (int m = ptr[c]; m < ptr[c + 1]; ++m) {
    int i = order[m];
    int64_t n = node_index[i];
    if (n < 0 || n >= N) continue;
    float p = __fmul_rn(to_f32<XT>(x[n * F + f]), weight ? weight[i] : 1.f);
    if (to_f32<OT>(from_f32<OT>(p)) == target) ++cnt;
  }
  inv_ties[t] = cnt > 0 ? 1.f / (float)cnt : 0.f;
}

// first[n] = position of node n's first entry in the (sorted) node_index, -1 (pre-filled) if it has none
static __global__ void k_first_entry(const int64_t* __restrict__ node_index, int64_t nnz, int64_t N,
                                     int32_t* __restrict__ first) {
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= nnz) return;
  const int64_t n = node_index[i];
  if (n < 0 || n >= N) return;
  if (i == 0 || node_index[i - 1] != n) first[n] = (int32_t)i;
}

// first entry of node n without the inverse map: lower bound in the sorted node_index (small inputs only: ~log2(nnz)
// cache-resident steps per node are cheaper than a separate map-building launch), -1 when the node has no entry
__device__ __forceinline__ int64_t first_entry_of(const int64_t* __restrict__ node_index, int64_t nnz, int64_t n) {
  int64_t lo = 0, hi = nnz;
  while (lo < hi) {
    const int64_t mid = (lo + hi) >> 1;
    if (node_index[mid] < n) lo = mid + 1; else hi = mid;
  }
  return (lo < nnz && node_index[lo] == n) ? lo : -1;
}

// ------------------------------------------------------------------------------------------
// Backward: one lane-group per NODE (node_index is sorted, so a node's entries are adjacent):
//   grad_x[n] = sum_{i in run(n)} w_i * gs_i,   grad_w[i] = <x[n], gs_i>,
//   gs_i = coefficient(op) * grad_pool[cluster_i].   Unselected nodes get zero rows.
// ------------------------------------------------------------------------------------------
template <typename XT, typename OT, bool kVec>
static __global__ void __launch_bounds__(256)
    k_segment_reduce_bwd(const XT* __restrict__ x, const int64_t* __restrict__ node_index,
                         const int64_t* __restrict__ cluster_index, const float* __restrict__ weight,
                         const int32_t* __restrict__ ptr, const int32_t* __restrict__ first,
                         const OT* __restrict__ pool, const OT* __restrict__ gpool,
                         const float* __restrict__ inv_ties, int64_t N, int64_t nnz, int64_t K, int64_t F, int op,
                         int lpr, XT* __restrict__ gx, float* __restrict__ gw) {
  constexpr int W = Vec<XT>::N;
  int64_t n = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) / lpr;
  int sub = threadIdx.x % lpr;
  if (n >= N) return;
  int lane = threadIdx.x & 31;
  unsigned gmask = lpr >= 32 ? kFull : (((1u << lpr) - 1u) << (lane & ~(lpr - 1)));

  // Entries of node n: first[n] (inverse map built by k_first_entry, -1 for an unselected node) and the adjacent
  // run behind it (node_index is sorted).  One dependent load instead of a log2(nnz)-step binary search.
  int64_t lo = first ? (int64_t)first[n] : first_entry_of(node_index, nnz, n), hi = 0;
  if (lo < 0) {
    lo = 0;
  } else {
    hi = lo + 1;
    while (hi < nnz && node_index[hi] == n) ++hi;
  }

  const XT* xr = x + n * F;
  for (int64_t i = lo; i < hi; ++i) {
    if (gw == nullptr) break;
    int64_t c = cluster_index[i];
    if (c < 0 || c >= K) { if (sub == 0) gw[i] = 0.f; continue; }
    float wi = weight ? weight[i] : 1.f;
    float coef = 1.f;
    if (op == TGPB200_MEAN) { int cnt = ptr[c + 1] - ptr[c]; coef = 1.f / (float)(cnt > 1 ? cnt : 1); }
    float dot = 0.f;
    for (int64_t f = (int64_t)sub * W; f < F; f += (int64_t)lpr * W) {
      float xv[W], gv[W];
      load_chunk<XT, W, kVec>(xr, f, F, xv);
      load_chunk<OT, W, kVec>(gpool + c * F, f, F, gv);
      if (op == TGPB200_MAX || op == TGPB200_MIN) {
        float pv[W];
        load_chunk<OT, W, kVec>(pool + c * F, f, F, pv);
#pragma unroll
        for (int k = 0; k < W; ++k) {
          float p = to_f32<OT>(from_f32<OT>(__fmul_rn(xv[k], wi)));
          float it = (f + k < F) ? inv_ties[c * F + f + k] : 0.f;
          gv[k] = (p == pv[k]) ? gv[k] * it : 0.f;
        }
      }
#pragma unroll
      for (int k = 0; k < W; ++k) dot += xv[k] * gv[k] * coef;
    }
    for (int o = lpr >> 1; o > 0; o >>= 1) dot += __shfl_xor_sync(gmask, dot, o);
    if (sub == 0) gw[i] = dot;
  }

  for (int64_t f = (int64_t)sub * W; f < F; f += (int64_t)lpr * W) {
    float acc[W];
#pragma unroll
    for (int k = 0; k < W; ++k) acc[k] = 0.f;
    float xv[W];
    bool need_x = (op == TGPB200_MAX || op == TGPB200_MIN) && hi > lo;
    if (need_x) load_chunk<XT, W, kVec>(xr, f, F, xv);
    for (int64_t i = lo; i < hi; ++i) {
      int64_t c = cluster_index[i];
      if (c < 0 || c >= K) continue;
      float wi = weight ? weight[i] : 1.f;
      float coef = wi;
      if (op == TGPB200_MEAN) { int cnt = ptr[c + 1] - ptr[c]; coef = wi / (float)(cnt > 1 ? cnt : 1); }
      float gv[W];
      load_chunk<OT, W, kVec>(gpool + c * F, f, F, gv);
      if (op == TGPB200_MAX || op == TGPB200_MIN) {
        float pv[W];
        load_chunk<OT, W, kVec>(pool + c * F, f, F, pv);
#pragma unroll
        for (int k = 0; k < W; ++k) {
          float p = to_f32<OT>(from_f32<OT>(__fmul_rn(xv[k], wi)));
          float it = (f + k < F) ? inv_ties[c * F + f + k] : 0.f;
          gv[k] = (p == pv[k]) ? gv[k] * it : 0.f;
        }
      }
#pragma unroll
      for (int k = 0; k < W; ++k) acc[k] = __fadd_rn(acc[k], __fmul_rn(gv[k], coef));
    }
    store_chunk<XT, W, kVec>(gx + n * F, f, F, acc);
  }
}

// Fast path of the backward (sum / mean, no weight gradient, vector rows): a warp takes NPW nodes at once.  Lanes
// 0..NPW-1 run the dependent lookup chains (node -> entry -> cluster -> cluster size) side by side, then all lanes
// copy the NPW gradient rows with the loads of all rows in flight together.  (One node per warp left the kernel
// latency-bound: four dependent global loads per 512-byte row.)  Same arithmetic as k_segment_reduce_bwd.
template <typename XT, typename OT, int NPW>
static __global__ void __launch_bounds__(256)
    k_segment_reduce_bwd_rows(const int64_t* __restrict__ node_index, const int64_t* __restrict__ cluster_index,
                              const float* __restrict__ weight, const int32_t* __restrict__ ptr,
                              const int32_t* __restrict__ first, const OT* __restrict__ gpool, int64_t N, int64_t nnz,
                              int64_t K, int64_t F, int op, XT* __restrict__ gx) {
  constexpr int W = Vec<XT>::N;
  const int lane = threadIdx.x & 31;
  const int64_t n0 = (((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5) * NPW;
  if (n0 >= N) return;
  int64_t lo = 0, hi = 0, c = -1;
  float coef = 0.f;
  if (lane < NPW && n0 + lane < N) {
    const int64_t n = n0 + lane;
    lo = first ? (int64_t)first[n] : first_entry_of(node_index, nnz, n);  // -1 for an unselected node
    if (lo < 0) {
      lo = 0;
    } else {
      hi = lo + 1;
      if (hi < nnz && node_index[hi] == n)
        while (hi < nnz && node_index[hi] == n) ++hi;
    }
    if (hi == lo + 1) {
      c = cluster_index[lo];
      if (c < 0 || c >= K) {
        c = -1;
      } else {
        const float wi = weight ? weight[lo] : 1.f;
        coef = wi;
        if (op == TGPB200_MEAN) { int cnt = ptr[c + 1] - ptr[c]; coef = wi / (float)(cnt > 1 ? cnt : 1); }
      }
    }
  }
  int lo_j[NPW], hi_j[NPW], c_j[NPW];  // nnz, K < 2^31 (checked by the entry point): 32-bit copies keep NPW = 8 in registers
  float coef_j[NPW];
#pragma unroll
  for (int j = 0; j < NPW; ++j) {
    lo_j[j] = __shfl_sync(kFull, (int)lo, j), hi_j[j] = __shfl_sync(kFull, (int)hi, j);
    c_j[j] = __shfl_sync(kFull, (int)c, j);
    coef_j[j] = __shfl_sync(kFull, coef, j);
  }
  for (int64_t f = (int64_t)lane * W; f < F; f += 32 * W) {
    float g[NPW][W];
#pragma unroll
    for (int j = 0; j < NPW; ++j)
      if (c_j[j] >= 0) load_chunk<OT, W, true>(gpool + (int64_t)c_j[j] * F, f, F, g[j]);
#pragma unroll
    for (int j = 0; j < NPW; ++j) {
      const int64_t n = n0 + j;
      if (n >= N) break;
      float acc[W];
      if (c_j[j] >= 0) {
#pragma unroll
        for (int k = 0; k < W; ++k) acc[k] = __fadd_rn(0.f, __fmul_rn(g[j][k], coef_j[j]));
      } else {
#pragma unroll
        for (int k = 0; k < W; ++k) acc[k] = 0.f;
        if (hi_j[j] > lo_j[j] + 1) {
          for (int64_t i = lo_j[j]; i < (int64_t)hi_j[j]; ++i) {  // a node assigned to several clusters (soft sparse S)
            const int64_t ci = cluster_index[i];
            if (ci < 0 || ci >= K) continue;
            const float wi = weight ? weight[i] : 1.f;
            float cf = wi;
            if (op == TGPB200_MEAN) { int cnt = ptr[ci + 1] - ptr[ci]; cf = wi / (float)(cnt > 1 ? cnt : 1); }
            float gv[W];
            load_chunk<OT, W, true>(gpool + ci * F, f, F, gv);
#pragma unroll
            for (int k = 0; k < W; ++k) acc[k] = __fadd_rn(acc[k], __fmul_rn(gv[k], cf));
          }
        }
      }
      store_chunk<XT, W, true>(gx + n * F, f, F, acc);
    }
  }
}

// out[c] = batch[node of the LAST member of c in position order] (CPU scatter_ semantics: the
// last writer wins), or c for an empty cluster (the arange initial value survives).
static __global__ void k_reduce_batch(const int64_t* __restrict__ batch, const int64_t* __restrict__ node_index,
                                      const int32_t* __restrict__ order, const int32_t* __restrict__ ptr, int64_t K,
                                      int64_t* __restrict__ out) {
  int64_t c = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= K) return;
  int b = ptr[c], e = ptr[c + 1];
  out[c] = e > b ? batch[node_index[order[e - 1]]] : c;
}

template <typename XT, typename OT>
static int launch_fwd(const void* x, const int64_t* node_index, const float* weight, const int32_t* order,
                      const int32_t* ptr, int64_t N, int64_t nnz, int64_t K, int64_t F, int op, void* out,
                      cudaStream_t st) {
  constexpr int W = Vec<XT>::N;
  // 16-byte chunks: whole rows AND 16-byte aligned bases (an unaligned view takes the scalar chunks, never the row
  // kernels, which exist in vector form only)
  bool vec = (F % W == 0) && (F % Vec<OT>::N == 0) && Vec<OT>::N == W && aligned16(x) && aligned16(out);
  int64_t chunks = ceil_div(F, W);
  int lpr = 1;
  while (lpr < 32 && lpr < chunks) lpr <<= 1;
  int64_t threads = K * lpr;
  if (threads == 0) return TGPB200_OK;
  dim3 grid((unsigned)ceil_div(threads, 256));
  if (vec && lpr == 32 && N < INT32_MAX) {  // rows of >= 32 vector chunks: several clusters per warp (latency-bound otherwise)
    if (nnz <= K + K / 4)  // almost every cluster has one member (TopK): eight clusters per warp, one member preloaded
      launch("k_segment_reduce_fwd", k_segment_reduce_fwd_rows<XT, OT, 8, 1>, (unsigned)ceil_div(ceil_div(K, 8) * 32, 256),
             256, 0, st, (const XT*)x, node_index, weight, order, ptr, N, K, F, op, (OT*)out);
    else
      launch("k_segment_reduce_fwd", k_segment_reduce_fwd_rows<XT, OT, 4, 2>, (unsigned)ceil_div(ceil_div(K, 4) * 32, 256),
             256, 0, st, (const XT*)x, node_index, weight, order, ptr, N, K, F, op, (OT*)out);
    return launch_status();
  }
  if (vec)
    launch("k_segment_reduce_fwd", k_segment_reduce_fwd<XT, OT, true>, grid, 256, 0, st, (const XT*)x, node_index, weight, order, ptr, N, K, F, op,
                                                             lpr, (OT*)out);
  else
    launch("k_segment_reduce_fwd", k_segment_reduce_fwd<XT, OT, false>, grid, 256, 0, st, (const XT*)x, node_index, weight, order, ptr, N, K, F,
                                                              op, lpr, (OT*)out);
  return launch_status();
}

template <typename XT, typename OT>
static int launch_bwd(const void* x, const int64_t* node_index, const int64_t* cluster_index, const float* weight,
                      const int32_t* order, const int32_t* ptr, const void* pool, const void* gpool, int64_t N,
                      int64_t nnz, int64_t K, int64_t F, int op, void* gx, float* gw, Workspace& ws, cudaStream_t st) {
  constexpr int W = Vec<XT>::N;
  const bool minmax = op == TGPB200_MAX || op == TGPB200_MIN;
  bool vec = (F % W == 0) && Vec<OT>::N == W && aligned16(x) && aligned16(gpool) && aligned16(gx) &&
             (!minmax || aligned16(pool));
  int32_t* first = ws.take<int32_t>((size_t)(N > 0 ? N : 1));
  if (!ws.ok) return TGPB200_ERR_WORKSPACE;
  if (N > 0 && N <= 32768 && nnz <= 32768) {
    first = nullptr;  // the backward kernels search the (cache-resident) sorted node_index themselves: one launch less
  } else {
    cudaMemsetAsync(first, 0xff, (size_t)(N > 0 ? N : 1) * sizeof(int32_t), st);
    if (nnz > 0)
      launch("k_first_entry", k_first_entry, (unsigned)ceil_div(nnz, 256), 256, 0, st, node_index, nnz, N, first);
  }
  float* inv_ties = nullptr;
  if (minmax) {
    inv_ties = ws.take<float>((size_t)K * F);
    if (!ws.ok) return TGPB200_ERR_WORKSPACE;
    if (K * F > 0)
      launch("k_count_ties", k_count_ties<XT, OT>, (unsigned)ceil_div(K * F, 256), 256, 0, st, (const XT*)x, node_index, weight, order, ptr,
                                                                          (const OT*)pool, N, K, F, inv_ties);
  }
  int64_t chunks = ceil_div(F, W);
  int lpr = 1;
  while (lpr < 32 && lpr < chunks) lpr <<= 1;
  int64_t threads = N * lpr;
  if (threads == 0) return TGPB200_OK;
  dim3 grid((unsigned)ceil_div(threads, 256));
  if (vec && gw == nullptr && (op == TGPB200_SUM || op == TGPB200_MEAN)) {
#ifndef TGPB200_BWD_NPW
#define TGPB200_BWD_NPW 8  // rows in flight per warp: 4 left the kernel bound by its four dependent lookups (3.8 TB/s)
#endif
    constexpr int NPW = TGPB200_BWD_NPW;
    const int64_t warps = ceil_div(N, NPW);
    launch("k_segment_reduce_bwd", k_segment_reduce_bwd_rows<XT, OT, NPW>, (unsigned)ceil_div(warps * 32, 256), 256, 0, st,
           node_index, cluster_index, weight, ptr, first, (const OT*)gpool, N, nnz, K, F, op, (XT*)gx);
    return launch_status();
  }
  if (vec)
    launch("k_segment_reduce_bwd", k_segment_reduce_bwd<XT, OT, true>, grid, 256, 0, st, (const XT*)x, node_index, cluster_index, weight, ptr,
                                                             first, (const OT*)pool, (const OT*)gpool, inv_ties, N, nnz, K, F,
                                                             op, lpr, (XT*)gx, gw);
  else
    launch("k_segment_reduce_bwd", k_segment_reduce_bwd<XT, OT, false>, grid, 256, 0, st, (const XT*)x, node_index, cluster_index, weight, ptr,
                                                              first, (const OT*)pool, (const OT*)gpool, inv_ties, N, nnz, K,
                                                              F, op, lpr, (XT*)gx, gw);
  return launch_status();
}

}  // namespace tgp

using namespace tgp;

extern "C" {

int tgpb200_abi_version(void) { return 1; }

size_t tgpb200_build_csr_workspace_bytes(int64_t nnz, int64_t K) {
  size_t n = (size_t)(nnz > 0 ? nnz : 1);
  return 4 * align_up(n * sizeof(uint32_t)) + radix_sort_workspace_bytes(nnz) + scan_workspace_bytes(K + 1) + 1024;
}

int tgpb200_build_csr(const int64_t* cluster_index, int64_t nnz, int64_t K, int32_t* order, int32_t* ptr,
                      void* workspace, size_t workspace_bytes, tgpb200_stream_t stream) {
  if (nnz < 0 || K < 0 || nnz >= INT32_MAX || K >= INT32_MAX || !ptr || (nnz > 0 && (!cluster_index || !order)))
    return TGPB200_ERR_INVALID;
  cudaStream_t st = (cudaStream_t)stream;
  Workspace ws(workspace, workspace_bytes);
  size_t n = (size_t)(nnz > 0 ? nnz : 1);
  uint32_t* keys0 = ws.take<uint32_t>(n);
  uint32_t* keys1 = ws.take<uint32_t>(n);
  uint32_t* valsA = ws.take<uint32_t>(n);
  if (!ws.ok) return TGPB200_ERR_WORKSPACE;
  if (nnz > 0 && K == 0) return TGPB200_ERR_INVALID;
  if (nnz <= kCsrSmallNnz && K <= kCsrSmallK) {
    launch("k_build_csr_small", k_build_csr_small, 1, kCsrSmallThreads, 0, st, cluster_index, (int)nnz, (int)K, order, ptr);
    return launch_status();
  }
  cudaMemsetAsync(ptr, 0, (size_t)(K + 1) * sizeof(int32_t), st);
  if (nnz > 0) {
    launch("k_cluster_keys_count", k_cluster_keys_count, (unsigned)ceil_div(nnz, 256), 256, 0, st, cluster_index, nnz, K, keys0, ptr);
    int bits = key_bits_for(K - 1);
    int passes = radix_passes(bits);
    // choose buffers so the final payload lands in `order`
    uint32_t* vals1 = (passes & 1) ? (uint32_t*)order : valsA;
    uint32_t* vals0 = (passes & 1) ? valsA : (uint32_t*)order;
    bool in1 = false;
    int rc = radix_sort_pairs<uint32_t>(keys0, nullptr, vals0, keys1, vals1, nnz, bits, &in1, ws, st);
    if (rc != TGPB200_OK) return rc;
  }
  int rc = exclusive_scan_i32(ptr, ptr, K + 1, nullptr, nullptr, ws, st);
  return rc != TGPB200_OK ? rc : launch_status();
}

int tgpb200_segment_reduce_fwd(const void* x, const int64_t* node_index, const float* weight, const int32_t* order,
                               const int32_t* ptr, int64_t N, int64_t nnz, int64_t K, int64_t F, int op, int x_dtype,
                               int out_dtype, void* x_pool, tgpb200_stream_t stream) {
  if (N < 0 || nnz < 0 || K < 0 || F < 0 || op < TGPB200_SUM || op > TGPB200_MIN) return TGPB200_ERR_INVALID;
  if (K * F == 0) return TGPB200_OK;
  if (!x_pool || !ptr || (nnz > 0 && (!x || !node_index || !order))) return TGPB200_ERR_INVALID;
  cudaStream_t st = (cudaStream_t)stream;
  if (x_dtype == TGPB200_F32 && out_dtype == TGPB200_F32)
    return launch_fwd<float, float>(x, node_index, weight, order, ptr, N, nnz, K, F, op, x_pool, st);
  if (x_dtype == TGPB200_BF16 && out_dtype == TGPB200_BF16)
    return launch_fwd<__nv_bfloat16, __nv_bfloat16>(x, node_index, weight, order, ptr, N, nnz, K, F, op, x_pool, st);
  if (x_dtype == TGPB200_BF16 && out_dtype == TGPB200_F32)
    return launch_fwd<__nv_bfloat16, float>(x, node_index, weight, order, ptr, N, nnz, K, F, op, x_pool, st);
  return TGPB200_ERR_UNSUPPORTED;
}

size_t tgpb200_segment_reduce_bwd_workspace_bytes(int64_t N, int64_t nnz, int64_t K, int64_t F, int op) {
  (void)nnz;
  size_t b = align_up((size_t)(N > 0 ? N : 1) * sizeof(int32_t)) + 256;  // node -> first entry
  if (op == TGPB200_MAX || op == TGPB200_MIN) b += align_up((size_t)(K * F > 0 ? K * F : 1) * sizeof(float));
  return b;
}

int tgpb200_segment_reduce_bwd(const void* x, const int64_t* node_index, const int64_t* cluster_index,
                               const float* weight, const int32_t* order, const int32_t* ptr, const void* x_pool,
                               const void* grad_pool, int64_t N, int64_t nnz, int64_t K, int64_t F, int op,
                               int x_dtype, int out_dtype, void* grad_x, float* grad_weight, void* workspace,
                               size_t workspace_bytes, tgpb200_stream_t stream) {
  if (N < 0 || nnz < 0 || K < 0 || F < 0 || op < TGPB200_SUM || op > TGPB200_MIN) return TGPB200_ERR_INVALID;
  if (nnz >= INT32_MAX || K >= INT32_MAX) return TGPB200_ERR_INVALID;  // the CSR (ptr / order) is 32-bit
  if (N * F == 0 && nnz == 0) return TGPB200_OK;
  if (!grad_x || !ptr || !grad_pool || (nnz > 0 && (!x || !node_index || !cluster_index))) return TGPB200_ERR_INVALID;
  if ((op == TGPB200_MAX || op == TGPB200_MIN) && (!x_pool || !order)) return TGPB200_ERR_INVALID;
  cudaStream_t st = (cudaStream_t)stream;
  Workspace ws(workspace, workspace_bytes);
  if (x_dtype == TGPB200_F32 && out_dtype == TGPB200_F32)
    return launch_bwd<float, float>(x, node_index, cluster_index, weight, order, ptr, x_pool, grad_pool, N, nnz, K, F,
                                    op, grad_x, grad_weight, ws, st);
  if (x_dtype == TGPB200_BF16 && out_dtype == TGPB200_BF16)
    return launch_bwd<__nv_bfloat16, __nv_bfloat16>(x, node_index, cluster_index, weight, order, ptr, x_pool, grad_pool,
                                                    N, nnz, K, F, op, grad_x, grad_weight, ws, st);
  return TGPB200_ERR_UNSUPPORTED;
}

int tgpb200_reduce_batch(const int64_t* batch, const int64_t* node_index, const int32_t* order, const int32_t* ptr,
                         int64_t K, int64_t* batch_pool, tgpb200_stream_t stream) {
  if (K < 0) return TGPB200_ERR_INVALID;
  if (K == 0) return TGPB200_OK;
  if (!batch_pool || !ptr || !batch || !node_index || !order) return TGPB200_ERR_INVALID;
  launch("k_reduce_batch", k_reduce_batch, (unsigned)ceil_div(K, 256), 256, 0, (cudaStream_t)stream, batch, node_index, order, ptr, K,
                                                                              batch_pool);
  return launch_status();
}

}  // extern "C"
