// Row-bucketed cluster connect (tgp/connect/base_conn.py:83-89: edge_index = cluster[edge_index], PyG coalesce).
//
// The generic path (sparse_connect.cu) remaps every edge to a 2 x bits(K) bit key and runs a global LSD radix sort:
// 5 passes over 20 M edges for the 1 M-node workload, ~12 passes over the edge list in total.  When the input edge
// list is sorted by row (PyG datasets, every coalesced list), the expensive half of that sort is already there: the
// edges of a fine node are contiguous, so the edges of a COARSE row are the union of its members' ranges, and the
// cluster CSR (members per coarse row, ascending node id) enumerates them in original edge order.  What is left is
// to order each coarse row's short neighbour list by coarse column, which fits in shared memory:
//
//   plan   fine row spans -> per-member entry counts -> exclusive scan ("virtual" positions: coarse row c owns
//          [rowoff[c], rowoff[c+1]), rows in ascending order) -> hub rows (more than kBkHub entries) flagged
//   tiles  one CTA per window of kBkTile virtual positions: gather the member ranges of the rows that start in the
//          window, map columns through the cluster map, rank every entry inside its own (short) row by counting,
//          combine each run in arrival (= original edge) order, apply the self-loop / tiny-weight filters and write
//          the surviving coarse edges at their virtual positions
//   hubs   coarse rows too long for a tile (power-law hubs) go through the radix sort restricted to their edges and
//          land in their own virtual ranges
//   emit   one order-preserving compaction of the virtual array into the int64 output (lexicographic by construction)
//
// The edge list is read twice (row spans, gather) and the output written once; everything in between moves 32-bit
// entries.  Exact same results as the generic path: stable order, in-order combination, same filters.
#include <limits.h>

#include "prims.cuh"

namespace tgp {

constexpr int kBkThreads = 512;
constexpr int kBkTile = 1536;  // virtual positions per tile window
constexpr int kBkHub = 512;    // coarse rows with more entries than this take the radix path
constexpr int kBkCap = 2048;   // >= kBkTile + kBkHub: entries (and members) a tile can hold
constexpr int kBkLongRun = 4096;  // hub runs longer than this are combined by a whole block

__device__ __forceinline__ int64_t clamp_cluster(int64_t c, int64_t K) { return (c < 0 || c >= K) ? K - 1 : c; }

__device__ __forceinline__ float combine_w(int op, float acc, float v) {
  if (op == TGPB200_SUM || op == TGPB200_MEAN) return __fadd_rn(acc, v);
  if (op == TGPB200_MAX) return fmaxf(acc, v);
  if (op == TGPB200_MIN) return fminf(acc, v);
  return __fmul_rn(acc, v);
}

// rs[v] / re[v] = first / one-past-last edge of fine row v in the row-sorted edge list (0 / 0 when absent)
static __global__ void k_fine_row_spans(const int64_t* __restrict__ row, int64_t E, int64_t N, int32_t* __restrict__ rs,
                                        int32_t* __restrict__ re) {
  // four consecutive edges per thread (two 128-bit loads), neighbours of the group from the adjacent lanes
  const int64_t e0 = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) * 4;
  if (e0 >= E) return;
  int64_t r[6];
  if (e0 + 4 <= E && (reinterpret_cast<uintptr_t>(row) & 15) == 0) {
    const longlong2 a = __ldcs(reinterpret_cast<const longlong2*>(row + e0));
    const longlong2 b = __ldcs(reinterpret_cast<const longlong2*>(row + e0 + 2));
    r[1] = a.x, r[2] = a.y, r[3] = b.x, r[4] = b.y;
  } else {
    for (int k = 0; k < 4; ++k) r[1 + k] = e0 + k < E ? row[e0 + k] : -1;
  }
  r[0] = e0 > 0 ? row[e0 - 1] : -1;
  r[5] = e0 + 4 < E ? row[e0 + 4] : -1;
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    const int64_t e = e0 + k, v = r[1 + k];
    if (e >= E || v < 0 || v >= N) continue;
    if (r[k] != v) rs[v] = (int32_t)e;
    if (r[k + 2] != v || e + 1 == E) re[v] = (int32_t)(e + 1);
  }
}

// cost[m] = entries of CSR member m: its degree, or one placeholder for an isolated node (so that the number of
// members of a tile is bounded by its number of entries); cost[N] = 0 closes the scan
static __global__ void k_member_cost(const int32_t* __restrict__ order, const int32_t* __restrict__ rs,
                                     const int32_t* __restrict__ re, int64_t N, int* __restrict__ cost) {
  int64_t m = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (m > N) return;
  if (m == N) {
    cost[N] = 0;
    return;
  }
  const int v = order[m];
  const int d = re[v] - rs[v];
  cost[m] = d > 1 ? d : 1;
}

// per member: start of its coarse row in the virtual array, its coarse row; hub rows flagged and counted
// plan[0] = total virtual entries (written by the scan), plan[1] = edges of hub rows, plan[2] = hub rows
static __global__ void k_member_rows(const int32_t* __restrict__ order, const int32_t* __restrict__ ptr,
                                     const int64_t* __restrict__ cluster, const int* __restrict__ voff,
                                     const int32_t* __restrict__ rs, const int32_t* __restrict__ re, int64_t N,
                                     int64_t K, int32_t* __restrict__ mrowoff, int32_t* __restrict__ mcrow,
                                     uint32_t* __restrict__ hubbits, unsigned long long* __restrict__ plan) {
  int64_t m = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (m >= N) return;
  const int v = order[m];
  const int64_t c = clamp_cluster(cluster[v], K);
  const int p0 = ptr[c], p1 = ptr[c + 1];
  const int ro = voff[p0];
  mrowoff[m] = ro;
  mcrow[m] = (int32_t)c;
  if (voff[p1] - ro > kBkHub) {
    atomicAdd(&plan[1], (unsigned long long)(re[v] - rs[v]));
    if (m == p0) {
      atomicOr(&hubbits[c >> 5], 1u << (c & 31));
      atomicAdd(&plan[2], 1ull);
    }
  }
}

static __global__ void k_fill_i32(int32_t* __restrict__ p, int64_t n, int32_t v) {
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) p[i] = v;
}

// tile_mlo[t] = first member whose coarse row starts in window t or later (tile_mlo is pre-filled with N)
static __global__ void k_tile_bounds(const int32_t* __restrict__ mrowoff, int64_t N, int ntiles,
                                     int32_t* __restrict__ tile_mlo) {
  int64_t m = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (m >= N) return;
  const int t = mrowoff[m] / kBkTile;
  const int tp = m > 0 ? mrowoff[m - 1] / kBkTile : -1;
  for (int u = tp + 1; u <= t && u <= ntiles; ++u) tile_mlo[u] = (int32_t)m;
}

// Counting keys of a row that are LARGER than cc: a + ~cc carries out of 32 bits exactly when a > cc, and the carries
// are summed with add-with-carry -- 4 IADD3 + 2 IADD3.X per four keys (two carries per IADD3.X) instead of the
// compare / add / predicated move the compiler emits for `n += a > cc` (12 instructions, one serial chain):
// `ncu` showed k_bucket_tiles issue-bound with 47 % of its instructions in this loop.
__device__ __forceinline__ void count_gt4(const uint4 v, uint32_t ncc, uint32_t& c0, uint32_t& c1) {
  [[maybe_unused]] uint32_t t;
  asm("add.cc.u32 %0, %3, %7;\n\taddc.u32 %1, %1, 0;\n\t"
      "add.cc.u32 %0, %4, %7;\n\taddc.u32 %2, %2, 0;\n\t"
      "add.cc.u32 %0, %5, %7;\n\taddc.u32 %1, %1, 0;\n\t"
      "add.cc.u32 %0, %6, %7;\n\taddc.u32 %2, %2, 0;"
      : "=r"(t), "+r"(c0), "+r"(c1)
      : "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w), "r"(ncc));
}
__device__ __forceinline__ void count_gt1(uint32_t a, uint32_t ncc, uint32_t& c) {
  [[maybe_unused]] uint32_t t;
  asm("add.cc.u32 %0, %2, %3;\n\taddc.u32 %1, %1, 0;" : "=r"(t), "+r"(c) : "r"(a), "r"(ncc));
}

struct BucketArgs {
  const int64_t* col;
  const float* w;  // null when unweighted
  const int64_t* cluster;
  const int32_t *order, *ptr, *rs, *re, *mrowoff, *mcrow;
  const int4* desc;
  const int* voff;
  const uint32_t* hubbits;
  int64_t N, K;
  int op;
  bool rsl;
  float eps;
  int32_t *t_row, *t_col, *t_len;  // virtual array (t_len optional)
  float *t_w, *t_aux;              // (t_aux optional: product of the non-zero members, MUL backward)
  int32_t* slot_tmp;               // optional: virtual position of the run every input edge joined
};

// tile descriptor {first member, one past the last member (hub row cut off), first virtual position, entries}
static __global__ void k_tile_desc(const int32_t* __restrict__ tile_mlo, const int32_t* __restrict__ mcrow,
                                   const int32_t* __restrict__ ptr, const int* __restrict__ voff,
                                   const uint32_t* __restrict__ hubbits, int ntiles, int4* __restrict__ desc) {
  int t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= ntiles) return;
  const int m_lo = tile_mlo[t];
  int m_hi = tile_mlo[t + 1];
  if (m_lo < m_hi) {
    const int cl = mcrow[m_hi - 1];  // at most one hub row starts in a window, and it is the last one
    if ((hubbits[cl >> 5] >> (cl & 31)) & 1u) m_hi = ptr[cl];
  }
  int4 d = make_int4(m_lo, m_hi, 0, 0);
  if (m_lo < m_hi) {
    d.z = voff[m_lo];
    d.w = voff[m_hi] - d.z;
  }
  desc[t] = d;
}

// One CTA per window.  Entries are gathered in arrival order (grouped by coarse row, original edge order inside a
// row), then every entry finds its rank inside its OWN row by counting (rows are short: 76 % of the entries of the
// power-law workload sit in rows of <= 64, and nothing longer than kBkHub reaches a tile) -- no sorting network, no
// block-wide synchronisation between steps, shared-memory reads that are broadcasts within a warp.  A thread owns
// at most kBkPer = kBkCap / kBkThreads entries, so every phase is a fixed, fully unrolled loop whose global loads
// are all issued before the first one is consumed.  kPacked: coarse column and arrival index share one 32-bit rank
// key (column < 2^21), so that the counting loop is one compare per element on 128-bit shared-memory reads.
constexpr int kBkPer = kBkCap / kBkThreads;

template <bool kPacked>
static __global__ void __launch_bounds__(kBkThreads) k_bucket_tiles(BucketArgs A) {
  __shared__ __align__(16) uint32_t s_cc[kBkCap + 4];  // rank key per entry (arrival order), kDummy for a placeholder
  __shared__ uint16_t s_mi[kBkCap];       // member of the entry
  __shared__ uint16_t s_sorted[kBkCap];   // arrival index at every (row, column, arrival)-sorted position
  __shared__ uint16_t m_voff[kBkCap + 1];  // member -> first entry (tile-relative)
  __shared__ uint16_t m_rk[kBkCap];       // member -> first member of its row (= row id inside the tile)
  __shared__ uint16_t r_end[kBkCap];      // first member of a row -> one past the row's last entry
  __shared__ int32_t m_es[kBkCap];        // member -> first edge, -1 for an isolated node
  constexpr uint32_t kDummy = 0xffffffffu;
  const int4 desc = A.desc[blockIdx.x];
  const int m_lo = desc.x, m_hi = desc.y, tile_base = desc.z, n_ent = desc.w;
  if (m_lo >= m_hi) return;
  const int n_mem = m_hi - m_lo;
  {
    int v[kBkPer], c[kBkPer];
#pragma unroll
    for (int k = 0; k < kBkPer; ++k) {
      const int i = threadIdx.x + k * kBkThreads;
      v[k] = i < n_mem ? A.order[m_lo + i] : 0;
      c[k] = i < n_mem ? A.mcrow[m_lo + i] : 0;
    }
#pragma unroll
    for (int k = 0; k < kBkPer; ++k) {
      const int i = threadIdx.x + k * kBkThreads;
      if (i < n_mem) {
        const int s = A.rs[v[k]], e = A.re[v[k]];
        m_voff[i] = (uint16_t)(A.voff[m_lo + i] - tile_base);
        m_es[i] = e > s ? s : -1;
        m_rk[i] = (uint16_t)(A.ptr[c[k]] - m_lo);  // first member of the row: ascending with the row, < n_mem
      }
    }
  }
  if (threadIdx.x == 0) m_voff[n_mem] = (uint16_t)n_ent;
  __syncthreads();
  for (int i = threadIdx.x; i < n_mem; i += kBkThreads)
    if (i + 1 == n_mem || m_rk[i + 1] != m_rk[i]) r_end[m_rk[i]] = m_voff[i + 1];
  // gather: entry j -> (member, edge) -> coarse column
  {
    int64_t e[kBkPer], q[kBkPer];
    int mem[kBkPer];
#pragma unroll
    for (int k = 0; k < kBkPer; ++k) {
      const int j = threadIdx.x + k * kBkThreads;
      e[k] = -1;
      mem[k] = 0;
      if (j < n_ent) {
        int lo = 0, hi = n_mem;  // largest member with m_voff <= j
        while (hi - lo > 1) {
          const int mid = (lo + hi) >> 1;
          if (m_voff[mid] <= j) lo = mid; else hi = mid;
        }
        mem[k] = lo;
        const int es = m_es[lo];
        if (es >= 0) e[k] = (int64_t)es + (j - m_voff[lo]);
      }
    }
#pragma unroll
    for (int k = 0; k < kBkPer; ++k) q[k] = e[k] >= 0 ? __ldg(A.col + e[k]) : 0;
#pragma unroll
    for (int k = 0; k < kBkPer; ++k) {
      if (q[k] < 0 || q[k] >= A.N) q[k] = 0;
      q[k] = e[k] >= 0 ? __ldg(A.cluster + q[k]) : (int64_t)((threadIdx.x * 7 + k) & 1023);
    }
#pragma unroll
    for (int k = 0; k < kBkPer; ++k) {
      const int j = threadIdx.x + k * kBkThreads;
      if (j < n_ent) {
        const uint32_t cc = (uint32_t)clamp_cluster(q[k], A.K);
        s_cc[j] = e[k] >= 0 ? (kPacked ? ((cc << 11) | (uint32_t)j) : cc) : kDummy;
        s_mi[j] = (uint16_t)mem[k];
      }
    }
  }
  __syncthreads();
  // rank inside the row: entries of the row with a smaller column, or the same column and an earlier arrival
#pragma unroll 1
  for (int k = 0; k < kBkPer; ++k) {
    const int j = threadIdx.x + k * kBkThreads;
    if (j >= n_ent) break;
    const uint32_t cc = s_cc[j];
    const uint16_t rk = m_rk[s_mi[j]];
    const int start = m_voff[rk], end = r_end[rk];
    int rank = 0;
    int q = start;
    if (kPacked) {  // keys are unique (arrival index in the low bits); dummies (all ones) rank last, ties impossible
      // rank = keys below cc = row length - 1 (the entry itself) - keys above cc
      const uint32_t ncc = ~cc;
      uint32_t g0 = 0, g1 = 0;
      for (; (q & 3) && q < end; ++q) count_gt1(s_cc[q], ncc, g0);
      for (; q + 4 <= end; q += 4) count_gt4(*reinterpret_cast<const uint4*>(s_cc + q), ncc, g0, g1);
      for (; q < end; ++q) count_gt1(s_cc[q], ncc, g1);
      rank = end - start - 1 - (int)(g0 + g1);
      if (cc == kDummy) {  // several placeholders of one row: order them by arrival
        rank = 0;
        for (q = start; q < end; ++q) rank += (s_cc[q] != kDummy) || q < j;
      }
    } else {
      for (; q < end; ++q) {
        const uint32_t cq = s_cc[q];
        rank += (cq < cc) || (cq == cc && q < j);
      }
    }
    s_sorted[start + rank] = (uint16_t)j;
  }
  __syncthreads();
  // run heads combine their members in arrival order; the first member's weight of every head is loaded up front
  {
    constexpr uint32_t kColMask = kPacked ? ~0x7ffu : ~0u;
    int64_t e0[kBkPer];
    float w0[kBkPer];
    int cr[kBkPer];
    bool head[kBkPer];
#pragma unroll
    for (int k = 0; k < kBkPer; ++k) {
      const int p = threadIdx.x + k * kBkThreads;
      head[k] = false;
      e0[k] = 0;
      cr[k] = 0;
      if (p < n_ent) {
        const int j = s_sorted[p];
        const uint32_t cc = s_cc[j];
        const int mi = s_mi[j];
        if (cc != kDummy && !(p > (int)m_voff[m_rk[mi]] && ((s_cc[s_sorted[p - 1]] ^ cc) & kColMask) == 0)) {
          head[k] = true;
          e0[k] = (int64_t)m_es[mi] + (j - m_voff[mi]);
          cr[k] = m_lo + mi;
        }
      }
    }
#pragma unroll
    for (int k = 0; k < kBkPer; ++k) {
      w0[k] = (head[k] && A.w) ? __ldg(A.w + e0[k]) : 1.f;
      cr[k] = head[k] ? __ldg(A.mcrow + cr[k]) : 0;
    }
#pragma unroll
    for (int k = 0; k < kBkPer; ++k) {
      if (!head[k]) continue;
      const int p = threadIdx.x + k * kBkThreads;
      const int j = s_sorted[p];
      const uint32_t cc = s_cc[j];
      const int end = r_end[m_rk[s_mi[j]]];
      const int tpos = tile_base + p;
      float acc = w0[k], prod_nz = 1.f;
      int len = 1, zeros = 0;
      if (A.t_aux) {
        if (acc == 0.f) zeros = 1; else prod_nz = acc;
      }
      if (A.slot_tmp) A.slot_tmp[e0[k]] = tpos;
      for (int q = p + 1; q < end; ++q) {  // duplicates of the coarse edge (rare, short)
        const int jq = s_sorted[q];
        if (((s_cc[jq] ^ cc) & kColMask) != 0) break;
        const int mi = s_mi[jq];
        const int64_t e = (int64_t)m_es[mi] + (jq - m_voff[mi]);
        if (A.w) {
          const float v = A.w[e];
          acc = combine_w(A.op, acc, v);
          if (A.t_aux) {
            if (v == 0.f) ++zeros; else prod_nz = __fmul_rn(prod_nz, v);
          }
        }
        if (A.slot_tmp) A.slot_tmp[e] = tpos;
        ++len;
      }
      const uint32_t col = kPacked ? (cc >> 11) : cc;
      if (A.w && A.op == TGPB200_MEAN) acc = __fdiv_rn(acc, (float)len);
      if (A.rsl && (uint32_t)cr[k] == col) continue;
      if (A.w && !(fabsf(acc) > A.eps)) continue;
      A.t_row[tpos] = cr[k];
      A.t_col[tpos] = (int32_t)col;
      if (A.w) A.t_w[tpos] = acc;
      if (A.t_len) A.t_len[tpos] = (A.t_aux && A.op == TGPB200_MUL) ? zeros : len;
      if (A.t_aux) A.t_aux[tpos] = prod_nz;
    }
  }
}

// The edges of the hub rows are enumerated through the hub MEMBERS (a compaction over the N members, not a scan of
// all E edges): member list + degree prefix, then one thread per hub edge.  Order = (coarse row, node, edge) =
// ascending original edge id inside a coarse row, so the stable sort keeps duplicates in arrival order.
struct HubMemPred {
  struct Payload {
    int v, c, deg;
  };
  const int32_t *order, *mcrow, *rs, *re;
  const uint32_t* hubbits;
  __device__ bool operator()(int64_t m, Payload& p) const {
    p.c = mcrow[m];
    if (!((hubbits[p.c >> 5] >> (p.c & 31)) & 1u)) return false;
    p.v = order[m];
    p.deg = re[p.v] - rs[p.v];
    return p.deg > 0;
  }
};
struct HubMemEmit {
  int32_t *hm_v, *hm_c;
  int* hoff;
  __device__ void operator()(int64_t, int pos, const HubMemPred::Payload& p) const {
    hm_v[pos] = p.v;
    hm_c[pos] = p.c;
    hoff[pos] = p.deg;
  }
};
static __global__ void k_hub_edges(const int64_t* __restrict__ col, const int64_t* __restrict__ cluster,
                                   const int32_t* __restrict__ rs, const int32_t* __restrict__ hm_v,
                                   const int32_t* __restrict__ hm_c, const int* __restrict__ hoff,
                                   const int64_t* __restrict__ n_mem_dev, const int64_t* __restrict__ n_edges_dev,
                                   int64_t N, int64_t K, int cb, unsigned long long* __restrict__ keys,
                                   uint32_t* __restrict__ vals) {
  const int64_t n = *n_edges_dev;
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  int lo = 0, hi = (int)*n_mem_dev;  // largest hub member with hoff <= i
  while (hi - lo > 1) {
    const int mid = (lo + hi) >> 1;
    if (hoff[mid] <= i) lo = mid; else hi = mid;
  }
  const int64_t e = (int64_t)rs[hm_v[lo]] + (i - hoff[lo]);
  int64_t q = col[e];
  if (q < 0 || q >= N) q = 0;
  const int64_t cc = clamp_cluster(cluster[q], K);
  keys[i] = ((unsigned long long)hm_c[lo] << cb) | (unsigned long long)cc;
  vals[i] = (uint32_t)e;
}

static __global__ void k_hub_first(const unsigned long long* __restrict__ ks, const int64_t* __restrict__ n_dev, int cb,
                                   int32_t* __restrict__ hubfirst) {
  const int64_t n = *n_dev;
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const unsigned long long c = ks[i] >> cb;
  if (i == 0 || (ks[i - 1] >> cb) != c) hubfirst[c] = (int32_t)i;
}

struct HubRunArgs {
  const unsigned long long* ks;
  const uint32_t* perm;
  const int64_t* n_dev;
  const float* w;
  const int32_t* hubfirst;
  const int32_t* ptr;
  const int* voff;
  int cb, op;
  bool rsl;
  float eps;
  int32_t *t_row, *t_col, *t_len;
  float *t_w, *t_aux;
  int32_t* slot_tmp;
  int* long_list;  // [0] = count, entries follow
};

__device__ __forceinline__ void hub_write(const HubRunArgs& A, unsigned long long key, int64_t i, float acc, int len,
                                          int zeros, float prod_nz) {
  const int64_t cr = (int64_t)(key >> A.cb), cc = (int64_t)(key & ((1ull << A.cb) - 1ull));
  if (A.w && A.op == TGPB200_MEAN) acc = __fdiv_rn(acc, (float)len);
  if (A.rsl && cr == cc) return;
  if (A.w && !(fabsf(acc) > A.eps)) return;
  const int tpos = A.voff[A.ptr[cr]] + (int)(i - A.hubfirst[cr]);
  A.t_row[tpos] = (int32_t)cr;
  A.t_col[tpos] = (int32_t)cc;
  if (A.w) A.t_w[tpos] = acc;
  if (A.t_len) A.t_len[tpos] = (A.t_aux && A.op == TGPB200_MUL) ? zeros : len;
  if (A.t_aux) A.t_aux[tpos] = prod_nz;
}

static __global__ void k_hub_runs(HubRunArgs A) {
  const int64_t n = *A.n_dev;
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const unsigned long long key = A.ks[i];
  if (i > 0 && A.ks[i - 1] == key) return;
  const int64_t cr = (int64_t)(key >> A.cb);
  const int tpos = A.voff[A.ptr[cr]] + (int)(i - A.hubfirst[cr]);
  float acc = 0.f, prod_nz = 1.f;
  int len = 0, zeros = 0;
  for (int64_t q = i; q < n && A.ks[q] == key; ++q) {
    if (len >= kBkLongRun) {  // hand the whole run to a block (fixed-shape reduction, see k_hub_long_runs)
      A.long_list[1 + atomicAdd(&A.long_list[0], 1)] = (int)i;
      return;
    }
    const uint32_t e = A.perm[q];
    if (A.w) {
      const float v = A.w[e];
      acc = len == 0 ? v : combine_w(A.op, acc, v);
      if (A.t_aux) {
        if (v == 0.f) ++zeros; else prod_nz = __fmul_rn(prod_nz, v);
      }
    }
    if (A.slot_tmp) A.slot_tmp[e] = tpos;
    ++len;
  }
  hub_write(A, key, i, acc, len, zeros, prod_nz);
}

// Runs longer than kBkLongRun (a few coarse columns taking most of a hub row): one block per run, thread-strided
// partials in double (sum / mean) or in the op itself, combined over the block in a fixed order.
static __global__ void __launch_bounds__(256) k_hub_long_runs(HubRunArgs A) {
  __shared__ double redd[256];
  __shared__ float redf[256];
  __shared__ int redi[256];
  __shared__ int s_len;
  const int64_t n = *A.n_dev;
  const int n_long = A.long_list[0];
  for (int r = blockIdx.x; r < n_long; r += gridDim.x) {
    const int64_t i = A.long_list[1 + r];
    const unsigned long long key = A.ks[i];
    const int64_t cr = (int64_t)(key >> A.cb);
    const int tpos = A.voff[A.ptr[cr]] + (int)(i - A.hubfirst[cr]);
    double sd = 0.0;
    float acc = 0.f, prod_nz = 1.f;
    int cnt = 0, zeros = 0;
    for (int64_t q = i + threadIdx.x; q < n && A.ks[q] == key; q += 256) {
      const uint32_t e = A.perm[q];
      if (A.w) {
        const float v = A.w[e];
        sd += (double)v;
        acc = cnt == 0 ? v : combine_w(A.op == TGPB200_MEAN ? TGPB200_SUM : A.op, acc, v);
        if (A.t_aux) {
          if (v == 0.f) ++zeros; else prod_nz = __fmul_rn(prod_nz, v);
        }
      }
      if (A.slot_tmp) A.slot_tmp[e] = tpos;
      ++cnt;
    }
    const bool add = A.op == TGPB200_SUM || A.op == TGPB200_MEAN;
    redd[threadIdx.x] = sd;
    redf[threadIdx.x] = acc;
    redi[threadIdx.x] = cnt;
    __syncthreads();
    if (threadIdx.x == 0) {  // threads with cnt == 0 hold no member (only past the end of the run)
      double tot = 0.0;
      float a = 0.f;
      int len = 0;
      for (int t = 0; t < 256; ++t) {
        if (redi[t] == 0) continue;
        tot += redd[t];
        a = len == 0 ? redf[t] : combine_w(add ? TGPB200_SUM : A.op, a, redf[t]);
        len += redi[t];
      }
      redf[0] = add ? (float)tot : a;
      s_len = len;
    }
    __syncthreads();
    const float total = redf[0];
    const int len = s_len;
    __syncthreads();
    // MUL bookkeeping (zero count, product of the non-zeros) over the block, fixed order
    redf[threadIdx.x] = prod_nz;
    redi[threadIdx.x] = zeros;
    __syncthreads();
    if (threadIdx.x == 0) {
      float p = 1.f;
      int z = 0;
      for (int t = 0; t < 256; ++t) p = __fmul_rn(p, redf[t]), z += redi[t];
      hub_write(A, key, i, total, len, z, p);
    }
    __syncthreads();
  }
}

// ---- emit: compaction of the virtual array ---------------------------------------------------------------------
struct VirtPred {
  struct Payload {};
  const int32_t* t_row;
  __device__ bool operator()(int64_t i, Payload&) const { return t_row[i] >= 0; }
};
struct VirtEmit {
  const int32_t *t_row, *t_col, *t_len;
  const float *t_w, *t_aux;
  int64_t *out_row, *out_col;
  float *out_w, *run_aux;
  int32_t *run_len, *tpos2out;
  __device__ void operator()(int64_t i, int pos, const VirtPred::Payload&) const {
    out_row[pos] = t_row[i];
    out_col[pos] = t_col[i];
    if (out_w) out_w[pos] = t_w[i];
    if (run_len) run_len[pos] = t_len[i];
    if (run_aux) run_aux[pos] = t_aux[i];
    if (tpos2out) tpos2out[i] = pos;
  }
};

// edge_slot[e] = output position of the run that input edge e went into (tile position -> compacted position).
// Four edges per thread: 128-bit reads / writes of the streams, the four table lookups in flight together.
static __global__ void k_slot_fixup(const int32_t* __restrict__ slot_tmp, const int32_t* __restrict__ tpos2out, int64_t E,
                                    int32_t* __restrict__ edge_slot) {
  const int64_t e = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) * 4;
  if (e >= E) return;
  if (e + 4 <= E && ((reinterpret_cast<uintptr_t>(slot_tmp) | reinterpret_cast<uintptr_t>(edge_slot)) & 15) == 0) {
    const int4 t = *reinterpret_cast<const int4*>(slot_tmp + e);
    int4 o;
    o.x = t.x >= 0 ? __ldg(tpos2out + t.x) : -1;
    o.y = t.y >= 0 ? __ldg(tpos2out + t.y) : -1;
    o.z = t.z >= 0 ? __ldg(tpos2out + t.z) : -1;
    o.w = t.w >= 0 ? __ldg(tpos2out + t.w) : -1;
    *reinterpret_cast<int4*>(edge_slot + e) = o;
  } else {
    for (int64_t i = e; i < E && i < e + 4; ++i) {
      const int t = slot_tmp[i];
      edge_slot[i] = t >= 0 ? tpos2out[t] : -1;
    }
  }
}

static int cb_of(int64_t K) {
  int b = 0;
  uint64_t v = K > 1 ? (uint64_t)K - 1 : 1;
  while (v) ++b, v >>= 1;
  return b < 1 ? 1 : b;
}

// Workspace layout shared by plan / count / emit (carved identically in the three calls).
struct BucketPlan {
  int32_t *rs, *re, *mrowoff, *mcrow, *tile_mlo, *hubfirst;
  int4* desc;
  int* voff;
  uint32_t* hubbits;
  unsigned long long* plan;  // [4] device copy of the plan
  int64_t* hub_count;
  int32_t *t_row, *t_col, *t_len, *tpos2out, *slot_tmp;
  float *t_w, *t_aux;
  unsigned long long *hk0, *hk1;
  uint32_t *hv0, *hv1;
  int32_t *hm_v, *hm_c;
  int* hoff;
  int64_t* hub_members;
  int* long_list;
  int* tile_counts;
  int64_t V;  // virtual capacity E + N
  int ntiles;
  bool ok;
  BucketPlan(Workspace& ws, int64_t E, int64_t N, int64_t K) {
    V = E + N;
    ntiles = (int)ceil_div(V > 0 ? V : 1, kBkTile);
    const size_t n = (size_t)(N > 0 ? N : 1), e = (size_t)(E > 0 ? E : 1), v = (size_t)(V > 0 ? V : 1);
    rs = ws.take<int32_t>(n);
    re = ws.take<int32_t>(n);
    voff = ws.take<int>(n + 1);
    mrowoff = ws.take<int32_t>(n);
    mcrow = ws.take<int32_t>(n);
    tile_mlo = ws.take<int32_t>((size_t)ntiles + 2);
    desc = ws.take<int4>((size_t)ntiles + 1);
    hubbits = ws.take<uint32_t>((size_t)(K / 32 + 1));
    hubfirst = ws.take<int32_t>((size_t)(K > 0 ? K : 1));
    plan = ws.take<unsigned long long>(4);
    hub_count = ws.take<int64_t>(1);
    t_row = ws.take<int32_t>(v);
    t_col = ws.take<int32_t>(v);
    t_w = ws.take<float>(v);
    t_len = ws.take<int32_t>(v);
    t_aux = ws.take<float>(v);
    tpos2out = ws.take<int32_t>(v);
    slot_tmp = ws.take<int32_t>(e);
    hk0 = ws.take<unsigned long long>(e);
    hk1 = ws.take<unsigned long long>(e);
    hv0 = ws.take<uint32_t>(e);
    hv1 = ws.take<uint32_t>(e);
    hm_v = ws.take<int32_t>(n);
    hm_c = ws.take<int32_t>(n);
    hoff = ws.take<int>(n + 1);
    hub_members = ws.take<int64_t>(1);
    long_list = ws.take<int>(e / kBkLongRun + 2);
    tile_counts = ws.take<int>((size_t)ceil_div(v, kCompactTile) + 1);
    ok = ws.ok;
  }
};

}  // namespace tgp

using namespace tgp;

extern "C" {

size_t tgpb200_bucket_coalesce_workspace_bytes(int64_t E, int64_t N, int64_t K) {
  const size_t n = (size_t)(N > 0 ? N : 1), e = (size_t)(E > 0 ? E : 1), v = n + e;
  return 8 * align_up((n + 1) * 4) + 256 + 5 * align_up((v / kBkTile + 4) * 4) + align_up((size_t)(K / 32 + 1) * 4) +
         align_up((size_t)(K > 0 ? K : 1) * 4) + 2 * 256 + 6 * align_up(v * 4) + align_up(e * 4) + 2 * align_up(e * 8) +
         2 * align_up(e * 4) + align_up((e / kBkLongRun + 2) * 4) + align_up((v / kCompactTile + 2) * 4) +
         2 * scan_workspace_bytes(N + 1) + radix_sort_workspace_bytes(E) + compact_onepass_workspace_bytes(N) + 8192;
}

// Phase 0: virtual layout of the coarse rows.  plan_out (device int64[4]) = {virtual entries, hub edges, hub rows, 0}.
// Large inputs read it back once to size the later launches exactly; small / graph-captured ones skip the read and
// launch at capacity (virt_cap = E + N, hub_cap = E).
int tgpb200_bucket_coalesce_plan(const int64_t* row, int64_t E, const int64_t* cluster_index, const int32_t* order,
                                 const int32_t* ptr, int64_t N, int64_t K, int64_t* plan_out, void* workspace,
                                 size_t workspace_bytes, tgpb200_stream_t stream) {
  if (E < 0 || N <= 0 || K <= 0 || !plan_out || !cluster_index || !order || !ptr) return TGPB200_ERR_INVALID;
  if (E + N >= INT32_MAX || K >= INT32_MAX) return TGPB200_ERR_UNSUPPORTED;
  if (E > 0 && !row) return TGPB200_ERR_INVALID;
  cudaStream_t st = (cudaStream_t)stream;
  Workspace ws(workspace, workspace_bytes);
  BucketPlan pl(ws, E, N, K);
  if (!pl.ok) return TGPB200_ERR_WORKSPACE;
  cudaMemsetAsync(pl.rs, 0, (size_t)N * 4, st);
  cudaMemsetAsync(pl.re, 0, (size_t)N * 4, st);
  cudaMemsetAsync(pl.hubbits, 0, (size_t)(K / 32 + 1) * 4, st);
  cudaMemsetAsync(pl.plan, 0, 4 * sizeof(unsigned long long), st);
  if (E > 0)
    launch("k_fine_row_spans", k_fine_row_spans, (unsigned)ceil_div(ceil_div(E, 4), 256), 256, 0, st, row, E, N, pl.rs, pl.re);
  launch("k_member_cost", k_member_cost, (unsigned)ceil_div(N + 1, 256), 256, 0, st, order, pl.rs, pl.re, N, pl.voff);
  int rc = exclusive_scan_i32(pl.voff, pl.voff, N + 1, nullptr, reinterpret_cast<int64_t*>(pl.plan), ws, st);
  if (rc != TGPB200_OK) return rc;
  launch("k_member_rows", k_member_rows, (unsigned)ceil_div(N, 256), 256, 0, st, order, ptr, cluster_index, pl.voff, pl.rs,
         pl.re, N, K, pl.mrowoff, pl.mcrow, pl.hubbits, pl.plan);
  launch("k_fill_i32", k_fill_i32, (unsigned)ceil_div(pl.ntiles + 2, 256), 256, 0, st, pl.tile_mlo,
         (int64_t)pl.ntiles + 2, (int32_t)N);
  launch("k_tile_bounds", k_tile_bounds, (unsigned)ceil_div(N, 256), 256, 0, st, pl.mrowoff, N, pl.ntiles + 1, pl.tile_mlo);
  launch("k_tile_desc", k_tile_desc, (unsigned)ceil_div(pl.ntiles, 256), 256, 0, st, pl.tile_mlo, pl.mcrow, ptr, pl.voff,
         pl.hubbits, pl.ntiles, pl.desc);
  cudaMemcpyAsync(plan_out, pl.plan, 4 * sizeof(int64_t), cudaMemcpyDeviceToDevice, st);
  return launch_status();
}

// Phase 1 + count: tiles, hub rows, survivor count.  virt_cap / hub_cap bound the launches (plan values, or E + N / E).
// need_slots: record the run of every input edge (backward).  Same workspace as the plan call.
int tgpb200_bucket_coalesce_count(const int64_t* row, const int64_t* col, const float* edge_weight, int64_t E,
                                  const int64_t* cluster_index, const int32_t* order, const int32_t* ptr, int64_t N,
                                  int64_t K, int op, uint32_t flags, float eps, int64_t virt_cap, int64_t hub_cap,
                                  int need_slots, int64_t* count_out, void* workspace, size_t workspace_bytes,
                                  tgpb200_stream_t stream) {
  if (E < 0 || N <= 0 || K <= 0 || !count_out || op < TGPB200_SUM || op > TGPB200_MUL) return TGPB200_ERR_INVALID;
  if (E + N >= INT32_MAX || K >= INT32_MAX) return TGPB200_ERR_UNSUPPORTED;
  cudaStream_t st = (cudaStream_t)stream;
  Workspace ws(workspace, workspace_bytes);
  BucketPlan pl(ws, E, N, K);
  if (!pl.ok) return TGPB200_ERR_WORKSPACE;
  if (virt_cap < 0 || virt_cap > pl.V) virt_cap = pl.V;
  if (hub_cap < 0 || hub_cap > E) hub_cap = E;
  const bool weighted = edge_weight != nullptr;
  const bool slots = need_slots != 0;
  const bool aux = slots && weighted && op == TGPB200_MUL;
  cudaMemsetAsync(pl.t_row, 0xff, (size_t)(virt_cap > 0 ? virt_cap : 1) * 4, st);
  if (slots) {
    cudaMemsetAsync(pl.slot_tmp, 0xff, (size_t)(E > 0 ? E : 1) * 4, st);
    cudaMemsetAsync(pl.tpos2out, 0xff, (size_t)(virt_cap > 0 ? virt_cap : 1) * 4, st);
  }
  const bool rsl = (flags & TGPB200_REMOVE_SELF_LOOPS) != 0;
  if (E > 0) {
    BucketArgs A;
    A.col = col, A.w = edge_weight, A.cluster = cluster_index;
    A.order = order, A.ptr = ptr, A.rs = pl.rs, A.re = pl.re, A.mrowoff = pl.mrowoff, A.mcrow = pl.mcrow;
    A.desc = pl.desc, A.voff = pl.voff, A.hubbits = pl.hubbits, A.N = N, A.K = K, A.op = op, A.rsl = rsl, A.eps = eps;
    A.t_row = pl.t_row, A.t_col = pl.t_col, A.t_len = slots ? pl.t_len : nullptr, A.t_w = pl.t_w;
    A.t_aux = aux ? pl.t_aux : nullptr, A.slot_tmp = slots ? pl.slot_tmp : nullptr;
    const int tiles = (int)ceil_div(virt_cap > 0 ? virt_cap : 1, kBkTile);
    if (K < (1 << 21))
      launch("k_bucket_tiles", k_bucket_tiles<true>, (unsigned)tiles, kBkThreads, 0, st, A);
    else
      launch("k_bucket_tiles", k_bucket_tiles<false>, (unsigned)tiles, kBkThreads, 0, st, A);
    if (hub_cap > 0) {
      const int cb = cb_of(K);
      HubMemPred pred{order, pl.mcrow, pl.rs, pl.re, pl.hubbits};
      HubMemEmit emit{pl.hm_v, pl.hm_c, pl.hoff};
      cudaMemsetAsync(pl.hoff, 0, (size_t)(N + 1) * sizeof(int), st);
      int rc = compact_onepass(pred, emit, N, pl.hub_members, ws, st);
      if (rc != TGPB200_OK) return rc;
      rc = exclusive_scan_i32(pl.hoff, pl.hoff, N + 1, nullptr, pl.hub_count, ws, st);
      if (rc != TGPB200_OK) return rc;
      launch("k_hub_edges", k_hub_edges, (unsigned)ceil_div(hub_cap, 256), 256, 0, st, col, cluster_index, pl.rs, pl.hm_v,
             pl.hm_c, pl.hoff, pl.hub_members, pl.hub_count, N, K, cb, pl.hk0, pl.hv0);
      bool in1 = false;
      rc = radix_sort_pairs<unsigned long long>(pl.hk0, pl.hv0, pl.hv0, pl.hk1, pl.hv1, hub_cap, 2 * cb, &in1, ws, st,
                                                pl.hub_count);
      if (rc != TGPB200_OK) return rc;
      HubRunArgs H;
      H.ks = in1 ? pl.hk1 : pl.hk0, H.perm = in1 ? pl.hv1 : pl.hv0, H.n_dev = pl.hub_count, H.w = edge_weight;
      H.hubfirst = pl.hubfirst, H.ptr = ptr, H.voff = pl.voff, H.cb = cb, H.op = op, H.rsl = rsl, H.eps = eps;
      H.t_row = pl.t_row, H.t_col = pl.t_col, H.t_len = slots ? pl.t_len : nullptr, H.t_w = pl.t_w;
      H.t_aux = aux ? pl.t_aux : nullptr, H.slot_tmp = slots ? pl.slot_tmp : nullptr, H.long_list = pl.long_list;
      cudaMemsetAsync(pl.long_list, 0, sizeof(int), st);
      const unsigned hg = (unsigned)ceil_div(hub_cap, 256);
      launch("k_hub_first", k_hub_first, hg, 256, 0, st, H.ks, pl.hub_count, cb, pl.hubfirst);
      launch("k_hub_runs", k_hub_runs, hg, 256, 0, st, H);
      const int64_t lcap = hub_cap / kBkLongRun + 1;
      launch("k_hub_long_runs", k_hub_long_runs, (unsigned)(lcap < 592 ? lcap : 592), 256, 0, st, H);
    }
  }
  VirtPred vp{pl.t_row};
  return compact_count(vp, virt_cap, pl.tile_counts, nullptr, count_out, st);
}

// Phase 2: write the coarse edge list (int64 at the boundary).  edge_slot / run_len / run_aux as in
// tgpb200_remap_coalesce_emit (run_len holds the number of zero members and run_aux the product of the non-zero
// members for op = MUL: exact product-rule gradients with zero weights); they need need_slots != 0 in the count call.
int tgpb200_bucket_coalesce_emit(int64_t E, int64_t N, int64_t K, int weighted, int64_t virt_cap, int64_t* out_row,
                                 int64_t* out_col, float* out_weight, int32_t* edge_slot, int32_t* run_len,
                                 float* run_aux, void* workspace, size_t workspace_bytes, tgpb200_stream_t stream) {
  if (E < 0 || N <= 0 || K <= 0) return TGPB200_ERR_INVALID;
  if (E + N >= INT32_MAX || K >= INT32_MAX) return TGPB200_ERR_UNSUPPORTED;
  if (!out_row || !out_col || (weighted && !out_weight)) return TGPB200_ERR_INVALID;
  cudaStream_t st = (cudaStream_t)stream;
  Workspace ws(workspace, workspace_bytes);
  BucketPlan pl(ws, E, N, K);
  if (!pl.ok) return TGPB200_ERR_WORKSPACE;
  if (virt_cap < 0 || virt_cap > pl.V) virt_cap = pl.V;
  VirtPred vp{pl.t_row};
  VirtEmit ve{pl.t_row, pl.t_col, pl.t_len, pl.t_w, pl.t_aux, out_row, out_col, weighted ? out_weight : nullptr,
              run_aux, run_len, edge_slot ? pl.tpos2out : nullptr};
  int rc = compact_emit(vp, ve, virt_cap, pl.tile_counts, st);
  if (rc != TGPB200_OK) return rc;
  if (edge_slot && E > 0)
    launch("k_slot_fixup", k_slot_fixup, (unsigned)ceil_div(ceil_div(E, 4), 256), 256, 0, st, pl.slot_tmp, pl.tpos2out, E, edge_slot);
  return launch_status();
}

}  // extern "C"
