// HOSC losses on a sparse adjacency (the unbatched mode): the same losses as dense_hosc.cu, with A given as a
// coalesced edge list over the padded node layout (node i of graph b at row b N + i), so no [B, N, N] array exists.
//   P_e  = (A A)_ij = sum_{k in out(i) ∩ in(j)} w_ik w_kj,   wM_e = P_e w_e    for every edge e = (i, j) of A
// is the one new product: a per-edge intersection of two sorted neighbour lists (k_hosc_isect_*).  The cut products
// [A S | d] and [A_M S | d^M] run through the segment-reduce kernel on S1 = [S | 1 | 0 ..], and the statistics, the
// loss reduction and the elementwise backward are the dense path's kernels (hosc.cuh) on the same padded arrays.
// Backward, per edge (gM_e = dL/dwM_e, H_e = gM_e w_e on A's pattern):
//   gA_e = <U_i, S1_j> + gM_e P_e + sum_{k in out(i) ∩ out(j)} H_ik w_jk + sum_{k in in(i) ∩ in(j)} w_ki H_kj
// with U = [Sa + grad(A S) | r + grad(d) | ..] (k_hosc_edge_dots), and the intersection kernel walks the other two
// list pairs.  Every sum has a fixed order and a fixed reduction tree; there are no float atomics.
#include <type_traits>

#include "hosc.cuh"

namespace tgp {
namespace {

constexpr int kHeavy = 1024;        // edges whose shorter lists exceed this go to one block each
constexpr int kHeavyBlocks = 592;   // 4 x 148 SMs: blocks of the heavy pass (a loop over the queue)
constexpr int kDotLanes = 8;        // lanes per edge of k_hosc_edge_dots

unsigned grid_of(int64_t threads, int block = 256) { return (unsigned)ceil_div(threads > 0 ? threads : 1, block); }

// The neighbour lists of one CSR: entries ptr[u] .. ptr[u + 1] of node u, keys ascending and unique (the adjacency
// is coalesced), one value per entry.
struct Lists {
  const int32_t* ptr;
  const int32_t* key;
  const float* val;
};

// This thread's share (thread t of G) of sum_{k in a(u) ∩ b(v)} a.val * b.val: the threads stride the shorter list
// and binary-search the longer one, so the partial depends on (t, G) and the lists only.
__device__ __forceinline__ float isect_partial(const Lists& a, int u, const Lists& b, int v, int t, int G) {
  const int a0 = a.ptr[u], a1 = a.ptr[u + 1], b0 = b.ptr[v], b1 = b.ptr[v + 1];
  const bool a_short = a1 - a0 <= b1 - b0;
  const int32_t *sk = a_short ? a.key : b.key, *lk = a_short ? b.key : a.key;
  const float *sv = a_short ? a.val : b.val, *lv = a_short ? b.val : a.val;
  const int s0 = a_short ? a0 : b0, s1 = a_short ? a1 : b1, l0 = a_short ? b0 : a0, l1 = a_short ? b1 : a1;
  float acc = 0.f;
  for (int p = s0 + t; p < s1; p += G) {
    const int k = sk[p];
    int lo = l0, hi = l1;
    while (lo < hi) {
      const int mid = (lo + hi) >> 1;
      if (lk[mid] < k) lo = mid + 1; else hi = mid;
    }
    if (lo < l1 && lk[lo] == k) acc = fmaf(sv[p], lv[lo], acc);
  }
  return acc;
}

__device__ __forceinline__ int short_len(const Lists& a, int u, const Lists& b, int v) {
  return min(a.ptr[u + 1] - a.ptr[u], b.ptr[v + 1] - b.ptr[v]);
}

// kPairs = 1 (forward): P_e = sum over (a[0], b[0]), wM_e = P_e w_e.
// kPairs = 2 (backward): gA_e += gM_e P_e + sum over (a[0], b[0]) + sum over (a[1], b[1]).
struct IsectArgs {
  Lists a[2], b[2];
  const int32_t *erow, *ecol;  // endpoints of every edge (32-bit)
  int64_t nnz;
  const float* w;    // forward: edge weights
  float *P, *wM;     // forward outputs
  const float *gM, *Pin;  // backward inputs
  float* gA;              // backward: in / out
  int* queue;             // [0] = count, then the heavy edges
};

template <int kPairs>
__device__ __forceinline__ void isect_store(const IsectArgs& A, int64_t e, float s0, float s1) {
  if (kPairs == 1) {
    A.P[e] = s0;
    A.wM[e] = s0 * A.w[e];
  } else {
    A.gA[e] = fmaf(A.gM[e], A.Pin[e], A.gA[e]) + (s0 + s1);
  }
}

// One warp per edge; edges with long lists on both sides are queued for k_hosc_isect_heavy.
template <int kPairs>
__global__ void __launch_bounds__(256) k_hosc_isect_warp(IsectArgs A) {
  const int64_t e = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (e >= A.nnz) return;
  const int u = A.erow[e], v = A.ecol[e];
  int work = short_len(A.a[0], u, A.b[0], v);
  if (kPairs == 2) work += short_len(A.a[1], u, A.b[1], v);
  if (work > kHeavy) {
    if (lane == 0) A.queue[1 + atomicAdd(A.queue, 1)] = (int)e;
    return;
  }
  const float s0 = warp_sum(isect_partial(A.a[0], u, A.b[0], v, lane, 32));
  const float s1 = kPairs == 2 ? warp_sum(isect_partial(A.a[1], u, A.b[1], v, lane, 32)) : 0.f;
  if (lane == 0) isect_store<kPairs>(A, e, s0, s1);
}

// One block per queued edge (the queue order does not matter: every edge's sum is its own fixed-shape reduction).
template <int kPairs>
__global__ void __launch_bounds__(256) k_hosc_isect_heavy(IsectArgs A) {
  __shared__ float red[32];
  const int n = A.queue[0];
  for (int q = blockIdx.x; q < n; q += gridDim.x) {
    const int64_t e = A.queue[1 + q];
    const int u = A.erow[e], v = A.ecol[e];
    const float s0 = block_sum(isect_partial(A.a[0], u, A.b[0], v, threadIdx.x, blockDim.x), red);
    const float s1 = kPairs == 2 ? block_sum(isect_partial(A.a[1], u, A.b[1], v, threadIdx.x, blockDim.x), red) : 0.f;
    if (threadIdx.x == 0) isect_store<kPairs>(A, e, s0, s1);
    __syncthreads();
  }
}

// 32-bit endpoints of the edges, the identity order of the row CSR (the edges are sorted by row), and -- when
// col_order is given -- the column lists: ckey[p] = row of edge col_order[p], cv0 / cv1 its values of v0 / v1.
__global__ void k_hosc_edge_index(const int64_t* __restrict__ row, const int64_t* __restrict__ col,
                                  const int32_t* __restrict__ col_order, const float* __restrict__ v0,
                                  const float* __restrict__ v1, int64_t nnz, int32_t* __restrict__ erow,
                                  int32_t* __restrict__ ecol, int32_t* __restrict__ iota, int32_t* __restrict__ ckey,
                                  float* __restrict__ cv0, float* __restrict__ cv1) {
  const int64_t p = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (p >= nnz) return;
  if (erow) erow[p] = (int32_t)row[p], ecol[p] = (int32_t)col[p];
  if (iota) iota[p] = (int32_t)p;
  if (ckey) {
    const int e = col_order[p];
    ckey[p] = (int32_t)row[e];
    if (cv0) cv0[p] = v0[e];
    if (cv1) cv1[p] = v1[e];
  }
}

// Edge gradient of the two cut products, kDotLanes lanes per edge (fixed tree):
//   g1_e = <Sa_i, S_j> + r_i + <U_i[:K], S_j> + U_iK   (dL/dA_ij through [A S | d]; Sa / U may be absent)
//   g2_e = <Sm_i, S_j> + rM_i                          (dL/dA_M[ij], motif term only)
// gA = g1; with the motif term gM = g2 and H = g2 w.
template <typename T>
__global__ void __launch_bounds__(256)
    k_hosc_edge_dots(const T* __restrict__ S, const T* __restrict__ Sa, const T* __restrict__ Sm,
                     const float* __restrict__ U, const float* __restrict__ r, const float* __restrict__ rM,
                     const float* __restrict__ w, const int32_t* __restrict__ erow, const int32_t* __restrict__ ecol,
                     int64_t nnz, int K, int K1, float* __restrict__ gA, float* __restrict__ gM,
                     float* __restrict__ H) {
  const int64_t e = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) / kDotLanes;
  const int sub = threadIdx.x % kDotLanes;
  const bool on = e < nnz;  // no early exit: the whole warp takes part in the shuffles
  const int64_t i = on ? erow[e] : 0, j = on ? ecol[e] : 0;
  float a1 = 0.f, a2 = 0.f;
  for (int k = sub; on && k < K; k += kDotLanes) {
    const float sj = to_f32<T>(S[j * K + k]);
    float u = 0.f;
    if (Sa) u = to_f32<T>(Sa[i * K + k]);
    if (U) u += U[i * K1 + k];
    a1 = fmaf(u, sj, a1);
    if (Sm) a2 = fmaf(to_f32<T>(Sm[i * K + k]), sj, a2);
  }
#pragma unroll
  for (int o = kDotLanes / 2; o > 0; o >>= 1) {
    a1 += __shfl_xor_sync(kFull, a1, o);
    a2 += __shfl_xor_sync(kFull, a2, o);
  }
  if (on && sub == 0) {
    float g1 = a1;
    if (Sa) g1 += r[i];
    if (U) g1 += U[i * K1 + K];
    gA[e] = g1;
    if (Sm) {
      const float g2 = a2 + rM[i];
      gM[e] = g2;
      H[e] = g2 * w[e];
    }
  }
}

// dS = sum of the present fp32 products (Y[4] has K1 columns: grad(A S) through A^T), in the operand dtype
template <typename T>
__global__ void k_hosc_ds_sum(const float* __restrict__ Y0, const float* __restrict__ Y1, const float* __restrict__ Y2,
                              const float* __restrict__ Y3, const float* __restrict__ Y4, int64_t total, int K, int K1,
                              T* __restrict__ dS) {
  const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= total) return;
  float v = 0.f;
  if (Y0) v += Y0[e] + Y1[e];
  if (Y2) v += Y2[e] + Y3[e];
  if (Y4) {
    const int64_t row = e / K;
    v += Y4[row * K1 + (e - row * K)];
  }
  dS[e] = from_f32<T>(v);
}

// The saved buffer: the per-edge motif terms and the dense path's statistics.
struct HoscSparseSaved {
  float *P, *wM;  // [nnz] (motif term only)
  float *d, *dM;  // [B N]
  float *n1, *m1, *nM, *mM, *sq;  // [B, K]
  HoscSparseSaved(Workspace& ws, int64_t B, int64_t N, int64_t K, int64_t nnz, int terms) {
    const size_t e = (size_t)(nnz > 0 ? nnz : 1);
    P = (terms & kMotif) ? ws.take<float>(e) : nullptr;
    wM = (terms & kMotif) ? ws.take<float>(e) : nullptr;
    d = ws.take<float>((size_t)(B * N));
    dM = ws.take<float>((size_t)(B * N));
    n1 = ws.take<float>((size_t)(B * K));
    m1 = ws.take<float>((size_t)(B * K));
    nM = ws.take<float>((size_t)(B * K));
    mM = ws.take<float>((size_t)(B * K));
    sq = ws.take<float>((size_t)(B * K));
  }
};

// The forward workspace: S1, [A_M S | d^M], the identity row order and, for the motif term, the 32-bit endpoints,
// the column lists and the heavy-edge queue.
template <typename T>
struct HoscSparseFwdLayout {
  T* S1;
  float* AMS1;
  int32_t *iota, *erow, *ecol, *ckey, *queue;
  float* cw;
  HoscSparseFwdLayout(Workspace& ws, int64_t B, int64_t N, int64_t K, int64_t nnz, int terms) {
    const size_t RK1 = (size_t)(B * N) * s1_width((int)K), e = (size_t)(nnz > 0 ? nnz : 1);
    const bool motif = terms & kMotif;
    S1 = ws.take<T>(RK1);
    AMS1 = motif ? ws.take<float>(RK1) : nullptr;
    iota = ws.take<int32_t>(e);
    erow = motif ? ws.take<int32_t>(e) : nullptr;
    ecol = motif ? ws.take<int32_t>(e) : nullptr;
    ckey = motif ? ws.take<int32_t>(e) : nullptr;
    cw = motif ? ws.take<float>(e) : nullptr;
    queue = motif ? ws.take<int32_t>(e + 1) : nullptr;
  }
};

// The backward workspace: the scaled assignments, the fp32 products of dS and, when the edge gradient is asked for,
// its per-edge terms and the lists of the motif backward.
template <typename T>
struct HoscSparseBwdLayout {
  T *Sa, *Sm;
  float* Y[5];
  float *r, *rM, *gM, *H, *cw, *cH;
  int32_t *iota, *erow, *ecol, *ckey, *queue;
  HoscSparseBwdLayout(Workspace& ws, int64_t B, int64_t N, int64_t K, int64_t nnz, int terms, bool grad_as1,
                      bool need_grad_weight) {
    const size_t R = (size_t)(B * N), RK = R * (size_t)K, e = (size_t)(nnz > 0 ? nnz : 1);
    const bool first = terms & kFirst, motif = terms & kMotif;
    Sa = first ? ws.take<T>(RK) : nullptr;
    Sm = motif ? ws.take<T>(RK) : nullptr;
    Y[0] = first ? ws.take<float>(RK) : nullptr;
    Y[1] = first ? ws.take<float>(RK) : nullptr;
    Y[2] = motif ? ws.take<float>(RK) : nullptr;
    Y[3] = motif ? ws.take<float>(RK) : nullptr;
    Y[4] = grad_as1 ? ws.take<float>(R * (size_t)s1_width((int)K)) : nullptr;
    iota = ws.take<int32_t>(e);
    r = ws.take<float>(R);
    rM = ws.take<float>(R);
    const bool edges = need_grad_weight, medges = need_grad_weight && motif;
    erow = edges ? ws.take<int32_t>(e) : nullptr;
    ecol = edges ? ws.take<int32_t>(e) : nullptr;
    gM = medges ? ws.take<float>(e) : nullptr;
    H = medges ? ws.take<float>(e) : nullptr;
    ckey = medges ? ws.take<int32_t>(e) : nullptr;
    cw = medges ? ws.take<float>(e) : nullptr;
    cH = medges ? ws.take<float>(e) : nullptr;
    queue = medges ? ws.take<int32_t>(e + 1) : nullptr;
  }
};

template <template <typename> class Layout, typename... Args>
size_t sparse_layout_bytes(int dtype, Args... args) {
  return dtype == TGPB200_F32 ? layout_bytes<Layout<float>>(args...) : layout_bytes<Layout<__nv_bfloat16>>(args...);
}

int sparse_check(const void* s, const int32_t* row_ptr, const int32_t* col_ptr, int64_t B, int64_t N, int64_t K,
                 int64_t nnz, int dtype, int terms) {
  if (!s || !row_ptr || !col_ptr || B < 0 || N < 1 || K < 2 || nnz < 0 || terms <= 0 || terms > 7)
    return TGPB200_ERR_INVALID;
  if (dtype != TGPB200_F32 && dtype != TGPB200_BF16) return TGPB200_ERR_UNSUPPORTED;
  if (B > kMaxGridY || B * N >= INT32_MAX || nnz >= INT32_MAX || K >= 32768) return TGPB200_ERR_UNSUPPORTED;
  return TGPB200_OK;
}

// out = A x (rows) or A^T x (columns) of fp32 / bf16 x [B N, F] into fp32: the segment-reduce kernel
int spmm(const void* x, int dtype, const int64_t* index, const float* w, const int32_t* order, const int32_t* ptr,
         int64_t R, int64_t nnz, int64_t F, float* out, cudaStream_t st) {
  return tgpb200_segment_reduce_fwd(x, index, w, order, ptr, R, nnz, R, F, TGPB200_SUM, dtype, TGPB200_F32, out,
                                    (tgpb200_stream_t)st);
}

IsectArgs isect_args(const int32_t* erow, const int32_t* ecol, int64_t nnz, int* queue) {
  IsectArgs A = {};
  A.erow = erow, A.ecol = ecol, A.nnz = nnz, A.queue = queue;
  return A;
}

template <int kPairs>
void isect_launch(const IsectArgs& A, cudaStream_t st) {
  cudaMemsetAsync(A.queue, 0, sizeof(int), st);
  launch("k_hosc_isect_warp", k_hosc_isect_warp<kPairs>, grid_of(A.nnz * 32), 256, 0, st, A);
  launch("k_hosc_isect_heavy", k_hosc_isect_heavy<kPairs>, kHeavyBlocks, 256, 0, st, A);
}

template <typename T>
int sparse_fwd(const int64_t* row, const int64_t* col, const float* w, const int32_t* row_ptr, const int32_t* col_ptr,
               const int32_t* col_order, const T* S, const float* graph_nodes, int B, int N, int K, int64_t nnz,
               int terms, float eps, float* losses, float* AS1, const HoscSparseSaved& sv,
               const HoscSparseFwdLayout<T>& l, cudaStream_t st) {
  const int K1 = s1_width(K), dt = std::is_same<T, float>::value ? TGPB200_F32 : TGPB200_BF16;
  const bool motif = terms & kMotif;
  const int64_t R = (int64_t)B * N;
  int rc;
  if (R > 0) {
    launch("k_hosc_pad", k_hosc_pad<T>, grid_of(R * K1), 256, 0, st, S, R, K, K1, l.S1);
    if (nnz > 0)
      launch("k_hosc_edge_index", k_hosc_edge_index, grid_of(nnz), 256, 0, st, row, col, col_order, w,
             (const float*)nullptr, nnz, l.erow, l.ecol, l.iota, l.ckey, l.cw, (float*)nullptr);
    rc = spmm(l.S1, dt, col, w, l.iota, row_ptr, R, nnz, K1, AS1, st);  // [A S | d], also the connect's A S
    if (rc) return rc;
    if (motif) {  // P, wM per edge, then [A_M S | d^M]
      if (nnz > 0) {
        IsectArgs A = isect_args(l.erow, l.ecol, nnz, l.queue);
        A.a[0] = Lists{row_ptr, l.ecol, w};     // out(i): w_ik
        A.b[0] = Lists{col_ptr, l.ckey, l.cw};  // in(j):  w_kj
        A.w = w, A.P = sv.P, A.wM = sv.wM;
        isect_launch<1>(A, st);
      }
      rc = spmm(l.S1, dt, col, sv.wM, l.iota, row_ptr, R, nnz, K1, l.AMS1, st);
      if (rc) return rc;
    }
    launch("k_hosc_stats", k_hosc_stats<T>, dim3((unsigned)ceil_div(K, 32), (unsigned)B), 256, 0, st, S,
           (const float*)AS1, (const float*)l.AMS1, N, K, K1, terms, eps, sv.d, sv.dM, sv.n1, sv.m1, sv.nM, sv.mM,
           sv.sq);
  }
  launch("k_hosc_finalize", k_hosc_finalize, 1, 256, 0, st, (const float*)sv.n1, (const float*)sv.m1,
         (const float*)sv.nM, (const float*)sv.mM, (const float*)sv.sq, graph_nodes, B, N, K, terms, losses);
  return launch_status();
}

template <typename T>
int sparse_bwd(const int64_t* row, const int64_t* col, const float* w, const int32_t* row_ptr, const int32_t* col_ptr,
               const int32_t* col_order, const T* S, const float* graph_nodes, const HoscSparseSaved& sv,
               const float* gl, const float* gAS1, int B, int N, int K, int64_t nnz, int terms, T* dS, float* gw,
               const HoscSparseBwdLayout<T>& l, cudaStream_t st) {
  const int K1 = s1_width(K), dt = std::is_same<T, float>::value ? TGPB200_F32 : TGPB200_BF16;
  const bool first = terms & kFirst, motif = terms & kMotif;
  const int64_t R = (int64_t)B * N, total = R * K;
  int rc;
  if (R == 0) return TGPB200_OK;
  launch("k_hosc_edge_index", k_hosc_edge_index, grid_of(nnz), 256, 0, st, row, col, col_order, w, (const float*)nullptr,
         nnz, l.erow, l.ecol, l.iota, (int32_t*)nullptr, (float*)nullptr, (float*)nullptr);
  if (first || motif)
    launch("k_hosc_scale", k_hosc_scale<T>, grid_of(total), 256, 0, st, S, (const float*)sv.m1, (const float*)sv.mM, gl,
           total, B, N, K, l.Sa, l.Sm);
  // dS = A Sa + A^T Sa + A_M Sm + A_M^T Sm (+ A^T grad(A S)) + the elementwise terms
  if (first) {
    if ((rc = spmm(l.Sa, dt, col, w, l.iota, row_ptr, R, nnz, K, l.Y[0], st))) return rc;
    if ((rc = spmm(l.Sa, dt, row, w, col_order, col_ptr, R, nnz, K, l.Y[1], st))) return rc;
  }
  if (motif) {
    if ((rc = spmm(l.Sm, dt, col, sv.wM, l.iota, row_ptr, R, nnz, K, l.Y[2], st))) return rc;
    if ((rc = spmm(l.Sm, dt, row, sv.wM, col_order, col_ptr, R, nnz, K, l.Y[3], st))) return rc;
  }
  if (gAS1 && (rc = spmm(gAS1, TGPB200_F32, row, w, col_order, col_ptr, R, nnz, K1, l.Y[4], st))) return rc;
  launch("k_hosc_ds_sum", k_hosc_ds_sum<T>, grid_of(total), 256, 0, st, (const float*)l.Y[0], (const float*)l.Y[1],
         (const float*)l.Y[2], (const float*)l.Y[3], (const float*)l.Y[4], total, K, K1, dS);
  launch("k_hosc_ds_elementwise", k_hosc_ds_elementwise<T>, grid_of(total), 256, 0, st, S, (const float*)sv.d,
         (const float*)sv.dM, (const float*)sv.n1, (const float*)sv.m1, (const float*)sv.nM, (const float*)sv.mM,
         (const float*)sv.sq, graph_nodes, gl, total, B, N, K, terms, dS);
  if (!gw || nnz == 0) return launch_status();
  launch("k_hosc_rows", k_hosc_rows<T>, grid_of(R * 32), 256, 0, st, S, (const float*)sv.n1, (const float*)sv.m1,
         (const float*)sv.nM, (const float*)sv.mM, gl, R, B, N, K, terms, l.r, l.rM);
  launch("k_hosc_edge_dots", k_hosc_edge_dots<T>, grid_of(nnz * kDotLanes), 256, 0, st, S, (const T*)l.Sa,
         (const T*)l.Sm, gAS1, (const float*)l.r, (const float*)l.rM, w, (const int32_t*)l.erow,
         (const int32_t*)l.ecol, nnz, K, K1, gw, l.gM, l.H);
  if (motif) {  // gA += gM P + sum_{out(i) ∩ out(j)} H_ik w_jk + sum_{in(i) ∩ in(j)} w_ki H_kj
    launch("k_hosc_edge_index", k_hosc_edge_index, grid_of(nnz), 256, 0, st, row, col, col_order, w,
           (const float*)l.H, nnz, (int32_t*)nullptr, (int32_t*)nullptr, (int32_t*)nullptr, l.ckey, l.cw, l.cH);
    IsectArgs A = isect_args(l.erow, l.ecol, nnz, l.queue);
    A.a[0] = Lists{row_ptr, l.ecol, l.H};   // out(i): H_ik
    A.b[0] = Lists{row_ptr, l.ecol, w};     // out(j): w_jk
    A.a[1] = Lists{col_ptr, l.ckey, l.cw};  // in(i):  w_ki
    A.b[1] = Lists{col_ptr, l.ckey, l.cH};  // in(j):  H_kj
    A.gM = l.gM, A.Pin = sv.P, A.gA = gw;
    isect_launch<2>(A, st);
  }
  return launch_status();
}

}  // namespace
}  // namespace tgp

using namespace tgp;

extern "C" {

size_t tgpb200_hosc_sparse_loss_saved_bytes(int64_t B, int64_t N, int64_t K, int64_t nnz, int terms) {
  if (B < 0 || N < 1 || K < 1 || nnz < 0) return 0;
  return layout_bytes<HoscSparseSaved>(B, N, K, nnz, terms);
}

size_t tgpb200_hosc_sparse_loss_fwd_workspace_bytes(int64_t B, int64_t N, int64_t K, int64_t nnz, int terms,
                                                    int dtype) {
  if (B < 0 || N < 1 || K < 1 || nnz < 0) return 0;
  return sparse_layout_bytes<HoscSparseFwdLayout>(dtype, B, N, K, nnz, terms);
}

size_t tgpb200_hosc_sparse_loss_bwd_workspace_bytes(int64_t B, int64_t N, int64_t K, int64_t nnz, int terms, int dtype,
                                                    int has_grad_as1, int need_grad_weight) {
  if (B < 0 || N < 1 || K < 1 || nnz < 0) return 0;
  return sparse_layout_bytes<HoscSparseBwdLayout>(dtype, B, N, K, nnz, terms, has_grad_as1 != 0,
                                                  need_grad_weight != 0);
}

int tgpb200_hosc_sparse_loss_fwd(const int64_t* row, const int64_t* col, const float* weight, const int32_t* row_ptr,
                                 const int32_t* col_ptr, const int32_t* col_order, const void* s,
                                 const float* graph_nodes, int64_t B, int64_t N, int64_t K, int64_t nnz, int dtype,
                                 int terms, float eps, float* losses, float* as1, void* saved, size_t saved_bytes,
                                 void* workspace, size_t workspace_bytes, tgpb200_stream_t stream) {
  int rc = sparse_check(s, row_ptr, col_ptr, B, N, K, nnz, dtype, terms);
  if (rc != TGPB200_OK) return rc;
  if (!losses || !as1 || (nnz > 0 && (!row || !col || !weight || !col_order))) return TGPB200_ERR_INVALID;
  Workspace sw(saved, saved_bytes), ws(workspace, workspace_bytes);
  cudaStream_t st = (cudaStream_t)stream;
  const HoscSparseSaved sv(sw, B, N, K, nnz, terms);
  if (dtype == TGPB200_F32) {
    const HoscSparseFwdLayout<float> l(ws, B, N, K, nnz, terms);
    if (!sw.ok || !ws.ok) return TGPB200_ERR_WORKSPACE;
    return sparse_fwd<float>(row, col, weight, row_ptr, col_ptr, col_order, (const float*)s, graph_nodes, (int)B,
                             (int)N, (int)K, nnz, terms, eps, losses, as1, sv, l, st);
  }
  const HoscSparseFwdLayout<__nv_bfloat16> l(ws, B, N, K, nnz, terms);
  if (!sw.ok || !ws.ok) return TGPB200_ERR_WORKSPACE;
  return sparse_fwd<__nv_bfloat16>(row, col, weight, row_ptr, col_ptr, col_order, (const __nv_bfloat16*)s,
                                   graph_nodes, (int)B, (int)N, (int)K, nnz, terms, eps, losses, as1, sv, l, st);
}

int tgpb200_hosc_sparse_loss_bwd(const int64_t* row, const int64_t* col, const float* weight, const int32_t* row_ptr,
                                 const int32_t* col_ptr, const int32_t* col_order, const void* s,
                                 const float* graph_nodes, const void* saved, size_t saved_bytes,
                                 const float* grad_losses, const float* grad_as1, int64_t B, int64_t N, int64_t K,
                                 int64_t nnz, int dtype, int terms, void* grad_s, float* grad_weight, void* workspace,
                                 size_t workspace_bytes, tgpb200_stream_t stream) {
  int rc = sparse_check(s, row_ptr, col_ptr, B, N, K, nnz, dtype, terms);
  if (rc != TGPB200_OK) return rc;
  if (!grad_s || !grad_losses || (nnz > 0 && (!row || !col || !weight || !col_order))) return TGPB200_ERR_INVALID;
  Workspace sw(const_cast<void*>(saved), saved_bytes), ws(workspace, workspace_bytes);
  cudaStream_t st = (cudaStream_t)stream;
  const HoscSparseSaved sv(sw, B, N, K, nnz, terms);
  const bool gas = grad_as1 != nullptr, gwt = grad_weight != nullptr;
  if (dtype == TGPB200_F32) {
    const HoscSparseBwdLayout<float> l(ws, B, N, K, nnz, terms, gas, gwt);
    if (!sw.ok || !ws.ok) return TGPB200_ERR_WORKSPACE;
    return sparse_bwd<float>(row, col, weight, row_ptr, col_ptr, col_order, (const float*)s, graph_nodes, sv,
                             grad_losses, grad_as1, (int)B, (int)N, (int)K, nnz, terms, (float*)grad_s, grad_weight, l,
                             st);
  }
  const HoscSparseBwdLayout<__nv_bfloat16> l(ws, B, N, K, nnz, terms, gas, gwt);
  if (!sw.ok || !ws.ok) return TGPB200_ERR_WORKSPACE;
  return sparse_bwd<__nv_bfloat16>(row, col, weight, row_ptr, col_ptr, col_order, (const __nv_bfloat16*)s,
                                   graph_nodes, sv, grad_losses, grad_as1, (int)B, (int)N, (int)K, nnz, terms,
                                   (__nv_bfloat16*)grad_s, grad_weight, l, st);
}

}  // extern "C"
