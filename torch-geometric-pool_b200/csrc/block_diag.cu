// Dense -> block-diagonal sparse conversion of the pooled adjacency, and the dense pre-processing scatters.
// Reference: dense_to_block_diag tgp/utils/ops.py:53-82; DenseSRCPooling._finalize_sparse_output tgp/src.py:500-557
// (mask the padded supernodes, keep |a| > eps in row-major (b, i, j) order, renumber the valid supernodes
// compactly); to_dense_batch / to_dense_adj of DenseSRCPooling.preprocessing tgp/src.py:434-450.
#include "prims.cuh"

namespace tgp {

static __global__ void k_mask_to_int(const uint8_t* __restrict__ mask, int64_t n, int* __restrict__ out) {
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) out[i] = mask[i] ? 1 : 0;
}

template <typename T>
struct BlockDiagPred {
  struct Payload {
    float w;
  };
  const T* adj;
  const uint8_t* mask;  // [B*K] or null
  int K;
  float eps;
  __device__ bool operator()(int64_t i, Payload& p) const {
    p.w = to_f32<T>(adj[i]);
    if (!(fabsf(p.w) > eps)) return false;
    if (mask) {
      int64_t kk = (int64_t)K * K;
      int64_t b = i / kk;
      int rc = (int)(i - b * kk);
      int r = rc / K, c = rc - r * K;
      if (!mask[b * K + r] || !mask[b * K + c]) return false;
    }
    return true;
  }
};
template <typename T>
struct BlockDiagEmit {
  int64_t* row;
  int64_t* col;
  T* w;
  int32_t* src;       // flat position in adj of every emitted edge (for the backward), may be null
  const int* new_id;  // exclusive scan of the mask (compact supernode ids), or null
  int K;
  __device__ void operator()(int64_t i, int pos, const typename BlockDiagPred<T>::Payload& p) const {
    int64_t kk = (int64_t)K * K;
    int64_t b = i / kk;
    int rc = (int)(i - b * kk);
    int r = rc / K, c = rc - r * K;
    int64_t gr = b * K + r, gc = b * K + c;
    row[pos] = new_id ? new_id[gr] : gr;
    col[pos] = new_id ? new_id[gc] : gc;
    w[pos] = from_f32<T>(p.w);
    if (src) src[pos] = (int32_t)i;
  }
};

// Workspace layout shared by the count and emit phases: the renumbering of the kept pooled nodes with its scan, and
// the compaction of the B K^2 entries.
struct BlockDiagPlan {
  int* new_id;
  Workspace scan, tiles;
  BlockDiagPlan(Workspace& ws, int64_t B, int64_t K) {
    new_id = ws.take<int>((size_t)(B * K > 0 ? B * K : 1));
    scan = ws.sub(scan_workspace_bytes(B * K));
    tiles = ws.sub(compact_workspace_bytes(B * K * K));
  }
};

// Workspace of tgpb200_graph_ptr: the scan of the B + 1 graph offsets.
struct GraphPtrLayout {
  Workspace scan;
  GraphPtrLayout(Workspace& ws, int64_t B) : scan(ws.sub(scan_workspace_bytes(B + 1))) {}
};

template <typename T>
static __global__ void k_scatter_grad(const T* __restrict__ gw, const int32_t* __restrict__ src, int64_t n,
                                      T* __restrict__ gadj) {
  int64_t j = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (j < n) gadj[src[j]] = gw[j];
}

// to_dense_batch: x [N, F] + sorted batch -> [B, Nmax, F] zero padded, mask [B, Nmax]
template <typename T>
static __global__ void k_to_dense_batch(const T* __restrict__ x, const int64_t* __restrict__ batch,
                                        const int* __restrict__ ptr, int64_t N, int F, int Nmax, T* __restrict__ out,
                                        uint8_t* __restrict__ mask) {
  int64_t n = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  int lane = threadIdx.x & 31;
  if (n >= N) return;
  int64_t b = batch[n];
  int local = (int)(n - ptr[b]);
  if (local >= Nmax) return;
  const T* src = x + n * F;
  T* dst = out + ((int64_t)b * Nmax + local) * F;
  for (int f = lane; f < F; f += 32) dst[f] = src[f];
  if (lane == 0 && mask) mask[(int64_t)b * Nmax + local] = 1;
}

// to_dense_adj: duplicates are summed (atomicAdd); default weight 1.0
static __global__ void k_to_dense_adj(const int64_t* __restrict__ row, const int64_t* __restrict__ col,
                                      const float* __restrict__ w, const int64_t* __restrict__ batch,
                                      const int* __restrict__ ptr, int64_t E, int Nmax, int transpose,
                                      float* __restrict__ adj) {
  int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= E) return;
  int64_t r = row[e], c = col[e];
  int64_t b = batch ? batch[r] : 0;
  int lr = (int)(r - ptr[b]), lc = (int)(c - ptr[b]);
  if (lr < 0 || lc < 0 || lr >= Nmax || lc >= Nmax) return;
  if (transpose) { int t = lr; lr = lc; lc = t; }
  atomicAdd(&adj[((int64_t)b * Nmax + lr) * Nmax + lc], w ? w[e] : 1.f);
}

static __global__ void k_graph_counts(const int64_t* __restrict__ batch, int64_t N, int64_t B, int* __restrict__ cnt) {
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= N) return;
  int64_t b = batch[i];
  if (b >= 0 && b < B) atomicAdd(&cnt[b], 1);
}

}  // namespace tgp

using namespace tgp;

extern "C" {

size_t tgpb200_block_diag_workspace_bytes(int64_t B, int64_t K) { return layout_bytes<BlockDiagPlan>(B, K); }

int tgpb200_block_diag_count(const void* adj, const uint8_t* out_mask, int64_t B, int64_t K, int dtype, float eps,
                             int64_t* num_valid_out, int64_t* count_out, void* workspace, size_t workspace_bytes,
                             tgpb200_stream_t stream) {
  if (B < 0 || K < 0 || !count_out || B * K * K >= INT32_MAX) return TGPB200_ERR_INVALID;
  cudaStream_t st = (cudaStream_t)stream;
  int64_t n = B * K * K;
  if (n == 0) {
    cudaMemsetAsync(count_out, 0, sizeof(int64_t), st);
    if (num_valid_out) cudaMemsetAsync(num_valid_out, 0, sizeof(int64_t), st);
    return launch_status();
  }
  if (!adj) return TGPB200_ERR_INVALID;
  Workspace ws(workspace, workspace_bytes);
  const BlockDiagPlan pl(ws, B, K);
  if (!ws.ok) return TGPB200_ERR_WORKSPACE;
  if (out_mask) {
    launch("k_mask_to_int", k_mask_to_int, (unsigned)ceil_div(B * K, 256), 256, 0, st, out_mask, B * K, pl.new_id);
    int rc = exclusive_scan_i32(pl.new_id, pl.new_id, B * K, nullptr, num_valid_out, pl.scan, st);
    if (rc) return rc;
  }
  if (dtype == TGPB200_F32) {
    BlockDiagPred<float> pred{(const float*)adj, out_mask, (int)K, eps};
    return compact_count(pred, n, pl.tiles, nullptr, count_out, st);
  }
  if (dtype == TGPB200_BF16) {
    BlockDiagPred<__nv_bfloat16> pred{(const __nv_bfloat16*)adj, out_mask, (int)K, eps};
    return compact_count(pred, n, pl.tiles, nullptr, count_out, st);
  }
  return TGPB200_ERR_UNSUPPORTED;
}

int tgpb200_block_diag_emit(const void* adj, const uint8_t* out_mask, int64_t B, int64_t K, int dtype, float eps,
                            int64_t* out_row, int64_t* out_col, void* out_weight, int32_t* src_pos, void* workspace,
                            size_t workspace_bytes, tgpb200_stream_t stream) {
  if (B < 0 || K < 0) return TGPB200_ERR_INVALID;
  int64_t n = B * K * K;
  if (n == 0) return TGPB200_OK;
  if (!adj || !out_row || !out_col || !out_weight) return TGPB200_ERR_INVALID;
  cudaStream_t st = (cudaStream_t)stream;
  Workspace ws(workspace, workspace_bytes);
  const BlockDiagPlan pl(ws, B, K);
  if (!ws.ok) return TGPB200_ERR_WORKSPACE;
  const int* new_id = out_mask ? pl.new_id : nullptr;
  if (dtype == TGPB200_F32) {
    BlockDiagPred<float> pred{(const float*)adj, out_mask, (int)K, eps};
    BlockDiagEmit<float> emit{out_row, out_col, (float*)out_weight, src_pos, new_id, (int)K};
    return compact_emit(pred, emit, n, pl.tiles, st);
  }
  if (dtype == TGPB200_BF16) {
    BlockDiagPred<__nv_bfloat16> pred{(const __nv_bfloat16*)adj, out_mask, (int)K, eps};
    BlockDiagEmit<__nv_bfloat16> emit{out_row, out_col, (__nv_bfloat16*)out_weight, src_pos, new_id, (int)K};
    return compact_emit(pred, emit, n, pl.tiles, st);
  }
  return TGPB200_ERR_UNSUPPORTED;
}

int tgpb200_block_diag_bwd(const void* grad_weight, const int32_t* src_pos, int64_t num_edges, int64_t total, int dtype,
                           void* grad_adj, tgpb200_stream_t stream) {
  if (num_edges < 0 || total < 0) return TGPB200_ERR_INVALID;
  if (total == 0) return TGPB200_OK;
  if (!grad_adj) return TGPB200_ERR_INVALID;
  cudaStream_t st = (cudaStream_t)stream;
  size_t es = dtype == TGPB200_BF16 ? 2 : 4;
  cudaMemsetAsync(grad_adj, 0, (size_t)total * es, st);
  if (num_edges > 0) {
    if (!grad_weight || !src_pos) return TGPB200_ERR_INVALID;
    unsigned grid = (unsigned)ceil_div(num_edges, 256);
    if (dtype == TGPB200_F32)
      launch("k_scatter_grad", k_scatter_grad<float>, grid, 256, 0, st, (const float*)grad_weight, src_pos, num_edges,
             (float*)grad_adj);
    else
      launch("k_scatter_grad", k_scatter_grad<__nv_bfloat16>, grid, 256, 0, st, (const __nv_bfloat16*)grad_weight,
             src_pos, num_edges, (__nv_bfloat16*)grad_adj);
  }
  return launch_status();
}

// ---- dense pre-processing (SURVEY 8f row 3): graph offsets, to_dense_batch, to_dense_adj
size_t tgpb200_graph_ptr_workspace_bytes(int64_t B) { return layout_bytes<GraphPtrLayout>(B); }

int tgpb200_graph_ptr(const int64_t* batch, int64_t N, int64_t B, int32_t* ptr, void* workspace, size_t workspace_bytes,
                      tgpb200_stream_t stream) {
  if (N < 0 || B <= 0 || !ptr) return TGPB200_ERR_INVALID;
  if (N > 0 && !batch) return TGPB200_ERR_INVALID;
  cudaStream_t st = (cudaStream_t)stream;
  Workspace ws(workspace, workspace_bytes);
  const GraphPtrLayout l(ws, B);
  if (!ws.ok) return TGPB200_ERR_WORKSPACE;
  cudaMemsetAsync(ptr, 0, (size_t)(B + 1) * sizeof(int32_t), st);
  if (N > 0) launch("k_graph_counts", k_graph_counts, (unsigned)ceil_div(N, 256), 256, 0, st, batch, N, B, ptr);
  return exclusive_scan_i32(ptr, ptr, B + 1, nullptr, nullptr, l.scan, st);
}

int tgpb200_to_dense_batch(const void* x, const int64_t* batch, const int32_t* ptr, int64_t N, int64_t F, int64_t B,
                           int64_t Nmax, int dtype, void* out, uint8_t* mask, tgpb200_stream_t stream) {
  if (N < 0 || F < 0 || B < 0 || Nmax < 0) return TGPB200_ERR_INVALID;
  cudaStream_t st = (cudaStream_t)stream;
  size_t es = dtype == TGPB200_BF16 ? 2 : 4;
  if (out && B * Nmax * F > 0) cudaMemsetAsync(out, 0, (size_t)(B * Nmax * F) * es, st);
  if (mask && B * Nmax > 0) cudaMemsetAsync(mask, 0, (size_t)(B * Nmax), st);
  if (N == 0 || F == 0) return launch_status();
  if (!x || !batch || !ptr || !out) return TGPB200_ERR_INVALID;
  unsigned grid = (unsigned)ceil_div(N * 32, 256);
  if (dtype == TGPB200_F32)
    launch("k_to_dense_batch", k_to_dense_batch<float>, grid, 256, 0, st, (const float*)x, batch, ptr, N, (int)F,
           (int)Nmax, (float*)out, mask);
  else if (dtype == TGPB200_BF16)
    launch("k_to_dense_batch", k_to_dense_batch<__nv_bfloat16>, grid, 256, 0, st, (const __nv_bfloat16*)x, batch, ptr, N,
           (int)F, (int)Nmax, (__nv_bfloat16*)out, mask);
  else
    return TGPB200_ERR_UNSUPPORTED;
  return launch_status();
}

int tgpb200_to_dense_adj(const int64_t* row, const int64_t* col, const float* w, const int64_t* batch,
                         const int32_t* ptr, int64_t E, int64_t B, int64_t Nmax, int transpose, float* adj,
                         tgpb200_stream_t stream) {
  if (E < 0 || B < 0 || Nmax < 0) return TGPB200_ERR_INVALID;
  cudaStream_t st = (cudaStream_t)stream;
  if (B * Nmax * Nmax > 0) {
    if (!adj) return TGPB200_ERR_INVALID;
    cudaMemsetAsync(adj, 0, (size_t)(B * Nmax * Nmax) * sizeof(float), st);
  }
  if (E == 0) return launch_status();
  if (!row || !col || !ptr) return TGPB200_ERR_INVALID;
  launch("k_to_dense_adj", k_to_dense_adj, (unsigned)ceil_div(E, 256), 256, 0, st, row, col, w, batch, ptr, E, (int)Nmax,
         transpose, adj);
  return launch_status();
}

}  // extern "C"
