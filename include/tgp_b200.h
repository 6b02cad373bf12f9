/*
 * tgp_b200.h -- C ABI of libtgp_b200.so: B200 (sm_100a) kernels for the Reduce + Connect
 * hot path of tgp-team/torch-geometric-pool (reference tree: /root/reference, v1.0.1).
 *
 * Conventions
 *   - plain pointers and sizes only; every pointer is a DEVICE pointer unless named host_*;
 *   - index tensors are int64 at the boundary (reference enforces it, tgp/utils/ops.py:472-476),
 *     narrowed to int32 internally (all extents must be < 2^31);
 *   - inputs are borrowed and never written; outputs are caller-allocated;
 *   - no allocation and no global state inside: scratch comes from `workspace`
 *     (size from the matching *_workspace_bytes query); kernels are enqueued on `stream`
 *     and never synchronise, so every call is CUDA-graph capturable;
 *   - return value: TGPB200_OK or a negative TGPB200_ERR_* code (no exceptions cross the ABI).
 *
 * Each entry point names the reference interface (file:line under /root/reference) it replaces.
 */
#ifndef TGP_B200_H_
#define TGP_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct CUstream_st* tgpb200_stream_t;

#define TGPB200_OK 0
#define TGPB200_ERR_INVALID (-1)     /* bad argument (null pointer, negative size, unknown enum) */
#define TGPB200_ERR_WORKSPACE (-2)   /* workspace too small */
#define TGPB200_ERR_CUDA (-3)        /* a launch failed: see cudaGetLastError */
#define TGPB200_ERR_UNSUPPORTED (-4) /* shape/dtype outside what the kernels cover */

/* element types of feature / weight / adjacency tensors */
#define TGPB200_F32 0
#define TGPB200_BF16 1

/* reduce ops: tgp/utils/typing.py:15 ConnectionType, tgp/reduce/get_aggr.py aliases */
#define TGPB200_SUM 0
#define TGPB200_MEAN 1
#define TGPB200_MAX 2
#define TGPB200_MIN 3
#define TGPB200_MUL 4

/* post-processing flags (SparseConnect / DenseConnect ctor attributes) */
#define TGPB200_REMOVE_SELF_LOOPS 1u
#define TGPB200_DEGREE_NORM 2u
#define TGPB200_ADJ_TRANSPOSE 4u
#define TGPB200_EDGE_WEIGHT_NORM 8u
#define TGPB200_HAS_WEIGHT 16u

int tgpb200_abi_version(void);
/* number of kernels this library has launched in the process so far (diagnostics; bench.py reports it) */
long long tgpb200_debug_launch_count(void);
/* Per-kernel timing for bench.py: bracket every kernel whose name contains `filter` with CUDA events on its launch
 * stream (NULL stops and resets); tgpb200_debug_kernel_time_ms returns the mean duration of the recorded launches. */
void tgpb200_debug_time_kernel(const char* filter);
double tgpb200_debug_kernel_time_ms(int* count);
/* Trace of the recorded launches ("*" as the filter records every kernel), in launch order: one
 * "name<TAB>ms" line per launch; returns the bytes written into host `buf`. */
size_t tgpb200_debug_kernel_times(char* host_buf, size_t cap);

/* ------------------------------------------------------------------------------------------
 * CSR-by-cluster of a sparse assignment (replaces the stable torch.sort in
 * tgp/reduce/aggr_reduce.py:13-23 and the atomic scatter order of base_reduce.py:147-153).
 * order[ptr[c] .. ptr[c+1]) = positions i (ascending) with cluster_index[i] == c.
 * ------------------------------------------------------------------------------------------ */
size_t tgpb200_build_csr_workspace_bytes(int64_t nnz, int64_t num_clusters);
int tgpb200_build_csr(const int64_t* cluster_index, int64_t nnz, int64_t num_clusters, int32_t* order,
                      int32_t* ptr, void* workspace, size_t workspace_bytes, tgpb200_stream_t stream);

/* ------------------------------------------------------------------------------------------
 * Sparse reduce:  x_pool[c] = op_{i in c} weight[i] * x[node_index[i]]
 * BaseReduce.forward sparse path  tgp/reduce/base_reduce.py:141-155  (op = SUM)
 * AggrReduce.forward sparse path  tgp/reduce/aggr_reduce.py:99-105   (SUM / MEAN / MAX / MIN)
 * Members are combined in ascending position order (deterministic); empty clusters give 0 rows.
 * weight is fp32 [nnz] (may be NULL = ones).  x is [num_nodes, F] row-major of x_dtype,
 * x_pool is [num_clusters, F] of out_dtype.
 * ------------------------------------------------------------------------------------------ */
int tgpb200_segment_reduce_fwd(const void* x, const int64_t* node_index, const float* weight, const int32_t* order,
                               const int32_t* ptr, int64_t num_nodes, int64_t nnz, int64_t num_clusters, int64_t F,
                               int op, int x_dtype, int out_dtype, void* x_pool, tgpb200_stream_t stream);

/* Backward of the above (the reference gets it from autograd).  grad_x [num_nodes, F] (x_dtype) is fully
 * written (rows of unselected nodes are zero); grad_weight [nnz] fp32 may be NULL.  For MAX / MIN the
 * gradient is split evenly among ties (torch scatter_reduce amax/amin rule, the PyG CPU path);
 * x_pool (forward output) is required for those ops.  node_index must be sorted ascending
 * (SelectOutput invariant, tgp/select/base_select.py:56-60). */
size_t tgpb200_segment_reduce_bwd_workspace_bytes(int64_t num_nodes, int64_t nnz, int64_t num_clusters, int64_t F,
                                                  int op);
int tgpb200_segment_reduce_bwd(const void* x, const int64_t* node_index, const int64_t* cluster_index,
                               const float* weight, const int32_t* order, const int32_t* ptr, const void* x_pool,
                               const void* grad_pool, int64_t num_nodes, int64_t nnz, int64_t num_clusters, int64_t F,
                               int op, int x_dtype, int out_dtype, void* grad_x, float* grad_weight, void* workspace,
                               size_t workspace_bytes, tgpb200_stream_t stream);

/* Reduce.reduce_batch sparse branch  tgp/reduce/base_reduce.py:37-41:
 * out = arange(K); out[cluster_index[i]] = batch[node_index[i]]  (CPU scatter_: the last writer in
 * position order wins = the last member in the CSR; an empty cluster keeps its arange value). */
int tgpb200_reduce_batch(const int64_t* batch, const int64_t* node_index, const int32_t* order, const int32_t* ptr,
                         int64_t num_clusters, int64_t* batch_pool, tgpb200_stream_t stream);

/* ------------------------------------------------------------------------------------------
 * Sparse connect, kept-node branch  tgp/connect/base_conn.py:79-82 (PyG subgraph, relabel_nodes=True)
 * fused with the filters of postprocess_adj_pool_sparse  tgp/utils/ops.py:370-380.
 * Keeps edge e iff both endpoints are in node_index, (flags & REMOVE_SELF_LOOPS) => row != col,
 * (edge_weight != NULL) => |w| > eps.  Input order is preserved; endpoints are relabelled to their
 * position in node_index.  Outputs are written compacted into caller buffers of capacity num_edges;
 * *count_out (device int64) receives the number of surviving edges;
 * src_edge[j] (int32, may be NULL) = input position of output edge j (saved for backward).
 * ------------------------------------------------------------------------------------------ */
size_t tgpb200_filter_relabel_workspace_bytes(int64_t num_edges, int64_t num_nodes);
/* Phase 1 builds the relabel table and counts survivors; the caller reads *count_out (the one
 * unavoidable device->host word, since the reference returns exact-size tensors), allocates the
 * outputs and calls phase 2 with the SAME workspace. */
int tgpb200_filter_relabel_count(const int64_t* row, const int64_t* col, const float* edge_weight, int64_t num_edges,
                                 const int64_t* node_index, int64_t num_kept, int64_t num_nodes, uint32_t flags,
                                 float eps, int64_t* count_out, void* workspace, size_t workspace_bytes,
                                 tgpb200_stream_t stream);
int tgpb200_filter_relabel_emit(const int64_t* row, const int64_t* col, const float* edge_weight, int64_t num_edges,
                                int64_t num_nodes, uint32_t flags, float eps, int64_t* out_row, int64_t* out_col,
                                float* out_weight, int32_t* src_edge, void* workspace, size_t workspace_bytes,
                                tgpb200_stream_t stream);
/* Single-pass form (decoupled look-back compaction): the edge list is read once.  The outputs must have capacity
 * num_edges; *count_out receives the survivor count when the stream has drained. */
size_t tgpb200_filter_relabel_onepass_workspace_bytes(int64_t num_edges, int64_t num_nodes);
int tgpb200_filter_relabel_onepass(const int64_t* row, const int64_t* col, const float* edge_weight, int64_t num_edges,
                                   const int64_t* node_index, int64_t num_kept, int64_t num_nodes, uint32_t flags,
                                   float eps, int64_t* out_row, int64_t* out_col, float* out_weight, int32_t* src_edge,
                                   int64_t* count_out, void* workspace, size_t workspace_bytes,
                                   tgpb200_stream_t stream);
/* Backward: grad_in[src_edge[j]] = grad_out[j], zero elsewhere.  num_out_dev (may be NULL) is a device-side
 * count <= num_out for callers that never read the survivor count back (grad_out then has capacity num_out). */
int tgpb200_filter_relabel_bwd(const float* grad_out, const int32_t* src_edge, int64_t num_out,
                               const int64_t* num_out_dev, int64_t num_edges, float* grad_in, tgpb200_stream_t stream);

/* ------------------------------------------------------------------------------------------
 * Sparse connect, cluster branch  tgp/connect/base_conn.py:83-89:
 * edge_index = cluster_index[edge_index]; PyG coalesce(num_nodes=K, reduce=op) (stable sort by row*K+col,
 * duplicates combined in original order), then the filters of tgp/utils/ops.py:370-380.
 * Output is lexicographic (row, col).  edge_weight == NULL => duplicates dropped, no weights out.
 * edge_slot[e] (int32 [E], may be NULL) = output position of the run edge e was merged into, or -1.
 * run_len[j] (int32, may be NULL) = number of input edges merged into output edge j.
 * Two phases sharing one workspace, as above.
 * ------------------------------------------------------------------------------------------ */
size_t tgpb200_remap_coalesce_workspace_bytes(int64_t num_edges, int64_t num_clusters);
int tgpb200_remap_coalesce_count(const int64_t* row, const int64_t* col, const float* edge_weight, int64_t num_edges,
                                 const int64_t* cluster_index, int64_t num_nodes, int64_t num_clusters, int op,
                                 uint32_t flags, float eps, int64_t* count_out, void* workspace,
                                 size_t workspace_bytes, tgpb200_stream_t stream);
int tgpb200_remap_coalesce_emit(int64_t num_edges, int64_t num_clusters, int weighted, uint32_t flags, float eps,
                                int64_t* out_row, int64_t* out_col, float* out_weight, int32_t* edge_slot,
                                int32_t* run_len, void* workspace, size_t workspace_bytes, tgpb200_stream_t stream);

/* Backward of the coalesce: grad_in[e] = d out_weight[slot(e)] / d w[e] * grad_out[slot(e)]  (0 if dropped).
 * SUM: 1; MEAN: 1/len; MAX/MIN: even split among ties; MUL: out/w[e] -- or, when run_aux is given (row-bucketed
 * path: run_len = number of zero members, run_aux = product of the non-zero members), the exact product rule. */
int tgpb200_coalesce_bwd(const float* edge_weight, const float* out_weight, const float* grad_out,
                         const int32_t* edge_slot, const int32_t* run_len, const float* run_aux, int64_t num_edges,
                         int64_t num_out, int op, float* grad_in, void* workspace, size_t workspace_bytes,
                         tgpb200_stream_t stream);

/* ------------------------------------------------------------------------------------------
 * Row-bucketed form of the cluster branch for ROW-SORTED edge lists (csrc/sparse_coalesce.cu): same results as
 * tgpb200_remap_coalesce_*, ~2 passes over the edges instead of ~12.  `order` / `ptr` = tgpb200_build_csr of
 * cluster_index (one entry per fine node: node_index = arange(N)).  Three calls sharing one workspace:
 *   plan   virtual layout; plan_out (device int64[4]) = {virtual entries, edges of hub rows, hub rows, 0};
 *   count  tiles + hub rows + survivor count.  virt_cap / hub_cap bound the launches: the values read back from
 *          plan_out (large inputs, one host read) or -1 = capacity (E + N, E) for callers that never synchronise;
 *   emit   writes the lexicographic coarse edge list; edge_slot / run_len / run_aux need need_slots != 0 in count.
 * Returns TGPB200_ERR_UNSUPPORTED when E + N >= 2^31 (use the generic path).
 * ------------------------------------------------------------------------------------------ */
size_t tgpb200_bucket_coalesce_workspace_bytes(int64_t num_edges, int64_t num_nodes, int64_t num_clusters);
int tgpb200_bucket_coalesce_plan(const int64_t* row, int64_t num_edges, const int64_t* cluster_index,
                                 const int32_t* order, const int32_t* ptr, int64_t num_nodes, int64_t num_clusters,
                                 int64_t* plan_out, void* workspace, size_t workspace_bytes, tgpb200_stream_t stream);
int tgpb200_bucket_coalesce_count(const int64_t* row, const int64_t* col, const float* edge_weight, int64_t num_edges,
                                  const int64_t* cluster_index, const int32_t* order, const int32_t* ptr,
                                  int64_t num_nodes, int64_t num_clusters, int op, uint32_t flags, float eps,
                                  int64_t virt_cap, int64_t hub_cap, int need_slots, int64_t* count_out,
                                  void* workspace, size_t workspace_bytes, tgpb200_stream_t stream);
int tgpb200_bucket_coalesce_emit(int64_t num_edges, int64_t num_nodes, int64_t num_clusters, int weighted,
                                 int64_t virt_cap, int64_t* out_row, int64_t* out_col, float* out_weight,
                                 int32_t* edge_slot, int32_t* run_len, float* run_aux, void* workspace,
                                 size_t workspace_bytes, tgpb200_stream_t stream);
size_t tgpb200_coalesce_bwd_workspace_bytes(int64_t num_edges, int64_t num_out, int op);

/* ------------------------------------------------------------------------------------------
 * Edge-weight normalisations of postprocess_adj_pool_sparse  tgp/utils/ops.py:383-417.
 * degree_norm:  deg = scatter_sum(w, row, K); dinv = clamp(deg, eps)^-1/2; w' = w * dinv[row] * dinv[col]
 *               (w == NULL means ones, ops.py:384-385).  deg_out [K] fp32 is kept for backward.
 * weight_norm:  mx[g] = max |w| over edges with batch_pooled[row] == g (0 -> 1); w'' = w / mx[g];
 *               arg_out[g] (int32) = first edge attaining the max, -1 if none (torch_scatter CPU rule).
 * All sums are DETERMINISTIC (no floating-point atomics): per-key segmented sums with a fixed combination shape.
 * rows_sorted != 0 asserts that `row` is non-decreasing (true for every cluster-path output and for the kept-node
 * output of a row-sorted input; tgpb200_rows_sorted checks it) and takes the sort-free path; otherwise the edges are
 * first grouped by key with the stable radix sort.  num_edges_dev (may be NULL) is a device-side edge count
 * <= num_edges (the launch capacity), for pipelines that never read the filtered edge count back to the host.
 * `workspace`: tgpb200_edge_norm_workspace_bytes(num_edges, num_clusters).
 * ------------------------------------------------------------------------------------------ */
size_t tgpb200_edge_norm_workspace_bytes(int64_t num_edges, int64_t num_clusters);
/* *sorted_out (device int32) = 1 if row[0..E) is non-decreasing else 0. */
int tgpb200_rows_sorted(const int64_t* row, int64_t num_edges, int32_t* sorted_out, tgpb200_stream_t stream);
int tgpb200_degree_norm_fwd(const int64_t* row, const int64_t* col, const float* w, int64_t num_edges,
                            const int64_t* num_edges_dev, int64_t num_clusters, float eps, int rows_sorted,
                            float* deg_out, float* w_out, void* workspace, size_t workspace_bytes,
                            tgpb200_stream_t stream);
int tgpb200_degree_norm_bwd(const int64_t* row, const int64_t* col, const float* w, const float* deg,
                            const float* grad_out, int64_t num_edges, const int64_t* num_edges_dev,
                            int64_t num_clusters, float eps, int rows_sorted,
                            float* grad_dinv /* [K] scratch, overwritten */, float* grad_w, void* workspace,
                            size_t workspace_bytes, tgpb200_stream_t stream);
/* Split forms for the edge-sharded multi-GPU path (SURVEY 8e): accumulate the [K] degree / [K] grad-dinv / [G] max
 * partials on the local edge shard, combine them across ranks (all-reduce sum / max), then apply. */
int tgpb200_degree_accumulate(const int64_t* row, const float* w, int64_t num_edges, const int64_t* num_edges_dev,
                              int64_t num_clusters, int rows_sorted, float* deg, void* workspace,
                              size_t workspace_bytes, tgpb200_stream_t stream);
int tgpb200_degree_apply(const int64_t* row, const int64_t* col, const float* w, const float* deg, int64_t num_edges,
                         const int64_t* num_edges_dev, int64_t num_clusters, float eps, float* w_out,
                         tgpb200_stream_t stream);
int tgpb200_degree_bwd_accumulate(const int64_t* row, const int64_t* col, const float* w, const float* deg,
                                  const float* grad_out, int64_t num_edges, const int64_t* num_edges_dev,
                                  int64_t num_clusters, float eps, int rows_sorted, float* grad_dinv, void* workspace,
                                  size_t workspace_bytes, tgpb200_stream_t stream);
int tgpb200_degree_bwd_apply(const int64_t* row, const int64_t* col, const float* deg, const float* grad_out,
                             const float* grad_dinv, int64_t num_edges, const int64_t* num_edges_dev,
                             int64_t num_clusters, float eps, float* grad_w, tgpb200_stream_t stream);
int tgpb200_weight_max_accumulate(const int64_t* row, const float* w, const int64_t* batch_pooled, int64_t num_edges,
                                  const int64_t* num_edges_dev, int64_t num_graphs, float* max_out,
                                  tgpb200_stream_t stream);
int tgpb200_weight_max_apply(const int64_t* row, const float* w, const int64_t* batch_pooled, const float* max_in,
                             int64_t num_edges, const int64_t* num_edges_dev, int64_t num_graphs, float* w_out,
                             tgpb200_stream_t stream);
int tgpb200_weight_norm_fwd(const int64_t* row, const float* w, const int64_t* batch_pooled, int64_t num_edges,
                            const int64_t* num_edges_dev, int64_t num_graphs, float* max_out, int32_t* arg_out,
                            float* w_out, tgpb200_stream_t stream);
int tgpb200_weight_norm_bwd(const int64_t* row, const float* w, const int64_t* batch_pooled, const float* max_in,
                            const int32_t* arg_in, const float* grad_out, int64_t num_edges,
                            const int64_t* num_edges_dev, int64_t num_clusters, int64_t num_graphs, int rows_sorted,
                            float* graph_acc /* [num_graphs] scratch */, float* grad_w, void* workspace,
                            size_t workspace_bytes, tgpb200_stream_t stream);

/* ------------------------------------------------------------------------------------------
 * Dense Reduce + Connect + auxiliary losses, one fused call per direction.
 *   x_pool   = S^T X                 BaseReduce.forward dense path  tgp/reduce/base_reduce.py:158-161
 *   raw      = (S^T A) S             DenseConnect._dense_connect    tgp/connect/dense_conn.py:112-122
 *   adj_pool = postprocess(raw)      postprocess_adj_pool_dense     tgp/utils/ops.py:282-335
 *   loss_kind 1: losses[0] = mincut_loss (mean over B), losses[1] = orthogonality_loss (mean over B)
 *                tgp/utils/losses.py:39-123, computed from the RAW product (tgp/poolers/mincut.py:226-237)
 *   loss_kind 2: losses[2] = link_pred_loss (one Frobenius norm over the batch, / link_div),
 *                losses[3] = entropy_loss (/ ent_div)   tgp/utils/losses.py:644-708, 476-500
 *   loss_kind 3: DMoN (PyG DMoNPooling's losses), with d = adj 1, 2m = sum_i d_i, t = tr(S^T adj S) raw,
 *                c = S^T d, e = S^T 1 per graph:  losses[0] = spectral = mean_b -(t - ||c||^2 / 2m) / 2m,
 *                losses[1] = orthogonality_loss (as kind 1), losses[2] = cluster = mean_b ||e|| sqrt(K) / n_b - 1,
 *                losses[3] = 0.  A graph with 2m = 0 gives a NaN spectral loss.  Needs adj.
 * adj [B,N,N], s [B,N,K], x [B,N,F] row-major of `dtype`; x may be NULL (connect only), adj may be NULL
 * (reduce only).  `saved` (tgpb200_dense_pool_saved_bytes) carries S^T A, S^T S, row statistics and the
 * per-graph loss terms from forward to backward; the backward also needs a scratch workspace.
 * grad_losses: 4 device floats (upstream gradients of losses[0..3]) or NULL.  grad_adj may be NULL.
 * The _v2 entry points take `graph_nodes`: [B] device floats, the valid node count n_b of each graph (the cluster
 * loss of kind 3 divides by it), or NULL for n_b = N.  It is read on the device only (no host synchronisation).
 * The entry points without _v2 are the _v2 ones with graph_nodes = NULL.
 * ------------------------------------------------------------------------------------------ */
size_t tgpb200_dense_pool_saved_bytes(int64_t B, int64_t N, int64_t K);
size_t tgpb200_dense_pool_bwd_workspace_bytes(int64_t B, int64_t N, int64_t K, int need_grad_adj);
int tgpb200_dense_pool_fwd(const void* adj, const void* s, const void* x, int64_t B, int64_t N, int64_t K, int64_t F,
                           int dtype, uint32_t flags, int loss_kind, float eps, float link_div, float ent_div,
                           void* x_pool, void* adj_pool, float* losses, void* saved, size_t saved_bytes,
                           tgpb200_stream_t stream);
int tgpb200_dense_pool_bwd(const void* adj, const void* s, const void* x, const void* grad_x_pool,
                           const void* grad_adj_pool, const float* grad_losses, int64_t B, int64_t N, int64_t K,
                           int64_t F, int dtype, uint32_t flags, int loss_kind, float eps, float link_div,
                           float ent_div, void* grad_s, void* grad_x, void* grad_adj, void* saved, size_t saved_bytes,
                           void* workspace, size_t workspace_bytes, tgpb200_stream_t stream);
int tgpb200_dense_pool_fwd_v2(const void* adj, const void* s, const void* x, int64_t B, int64_t N, int64_t K,
                              int64_t F, int dtype, uint32_t flags, int loss_kind, float eps, float link_div,
                              float ent_div, void* x_pool, void* adj_pool, float* losses, void* saved,
                              size_t saved_bytes, tgpb200_stream_t stream, const float* graph_nodes);
int tgpb200_dense_pool_bwd_v2(const void* adj, const void* s, const void* x, const void* grad_x_pool,
                              const void* grad_adj_pool, const float* grad_losses, int64_t B, int64_t N, int64_t K,
                              int64_t F, int dtype, uint32_t flags, int loss_kind, float eps, float link_div,
                              float ent_div, void* grad_s, void* grad_x, void* grad_adj, void* saved,
                              size_t saved_bytes, void* workspace, size_t workspace_bytes, tgpb200_stream_t stream,
                              const float* graph_nodes);

/* ------------------------------------------------------------------------------------------
 * Tensor-core batched product (tcgen05 / TMEM / TMA), the engine under the dense path; exported for tests
 * and for callers that need a raw S^T X / S^T A S style contraction:
 *   out[b] (M x N) = alpha * A[b] (M x Kd) * B[b] (Kd x N)  (+ out[b] when accumulate)
 * Operand layouts per batch item (cols contiguous):  K-major  = [MN extent rows][Kd cols],
 *                                                     MN-major = [Kd rows][MN extent cols].
 * fp32 operands run as error-compensated 3xTF32 (fp32-level accuracy), bf16 as a single pass; fp32 accumulate.
 * Returns TGPB200_ERR_UNSUPPORTED when a TMA constraint fails (16-byte aligned strides; an MN-major extent
 * must be a multiple of 32 fp32 / 64 bf16 elements).
 * ------------------------------------------------------------------------------------------ */
int tgpb200_tc_gemm(const void* a, const void* b, void* out, int64_t batch, int64_t M, int64_t N, int64_t Kd,
                    int64_t a_batch_stride, int64_t a_row_stride, int a_mn_major, int64_t b_batch_stride,
                    int64_t b_row_stride, int b_mn_major, int64_t out_batch_stride, int64_t out_row_stride,
                    int64_t out_col_stride, int in_dtype, int out_dtype, float alpha, int accumulate,
                    tgpb200_stream_t stream);

/* Batched product with shape-general fallback (the engine above when the layout satisfies its TMA constraints,
 * FP32-pipe tiles otherwise): out[b] (M x N, row-major, contiguous) = A[b] B[b].  Used by the dense lift
 * (tgp/lift/base_lift.py:125-160: S x_pool) for cluster / feature counts off the 16-byte stride grid. */
int tgpb200_bmm(const void* a, const void* b, void* out, int64_t batch, int64_t M, int64_t N, int64_t Kd,
                int64_t a_batch_stride, int64_t a_row_stride, int a_mn_major, int64_t b_batch_stride,
                int64_t b_row_stride, int b_mn_major, int dtype, tgpb200_stream_t stream);

/* ------------------------------------------------------------------------------------------
 * TopK selection (producer of the kept-node SelectOutput; SURVEY 8f row 1):
 * TopkSelect.forward  tgp/select/topk_select.py:194-203 (PyG topk, ratio mode) + the ascending node sort of
 * cluster_to_s  tgp/select/base_select.py:56-60.  Per graph the top ceil(ratio * n_g) scores (int(ratio) when
 * ratio >= 1), descending, ties -> lower node id.  Outputs (capacity N): node_index ascending and
 * cluster_index[j] = rank of node_index[j] in (graph asc, score desc) order; *count_out = K.
 * batch may be NULL (one graph).  score is fp32.
 * ------------------------------------------------------------------------------------------ */
size_t tgpb200_topk_select_workspace_bytes(int64_t num_nodes, int64_t num_graphs);
int tgpb200_topk_select(const float* score, const int64_t* batch, int64_t num_nodes, int64_t num_graphs, float ratio,
                        int64_t* node_index, int64_t* cluster_index, int64_t* count_out, void* workspace,
                        size_t workspace_bytes, tgpb200_stream_t stream);

/* ------------------------------------------------------------------------------------------
 * Dense -> block-diagonal sparse output (SURVEY 8a row a16):
 * dense_to_block_diag  tgp/utils/ops.py:53-82  fused with the masking / compact renumbering of
 * DenseSRCPooling._finalize_sparse_output  tgp/src.py:526-552.
 * Keeps adj[b, r, c] with |a| > eps and (out_mask == NULL or out_mask[b, r] && out_mask[b, c]) in row-major
 * (b, r, c) order; endpoints are b*K + r, or the compact id (exclusive scan of out_mask) when a mask is given.
 * out_mask is a uint8 [B, K] array.  Two phases sharing one workspace; src_pos (int32, optional) records the
 * flat position of every emitted entry for the backward (grad_adj = scatter of grad_weight, zero elsewhere).
 * ------------------------------------------------------------------------------------------ */
size_t tgpb200_block_diag_workspace_bytes(int64_t B, int64_t K);
int tgpb200_block_diag_count(const void* adj, const uint8_t* out_mask, int64_t B, int64_t K, int dtype, float eps,
                             int64_t* num_valid_out, int64_t* count_out, void* workspace, size_t workspace_bytes,
                             tgpb200_stream_t stream);
int tgpb200_block_diag_emit(const void* adj, const uint8_t* out_mask, int64_t B, int64_t K, int dtype, float eps,
                            int64_t* out_row, int64_t* out_col, void* out_weight, int32_t* src_pos, void* workspace,
                            size_t workspace_bytes, tgpb200_stream_t stream);
int tgpb200_block_diag_bwd(const void* grad_weight, const int32_t* src_pos, int64_t num_edges, int64_t total, int dtype,
                           void* grad_adj, tgpb200_stream_t stream);

/* ------------------------------------------------------------------------------------------
 * Dense pre-processing (SURVEY 8f row 3): DenseSRCPooling.preprocessing  tgp/src.py:434-450
 *   graph_ptr:      ptr[b] = first node of graph b (batch sorted ascending), ptr[B] = N     (PyG cumsum of bincount)
 *   to_dense_batch: x [N, F] -> [B, Nmax, F] zero padded, mask [B, Nmax] (uint8)            (PyG to_dense_batch)
 *   to_dense_adj:   edges -> [B, Nmax, Nmax] fp32, duplicates summed, default weight 1.0,
 *                   transpose != 0 writes A^T (src.py:442-443)                               (PyG to_dense_adj)
 * ------------------------------------------------------------------------------------------ */
int tgpb200_graph_ptr(const int64_t* batch, int64_t num_nodes, int64_t num_graphs, int32_t* ptr, void* workspace,
                      size_t workspace_bytes, tgpb200_stream_t stream);
int tgpb200_to_dense_batch(const void* x, const int64_t* batch, const int32_t* ptr, int64_t num_nodes, int64_t F,
                           int64_t num_graphs, int64_t max_nodes, int dtype, void* out, uint8_t* mask,
                           tgpb200_stream_t stream);
int tgpb200_to_dense_adj(const int64_t* row, const int64_t* col, const float* w, const int64_t* batch,
                         const int32_t* ptr, int64_t num_edges, int64_t num_graphs, int64_t max_nodes, int transpose,
                         float* adj, tgpb200_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* TGP_B200_H_ */
