// torch custom-op shim over the C ABI of libtgp_b200.so (include/tgp_b200.h): the hot ops of the Reduce + Connect
// path as dispatcher-visible `torch.ops.tgp_b200.*` operators (SURVEY 8b).  This file only allocates outputs with
// the caching allocator, picks the current CUDA stream and forwards plain pointers and sizes; every kernel lives in
// libtgp_b200.so.  Autograd (torch.library.register_autograd) and the fake / meta kernels are registered from
// Python (tgp_b200/ops.py), next to the remaining operators of the path.
//
// Built by csrc/build.sh into tgp_b200/libtgp_b200_ops.so (g++, no nvcc: there is no device code here).
#include <ATen/ATen.h>
#include <c10/cuda/CUDAGuard.h>
#include <c10/cuda/CUDAStream.h>
#include <torch/library.h>

#include "../../include/tgp_b200.h"

namespace {

using at::Tensor;
using OptTensor = std::optional<Tensor>;

const void* ptr(const OptTensor& t) { return (t.has_value() && t->defined() && t->numel() > 0) ? t->data_ptr() : nullptr; }
const void* ptr(const Tensor& t) { return (t.defined() && t.numel() > 0) ? t.data_ptr() : nullptr; }

int dtype_code(const Tensor& t) {
  if (t.scalar_type() == at::kFloat) return TGPB200_F32;
  if (t.scalar_type() == at::kBFloat16) return TGPB200_BF16;
  TORCH_CHECK(false, "tgp_b200: unsupported dtype ", t.scalar_type(), " (float32 and bfloat16 only)");
}

void check(int rc, const char* what) {
  static const char* names[] = {"ok", "invalid argument", "workspace too small", "CUDA launch failed",
                                "unsupported shape/dtype"};
  TORCH_CHECK(rc == TGPB200_OK, "tgp_b200.", what, " failed: ", (rc <= 0 && rc >= -4) ? names[-rc] : "unknown error");
}

void require_cuda(const Tensor& t, const char* name) {
  TORCH_CHECK(t.is_cuda(), "tgp_b200 runs on CUDA tensors only (no CPU fallback by design): ", name);
  TORCH_CHECK(t.is_contiguous(), "tgp_b200: tensor must be contiguous: ", name);
}

tgpb200_stream_t stream_of(const Tensor& t) {
  return reinterpret_cast<tgpb200_stream_t>(c10::cuda::getCurrentCUDAStream(t.device().index()).stream());
}

Tensor workspace(size_t bytes, const Tensor& like) {
  return at::empty({(int64_t)(bytes < 256 ? 256 : bytes)}, like.options().dtype(at::kByte));
}

// (x_pool, adj_pool, losses[4], saved) = fused S^T X, postprocess(S^T A S), auxiliary losses
// tgp/reduce/base_reduce.py:158-161, tgp/connect/dense_conn.py:112-138,257-271, tgp/utils/ops.py:282-335,
// tgp/utils/losses.py:39-123,476-500,644-708
// graph_nodes (optional): [B] float32 valid-node counts n_b on the device (DMoN's cluster loss); absent means N.
const float* graph_nodes_ptr(const OptTensor& graph_nodes, int64_t B) {
  if (!graph_nodes.has_value() || !graph_nodes->defined()) return nullptr;
  require_cuda(*graph_nodes, "graph_nodes");
  TORCH_CHECK(graph_nodes->scalar_type() == at::kFloat, "tgp_b200: graph_nodes must be float32");
  TORCH_CHECK(graph_nodes->dim() == 1 && graph_nodes->size(0) == B, "tgp_b200: graph_nodes must have shape [B] = [", B,
              "], got ", graph_nodes->sizes());
  return B > 0 ? graph_nodes->data_ptr<float>() : nullptr;
}

std::tuple<Tensor, Tensor, Tensor, Tensor> stas_fused(const OptTensor& x, const OptTensor& adj, const Tensor& s,
                                                      int64_t flags, int64_t loss_kind, double link_div,
                                                      double ent_div, const OptTensor& graph_nodes) {
  require_cuda(s, "s");
  TORCH_CHECK(s.dim() == 3, "stas_fused expects s of shape [B, N, K]");
  c10::cuda::CUDAGuard guard(s.device());
  const int64_t B = s.size(0), N = s.size(1), K = s.size(2);
  const float* gn = graph_nodes_ptr(graph_nodes, B);
  const bool has_x = x.has_value() && x->defined(), has_a = adj.has_value() && adj->defined();
  if (has_x) require_cuda(*x, "x");
  if (has_a) require_cuda(*adj, "adj");
  const int64_t F = has_x ? x->size(-1) : 0;
  Tensor saved = workspace(tgpb200_dense_pool_saved_bytes(B, N, K), s);
  Tensor x_pool = at::empty({has_x ? B : 0, K, F}, s.options());
  Tensor adj_pool = at::empty({has_a ? B : 0, K, K}, s.options());
  Tensor losses = at::zeros({4}, s.options().dtype(at::kFloat));
  check(tgpb200_dense_pool_fwd_v2(ptr(adj), s.data_ptr(), ptr(x), B, N, K, F, dtype_code(s), (uint32_t)flags,
                                  (int)loss_kind, 1e-8f, (float)link_div, (float)ent_div,
                                  has_x ? x_pool.data_ptr() : nullptr, has_a ? adj_pool.data_ptr() : nullptr,
                                  losses.data_ptr<float>(), saved.data_ptr(), (size_t)saved.numel(), stream_of(s), gn),
        "stas_fused");
  return {x_pool, adj_pool, losses, saved};
}

std::tuple<Tensor, Tensor, Tensor> stas_fused_bwd(const OptTensor& x, const OptTensor& adj, const Tensor& s,
                                                  const Tensor& saved, const OptTensor& gx_pool,
                                                  const OptTensor& gadj_pool, const OptTensor& glosses, int64_t flags,
                                                  int64_t loss_kind, double link_div, double ent_div, bool need_gadj,
                                                  const OptTensor& graph_nodes) {
  c10::cuda::CUDAGuard guard(s.device());
  const int64_t B = s.size(0), N = s.size(1), K = s.size(2);
  const float* gn = graph_nodes_ptr(graph_nodes, B);
  const bool has_x = x.has_value() && x->defined(), has_a = adj.has_value() && adj->defined();
  const int64_t F = has_x ? x->size(-1) : 0;
  const bool want_gx = has_x && gx_pool.has_value() && gx_pool->defined();
  const bool want_ga = has_a && need_gadj;
  Tensor ws = workspace(tgpb200_dense_pool_bwd_workspace_bytes(B, N, K, want_ga), s);
  Tensor gs = at::empty_like(s);
  Tensor gx = want_gx ? at::empty_like(*x) : (has_x ? at::zeros_like(*x) : at::empty({0}, s.options()));
  Tensor ga = want_ga ? at::empty_like(*adj) : at::empty({0}, s.options());
  Tensor gxp = want_gx ? gx_pool->contiguous() : Tensor();
  Tensor gap = (has_a && gadj_pool.has_value() && gadj_pool->defined()) ? gadj_pool->contiguous() : Tensor();
  Tensor gl = (glosses.has_value() && glosses->defined()) ? glosses->to(at::kFloat).contiguous() : Tensor();
  check(tgpb200_dense_pool_bwd_v2(ptr(adj), s.data_ptr(), ptr(x), ptr(gxp), ptr(gap),
                                  gl.defined() ? gl.data_ptr<float>() : nullptr, B, N, K, F, dtype_code(s),
                                  (uint32_t)flags, (int)loss_kind, 1e-8f, (float)link_div, (float)ent_div, gs.data_ptr(),
                                  want_gx ? gx.data_ptr() : nullptr, want_ga ? ga.data_ptr() : nullptr,
                                  saved.data_ptr(), (size_t)saved.numel(), ws.data_ptr(), (size_t)ws.numel(),
                                  stream_of(s), gn),
        "stas_fused_bwd");
  return {gx, ga, gs};
}

// The [B, N, N] adjacency and the [B, N, K] assignment of the dense loss ops: CUDA, contiguous, one dtype, K >= 2
// and N >= 1.  `op` names the operator in the messages; `k_reason` says why it needs two clusters (may be empty).
void check_adj_s(const Tensor& adj, const Tensor& s, const char* op, const char* k_reason = "") {
  require_cuda(s, "s");
  require_cuda(adj, "adj");
  TORCH_CHECK(s.dim() == 3, op, " expects s of shape [B, N, K], got ", s.sizes());
  TORCH_CHECK(adj.dim() == 3 && adj.size(0) == s.size(0) && adj.size(1) == s.size(1) && adj.size(2) == s.size(1),
              op, " expects adj of shape [B, N, N] = [", s.size(0), ", ", s.size(1), ", ", s.size(1), "], got ",
              adj.sizes());
  TORCH_CHECK(adj.scalar_type() == s.scalar_type(), "tgp_b200.", op, ": adj and s must share one dtype");
  TORCH_CHECK_VALUE(s.size(2) >= 2, op, " needs K >= 2 clusters", k_reason, ", got K = ", s.size(2));
  TORCH_CHECK_VALUE(s.size(1) >= 1, op, " needs N >= 1 nodes");
}

constexpr const char* kAccKReason = " (the balance loss divides by K - 1)";

// (losses[2] = {total variation, balance}, quant [B, K], saved) of Asymmetric Cheeger Cut pooling
// (totvar_loss / asym_norm_loss as restated in tests/acc_oracle.py)
std::tuple<Tensor, Tensor, Tensor> acc_losses(const Tensor& adj, const Tensor& s) {
  check_adj_s(adj, s, "acc_losses", kAccKReason);
  c10::cuda::CUDAGuard guard(s.device());
  const int64_t B = s.size(0), N = s.size(1), K = s.size(2);
  Tensor saved = workspace(tgpb200_acc_loss_saved_bytes(B, K), s);
  Tensor ws = workspace(tgpb200_acc_loss_fwd_workspace_bytes(B, N, K), s);
  Tensor losses = at::empty({2}, s.options().dtype(at::kFloat));
  Tensor quant = at::empty({B, K}, s.options());
  check(tgpb200_acc_loss_fwd(adj.data_ptr(), s.data_ptr(), B, N, K, dtype_code(s), losses.data_ptr<float>(),
                             quant.data_ptr(), saved.data_ptr(), (size_t)saved.numel(), ws.data_ptr(),
                             (size_t)ws.numel(), stream_of(s)),
        "acc_losses");
  return {losses, quant, saved};
}

std::tuple<Tensor, Tensor> acc_losses_bwd(const Tensor& adj, const Tensor& s, const Tensor& saved,
                                          const Tensor& glosses, bool need_gadj) {
  check_adj_s(adj, s, "acc_losses", kAccKReason);
  c10::cuda::CUDAGuard guard(s.device());
  const int64_t B = s.size(0), N = s.size(1), K = s.size(2);
  TORCH_CHECK(glosses.numel() == 2, "acc_losses_bwd expects 2 upstream loss gradients");
  Tensor gl = glosses.to(at::kFloat).contiguous();
  Tensor gs = at::empty_like(s);
  Tensor ga = need_gadj ? at::empty_like(adj) : at::empty({0}, s.options());
  check(tgpb200_acc_loss_bwd(adj.data_ptr(), s.data_ptr(), saved.data_ptr(), (size_t)saved.numel(),
                             gl.data_ptr<float>(), B, N, K, dtype_code(s), gs.data_ptr(),
                             need_gadj ? ga.data_ptr() : nullptr, stream_of(s)),
        "acc_losses_bwd");
  return {ga, gs};
}

// (losses[3] = {first-order cut, motif cut, HOSC orthogonality}, saved) of HOSC pooling (restated in
// tests/hosc_oracle.py); `terms` is the bitmask of tgpb200_hosc_loss_fwd
std::tuple<Tensor, Tensor> hosc_losses(const Tensor& adj, const Tensor& s, const OptTensor& graph_nodes,
                                       int64_t terms, double eps) {
  check_adj_s(adj, s, "hosc_losses");
  TORCH_CHECK_VALUE(terms >= 1 && terms <= 7, "hosc_losses: terms must be a non-empty mask of 1 | 2 | 4, got ", terms);
  c10::cuda::CUDAGuard guard(s.device());
  const int64_t B = s.size(0), N = s.size(1), K = s.size(2);
  const int dt = dtype_code(s);
  Tensor saved = workspace(tgpb200_hosc_loss_saved_bytes(B, N, K, (int)terms, dt), s);
  Tensor ws = workspace(tgpb200_hosc_loss_fwd_workspace_bytes(B, N, K, (int)terms, dt), s);
  Tensor losses = at::empty({3}, s.options().dtype(at::kFloat));
  check(tgpb200_hosc_loss_fwd(adj.data_ptr(), s.data_ptr(), graph_nodes_ptr(graph_nodes, B), B, N, K, dt, (int)terms,
                              (float)eps, losses.data_ptr<float>(), saved.data_ptr(), (size_t)saved.numel(),
                              ws.data_ptr(), (size_t)ws.numel(), stream_of(s)),
        "hosc_losses");
  return {losses, saved};
}

std::tuple<Tensor, Tensor> hosc_losses_bwd(const Tensor& adj, const Tensor& s, const OptTensor& graph_nodes,
                                           const Tensor& saved, const Tensor& glosses, int64_t terms, bool need_gadj) {
  check_adj_s(adj, s, "hosc_losses");
  TORCH_CHECK_VALUE(terms >= 1 && terms <= 7, "hosc_losses: terms must be a non-empty mask of 1 | 2 | 4, got ", terms);
  c10::cuda::CUDAGuard guard(s.device());
  const int64_t B = s.size(0), N = s.size(1), K = s.size(2);
  const int dt = dtype_code(s);
  TORCH_CHECK(glosses.numel() == 3, "hosc_losses_bwd expects 3 upstream loss gradients");
  Tensor gl = glosses.to(at::kFloat).contiguous();
  Tensor gs = at::empty_like(s);
  Tensor ga = need_gadj ? at::empty_like(adj) : at::empty({0}, s.options());
  Tensor ws = workspace(tgpb200_hosc_loss_bwd_workspace_bytes(B, N, K, dt, need_gadj ? 1 : 0), s);
  check(tgpb200_hosc_loss_bwd(adj.data_ptr(), s.data_ptr(), graph_nodes_ptr(graph_nodes, B), saved.data_ptr(),
                              (size_t)saved.numel(), gl.data_ptr<float>(), B, N, K, dt, (int)terms, gs.data_ptr(),
                              need_gadj ? ga.data_ptr() : nullptr, ws.data_ptr(), (size_t)ws.numel(), stream_of(s)),
        "hosc_losses_bwd");
  return {ga, gs};
}

// The coalesced edge list (row, col, weight), its row CSR and column CSR, and s [B, N, K] of the sparse HOSC ops
void check_sparse_hosc(const Tensor& row, const Tensor& col, const Tensor& weight, const Tensor& row_ptr,
                       const Tensor& col_ptr, const Tensor& col_order, const Tensor& s, int64_t terms) {
  require_cuda(s, "s");
  for (const Tensor* t : {&row, &col, &weight, &row_ptr, &col_ptr, &col_order}) require_cuda(*t, "edge list / CSR");
  TORCH_CHECK(s.dim() == 3, "hosc_losses_sparse expects s of shape [B, N, K], got ", s.sizes());
  TORCH_CHECK_VALUE(s.size(2) >= 2, "hosc_losses_sparse needs K >= 2 clusters, got K = ", s.size(2));
  TORCH_CHECK_VALUE(s.size(1) >= 1, "hosc_losses_sparse needs N >= 1 nodes");
  TORCH_CHECK_VALUE(terms >= 1 && terms <= 7, "hosc_losses_sparse: terms must be a non-empty mask of 1 | 2 | 4, got ",
                    terms);
  const int64_t nnz = row.numel(), R = s.size(0) * s.size(1);
  TORCH_CHECK(row.scalar_type() == at::kLong && col.scalar_type() == at::kLong && col.numel() == nnz,
              "hosc_losses_sparse: row / col must be int64 [nnz]");
  TORCH_CHECK(weight.scalar_type() == at::kFloat && weight.numel() == nnz, "hosc_losses_sparse: weight must be float32 [nnz]");
  TORCH_CHECK(row_ptr.scalar_type() == at::kInt && col_ptr.scalar_type() == at::kInt && col_order.scalar_type() == at::kInt &&
                  row_ptr.numel() == R + 1 && col_ptr.numel() == R + 1 && col_order.numel() >= nnz,
              "hosc_losses_sparse: row_ptr / col_ptr must be int32 [B N + 1] and col_order int32 [nnz]");
}

// (losses[3] = {first-order cut, motif cut, HOSC orthogonality}, as1 = [A S | A 1 | 0..] [B, N, K1], saved) of HOSC
// pooling on a sparse adjacency; `terms` is the bitmask of tgpb200_hosc_sparse_loss_fwd
std::tuple<Tensor, Tensor, Tensor> hosc_losses_sparse(const Tensor& row, const Tensor& col, const Tensor& weight,
                                                      const Tensor& row_ptr, const Tensor& col_ptr,
                                                      const Tensor& col_order, const Tensor& s,
                                                      const OptTensor& graph_nodes, int64_t terms, double eps) {
  check_sparse_hosc(row, col, weight, row_ptr, col_ptr, col_order, s, terms);
  c10::cuda::CUDAGuard guard(s.device());
  const int64_t B = s.size(0), N = s.size(1), K = s.size(2), nnz = row.numel(), K1 = (K + 8) / 8 * 8;
  const int dt = dtype_code(s);
  Tensor saved = workspace(tgpb200_hosc_sparse_loss_saved_bytes(B, N, K, nnz, (int)terms), s);
  Tensor ws = workspace(tgpb200_hosc_sparse_loss_fwd_workspace_bytes(B, N, K, nnz, (int)terms, dt), s);
  Tensor losses = at::empty({3}, s.options().dtype(at::kFloat));
  Tensor as1 = at::empty({B, N, K1}, s.options().dtype(at::kFloat));
  check(tgpb200_hosc_sparse_loss_fwd((const int64_t*)ptr(row), (const int64_t*)ptr(col), (const float*)ptr(weight),
                                     row_ptr.data_ptr<int32_t>(), col_ptr.data_ptr<int32_t>(),
                                     (const int32_t*)ptr(col_order), s.data_ptr(), graph_nodes_ptr(graph_nodes, B), B,
                                     N, K, nnz, dt, (int)terms, (float)eps, losses.data_ptr<float>(),
                                     as1.data_ptr<float>(), saved.data_ptr(), (size_t)saved.numel(), ws.data_ptr(),
                                     (size_t)ws.numel(), stream_of(s)),
        "hosc_losses_sparse");
  return {losses, as1, saved};
}

std::tuple<Tensor, Tensor> hosc_losses_sparse_bwd(const Tensor& row, const Tensor& col, const Tensor& weight,
                                                  const Tensor& row_ptr, const Tensor& col_ptr, const Tensor& col_order,
                                                  const Tensor& s, const OptTensor& graph_nodes, const Tensor& saved,
                                                  const Tensor& glosses, const OptTensor& gas1, int64_t terms,
                                                  bool need_gweight) {
  check_sparse_hosc(row, col, weight, row_ptr, col_ptr, col_order, s, terms);
  c10::cuda::CUDAGuard guard(s.device());
  const int64_t B = s.size(0), N = s.size(1), K = s.size(2), nnz = row.numel();
  const int dt = dtype_code(s);
  TORCH_CHECK(glosses.numel() == 3, "hosc_losses_sparse_bwd expects 3 upstream loss gradients");
  Tensor gl = glosses.to(at::kFloat).contiguous();
  const bool has_gas = gas1.has_value() && gas1->defined();
  Tensor ga = has_gas ? gas1->to(at::kFloat).contiguous() : Tensor();
  Tensor gs = at::empty_like(s);
  Tensor gw = at::empty({need_gweight ? nnz : 0}, s.options().dtype(at::kFloat));
  Tensor ws = workspace(tgpb200_hosc_sparse_loss_bwd_workspace_bytes(B, N, K, nnz, (int)terms, dt, has_gas ? 1 : 0,
                                                                     need_gweight ? 1 : 0), s);
  check(tgpb200_hosc_sparse_loss_bwd((const int64_t*)ptr(row), (const int64_t*)ptr(col), (const float*)ptr(weight),
                                     row_ptr.data_ptr<int32_t>(), col_ptr.data_ptr<int32_t>(),
                                     (const int32_t*)ptr(col_order), s.data_ptr(), graph_nodes_ptr(graph_nodes, B),
                                     saved.data_ptr(), (size_t)saved.numel(), gl.data_ptr<float>(),
                                     has_gas ? ga.data_ptr<float>() : nullptr, B, N, K, nnz, dt, (int)terms,
                                     gs.data_ptr(), need_gweight ? (float*)ptr(gw) : nullptr, ws.data_ptr(),
                                     (size_t)ws.numel(), stream_of(s)),
        "hosc_losses_sparse_bwd");
  return {gw, gs};
}

// CSR-by-cluster of a sparse assignment (tgp/reduce/aggr_reduce.py:13-23)
std::tuple<Tensor, Tensor> build_csr(const Tensor& cluster_index, int64_t num_clusters) {
  require_cuda(cluster_index, "cluster_index");
  c10::cuda::CUDAGuard guard(cluster_index.device());
  const int64_t nnz = cluster_index.numel();
  Tensor order = at::empty({nnz > 0 ? nnz : 1}, cluster_index.options().dtype(at::kInt));
  Tensor p = at::empty({num_clusters + 1}, cluster_index.options().dtype(at::kInt));
  Tensor ws = workspace(tgpb200_build_csr_workspace_bytes(nnz, num_clusters), cluster_index);
  check(tgpb200_build_csr(cluster_index.data_ptr<int64_t>(), nnz, num_clusters, order.data_ptr<int32_t>(),
                          p.data_ptr<int32_t>(), ws.data_ptr(), (size_t)ws.numel(), stream_of(cluster_index)),
        "build_csr");
  return {order, p};
}

// x_pool[c] = op_{i in c} weight[i] * x[node_index[i]]  (tgp/reduce/base_reduce.py:141-155, aggr_reduce.py:99-105)
Tensor segment_reduce(const Tensor& x, const Tensor& node_index, const Tensor& cluster_index, const OptTensor& weight,
                      const Tensor& order, const Tensor& p, int64_t num_clusters, int64_t op) {
  require_cuda(x, "x");
  require_cuda(node_index, "node_index");
  (void)cluster_index;
  c10::cuda::CUDAGuard guard(x.device());
  const int64_t N = x.size(0), F = x.size(1), nnz = node_index.numel();
  Tensor out = at::empty({num_clusters, F}, x.options());
  const float* w = (weight.has_value() && weight->defined()) ? weight->data_ptr<float>() : nullptr;
  check(tgpb200_segment_reduce_fwd(x.data_ptr(), node_index.data_ptr<int64_t>(), w, order.data_ptr<int32_t>(),
                                   p.data_ptr<int32_t>(), N, nnz, num_clusters, F, (int)op, dtype_code(x),
                                   dtype_code(x), out.data_ptr(), stream_of(x)),
        "segment_reduce");
  return out;
}

std::tuple<Tensor, Tensor> segment_reduce_bwd(const Tensor& x, const Tensor& node_index, const Tensor& cluster_index,
                                              const OptTensor& weight, const Tensor& order, const Tensor& p,
                                              const Tensor& x_pool, const Tensor& grad, int64_t num_clusters, int64_t op,
                                              bool need_weight_grad) {
  c10::cuda::CUDAGuard guard(x.device());
  const int64_t N = x.size(0), F = x.size(1), nnz = node_index.numel();
  Tensor g = grad.contiguous();
  TORCH_CHECK(g.scalar_type() == x.scalar_type(),
              "tgp_b200 segment_reduce backward: mixed x / output dtypes are not supported");
  Tensor gx = at::empty_like(x);
  const bool has_w = weight.has_value() && weight->defined();
  Tensor gw = (has_w && need_weight_grad) ? at::empty({nnz}, x.options().dtype(at::kFloat))
                                          : at::empty({0}, x.options().dtype(at::kFloat));
  Tensor ws = workspace(tgpb200_segment_reduce_bwd_workspace_bytes(N, nnz, num_clusters, F, (int)op), x);
  check(tgpb200_segment_reduce_bwd(x.data_ptr(), node_index.data_ptr<int64_t>(), cluster_index.data_ptr<int64_t>(),
                                   has_w ? weight->data_ptr<float>() : nullptr, order.data_ptr<int32_t>(),
                                   p.data_ptr<int32_t>(), x_pool.data_ptr(), g.data_ptr(), N, nnz, num_clusters, F,
                                   (int)op, dtype_code(x), dtype_code(g), gx.data_ptr(),
                                   (has_w && need_weight_grad) ? gw.data_ptr<float>() : nullptr, ws.data_ptr(),
                                   (size_t)ws.numel(), stream_of(x)),
        "segment_reduce_bwd");
  return {gx, gw};
}

}  // namespace

TORCH_LIBRARY(tgp_b200, m) {
  m.def("stas_fused(Tensor? x, Tensor? adj, Tensor s, int flags, int loss_kind, float link_div, float ent_div, "
        "Tensor? graph_nodes=None) -> (Tensor, Tensor, Tensor, Tensor)");
  m.def("stas_fused_bwd(Tensor? x, Tensor? adj, Tensor s, Tensor saved, Tensor? gx_pool, Tensor? gadj_pool, "
        "Tensor? glosses, int flags, int loss_kind, float link_div, float ent_div, bool need_gadj, "
        "Tensor? graph_nodes=None) -> (Tensor, Tensor, Tensor)");
  m.def("acc_losses(Tensor adj, Tensor s) -> (Tensor, Tensor, Tensor)");
  m.def("acc_losses_bwd(Tensor adj, Tensor s, Tensor saved, Tensor glosses, bool need_gadj) -> (Tensor, Tensor)");
  m.def("hosc_losses(Tensor adj, Tensor s, Tensor? graph_nodes, int terms, float eps) -> (Tensor, Tensor)");
  m.def("hosc_losses_bwd(Tensor adj, Tensor s, Tensor? graph_nodes, Tensor saved, Tensor glosses, int terms, "
        "bool need_gadj) -> (Tensor, Tensor)");
  m.def("hosc_losses_sparse(Tensor row, Tensor col, Tensor weight, Tensor row_ptr, Tensor col_ptr, Tensor col_order, "
        "Tensor s, Tensor? graph_nodes, int terms, float eps) -> (Tensor, Tensor, Tensor)");
  m.def("hosc_losses_sparse_bwd(Tensor row, Tensor col, Tensor weight, Tensor row_ptr, Tensor col_ptr, "
        "Tensor col_order, Tensor s, Tensor? graph_nodes, Tensor saved, Tensor glosses, Tensor? gas1, int terms, "
        "bool need_gweight) -> (Tensor, Tensor)");
  m.def("build_csr(Tensor cluster_index, int num_clusters) -> (Tensor, Tensor)");
  m.def("segment_reduce(Tensor x, Tensor node_index, Tensor cluster_index, Tensor? weight, Tensor order, Tensor ptr, "
        "int num_clusters, int op) -> Tensor");
  m.def("segment_reduce_bwd(Tensor x, Tensor node_index, Tensor cluster_index, Tensor? weight, Tensor order, "
        "Tensor ptr, Tensor x_pool, Tensor grad, int num_clusters, int op, bool need_weight_grad) -> (Tensor, Tensor)");
}

TORCH_LIBRARY_IMPL(tgp_b200, CUDA, m) {
  m.impl("stas_fused", &stas_fused);
  m.impl("stas_fused_bwd", &stas_fused_bwd);
  m.impl("acc_losses", &acc_losses);
  m.impl("acc_losses_bwd", &acc_losses_bwd);
  m.impl("hosc_losses", &hosc_losses);
  m.impl("hosc_losses_bwd", &hosc_losses_bwd);
  m.impl("hosc_losses_sparse", &hosc_losses_sparse);
  m.impl("hosc_losses_sparse_bwd", &hosc_losses_sparse_bwd);
  m.impl("build_csr", &build_csr);
  m.impl("segment_reduce", &segment_reduce);
  m.impl("segment_reduce_bwd", &segment_reduce_bwd);
}
