"""Functional layer: the reference's functional API on top of the ``torch.ops.tgp_b200.*`` custom ops.

The differentiable operators of the path are torch custom ops (``tgp_b200/ops.py``: C++ dispatcher ops for the
dense path and the segment reduce, ``torch.library.custom_op`` for the sparse connect), each with a fake kernel and
a registered autograd formula; the helpers here (dense pre-processing, block-diagonal output) call the C ABI of
``libtgp_b200.so`` through ``_lib.call`` directly.  Everything runs on the current CUDA stream.  There is no eager /
CPU fallback: CPU tensors raise ``RuntimeError``.
"""
from __future__ import annotations

from typing import Optional, Tuple

import torch
from torch import Tensor

from . import _lib as L
from . import ops as O

EPS = 1e-8  # tgp/__init__.py:6
_T = torch.ops.tgp_b200


def _require_cuda(*tensors) -> None:
    for t in tensors:
        if t is not None and not t.is_cuda:
            raise RuntimeError("tgp_b200 runs on CUDA tensors only (no CPU fallback by design)")


# --------------------------------------------------------------------------- #
# CSR-by-cluster (cached on the SelectOutput, like the reference caches `_so_cached`)
# --------------------------------------------------------------------------- #
def build_csr(cluster_index: Tensor, num_clusters: int) -> Tuple[Tensor, Tensor]:
    _require_cuda(cluster_index)
    return _T.build_csr(cluster_index.contiguous(), num_clusters)


def csr_of(so) -> Tuple[Tensor, Tensor]:
    cached = getattr(so, "_b200_csr", None)
    if cached is None:
        cached = build_csr(so.cluster_index, so.num_supernodes)
        try:
            so._b200_csr = cached
        except AttributeError:
            pass
    return cached


# --------------------------------------------------------------------------- #
# Sparse reduce
# --------------------------------------------------------------------------- #
def segment_reduce(
    x: Tensor,
    node_index: Tensor,
    cluster_index: Tensor,
    weight: Optional[Tensor],
    num_clusters: int,
    op: str = "sum",
    csr: Optional[Tuple[Tensor, Tensor]] = None,
) -> Tensor:
    """``x_pool[c] = op_{i in c} weight[i] * x[node_index[i]]`` (deterministic member order).

    ``node_index`` must be sorted ascending (the SelectOutput invariant, tgp/select/base_select.py:56-60): the
    backward locates a node's entries by binary search.  A ``csr`` taken from a ``SelectOutput`` vouches for it;
    a bare call is checked (once per tensor) and raises ``ValueError`` otherwise."""
    _require_cuda(x, node_index, cluster_index, weight)
    if csr is None and node_index.numel() > 1 and not is_sorted(node_index):
        raise ValueError("segment_reduce: node_index must be sorted ascending (SelectOutput invariant)")
    if op not in ("sum", "add", "mean", "max", "min"):
        raise ValueError(f"unsupported reduce op '{op}'")
    if x.dim() != 2:
        raise ValueError("segment_reduce expects x of shape [N, F]")
    out_dtype = x.dtype if weight is None else torch.result_type(x, weight)
    if x.dtype != out_dtype:  # torch type promotion of x * weight (rare: bf16 features, fp32 weights)
        x = x.to(out_dtype)
    x = x.contiguous()
    w32 = None if weight is None else weight.to(torch.float32).contiguous()
    order, ptr = csr if csr is not None else build_csr(cluster_index, num_clusters)
    return _T.segment_reduce(x, node_index.contiguous(), cluster_index.contiguous(), w32, order, ptr, num_clusters,
                             L.OPS[op])


def reduce_batch_sparse(so, batch: Tensor) -> Tensor:
    """Reduce.reduce_batch, sparse branch (tgp/reduce/base_reduce.py:37-41)."""
    _require_cuda(batch)
    order, ptr = csr_of(so)
    K = so.num_supernodes
    out = torch.empty(K, dtype=torch.long, device=batch.device)
    L.call("tgpb200_reduce_batch", L.ptr(batch.contiguous()), L.ptr(so.node_index.contiguous()), L.ptr(order),
           L.ptr(ptr), K, L.ptr(out), L.stream())
    return out


# --------------------------------------------------------------------------- #
# Sparse connect
# --------------------------------------------------------------------------- #
def _read_count(count: Tensor) -> int:
    return int(count.item())  # the one device->host word per data-dependent output size


def _sorted_check(holder: Tensor, index: Tensor) -> bool:
    """Device-side "is non-decreasing" of ``index`` (one host read), remembered ON the tensor object ``holder``
    together with its version counter: a static graph pays the check on the first call only, and the memo can never
    outlive the data it describes (an address-keyed cache would, once the allocator recycles the block)."""
    memo = getattr(holder, "_b200_sorted", None)
    if memo is not None and memo[0] == holder._version:
        return memo[1]
    idx = index.contiguous()
    flag = torch.empty(1, dtype=torch.int32, device=idx.device)
    L.call("tgpb200_rows_sorted", L.ptr(idx), idx.numel(), L.ptr(flag), L.stream())
    hit = bool(flag.item())
    try:
        holder._b200_sorted = (holder._version, hit)
    except (AttributeError, RuntimeError):
        pass
    return hit


def is_sorted(index: Tensor) -> bool:
    """Is the 1-D int64 tensor non-decreasing?"""
    return _sorted_check(index, index)


def rows_sorted(edge_index: Tensor) -> bool:
    """Is ``edge_index[0]`` non-decreasing (PyG datasets and every coalesced list are)?  Row-sorted lists take the
    sort-free deterministic normalisation sums and the row-bucketed coalesce."""
    return _sorted_check(edge_index, edge_index[0])


def _as_f32_weight(edge_weight: Optional[Tensor]) -> Optional[Tensor]:
    """tgp/utils/ops.py:1043-1058: [E] or [E,1] only."""
    if edge_weight is None:
        return None
    if edge_weight.ndim > 1:
        if edge_weight.ndim == 2 and edge_weight.size(-1) == 1:
            edge_weight = edge_weight.flatten()
        else:
            raise RuntimeError(f"Edge weights must be of shape [E] or [E, 1], but got {edge_weight.shape}.")
    return edge_weight.to(torch.float32).contiguous()


def _validate_edge_index(edge_index: Tensor) -> None:
    """Dense-tensor branch of connectivity_to_edge_index (tgp/utils/ops.py:455-476)."""
    if edge_index.dim() == 3 or (edge_index.dim() == 2 and edge_index.size(0) != 2):
        raise ValueError(
            "Dense adjacency matrices are not supported by connectivity_to_edge_index(). "
            "Expected a sparse connectivity representation (edge_index with shape [2, E] or a torch COO tensor)."
        )
    if edge_index.dim() != 2:
        raise ValueError(
            "connectivity_to_edge_index() expected edge_index with shape [2, E] "
            f"when given a dense Tensor, got a Tensor with {edge_index.dim()} dimensions."
        )
    if edge_index.dtype != torch.int64:
        raise ValueError(
            "connectivity_to_edge_index() expected edge_index indices to be an integer tensor "
            f"(dtype torch.long), got dtype={edge_index.dtype}."
        )


def edge_postprocess(
    edge_index: Tensor,
    edge_weight: Optional[Tensor],
    num_nodes: int,
    degree_norm: bool = False,
    edge_weight_norm: bool = False,
    batch_pooled: Optional[Tensor] = None,
    num_graphs: Optional[int] = None,
    sorted_rows: Optional[bool] = None,
    count: Optional[Tensor] = None,
) -> Optional[Tensor]:
    """Degree / max-weight normalisation of tgp/utils/ops.py:383-417 on already-filtered edges.

    ``sorted_rows``: whether ``edge_index[0]`` is non-decreasing (``None`` = check, cached per tensor);
    ``count``: device-side number of valid edges of a padded list (``None`` = all)."""
    row, col = edge_index[0], edge_index[1]
    if not (degree_norm or (edge_weight_norm and edge_weight is not None)):
        return edge_weight
    if not row.is_contiguous():
        row, col = row.contiguous(), col.contiguous()
    if sorted_rows is None:
        sorted_rows = rows_sorted(edge_index)
    if degree_norm:
        edge_weight, _ = O.degree_norm(edge_weight, row, col, num_nodes, EPS, sorted_rows, count)
    if edge_weight_norm and edge_weight is not None:
        if num_graphs is None:  # costs a device sync: pass num_graphs to avoid it
            num_graphs = int(batch_pooled.max().item()) + 1 if batch_pooled.numel() > 0 else 0
        edge_weight, _, _ = O.weight_norm(edge_weight, row, batch_pooled.contiguous(), num_nodes, num_graphs,
                                          sorted_rows, count)
    return edge_weight


def _sparse_connect_core(edge_index, edge_weight, node_index, cluster_index, num_nodes, num_supernodes,
                         remove_self_loops, reduce_op, edge_weight_norm, batch_pooled, degree_norm, num_graphs,
                         padded, csr=None):
    w = _as_f32_weight(edge_weight)
    if reduce_op not in L.OPS:
        raise ValueError(f"unknown reduce_op '{reduce_op}'")
    edge_index = edge_index.contiguous()
    row, col = edge_index[0], edge_index[1]
    if num_nodes is None:  # maybe_num_nodes (base_conn.py:78) -- costs a device sync
        num_nodes = int(edge_index.max().item()) + 1 if edge_index.numel() > 0 else 0
    flags = L.REMOVE_SELF_LOOPS if remove_self_loops else 0
    need_norm = degree_norm or (edge_weight_norm and w is not None)
    need_grad = w is not None and w.requires_grad and torch.is_grad_enabled()

    if node_index is not None and len(node_index) < num_nodes:
        # the relabelling is monotone (node_index ascending), so the output keeps the row order of the input
        out_sorted = rows_sorted(edge_index) if need_norm else None
        ei, w_out, _, count = O.filter_relabel_edges(row, col, w, node_index.contiguous(), num_nodes, flags, EPS,
                                                     padded, need_grad)
    elif cluster_index is not None and len(cluster_index) == num_nodes:
        out_sorted = True  # coalesced output is lexicographic
        cluster_index = cluster_index.contiguous()
        if rows_sorted(edge_index):  # row-bucketed coalesce over the cluster CSR (cached on the SelectOutput)
            csr = csr if csr is not None else build_csr(cluster_index, num_supernodes)
        else:
            csr = (None, None)
        ei, w_out, _, _, _, count = O.remap_coalesce(row, col, w, cluster_index, csr[0], csr[1], num_nodes,
                                                     num_supernodes, L.OPS[reduce_op], flags, EPS, padded, need_grad)
    else:
        raise RuntimeError
    w = None if w is None else w_out
    w = edge_postprocess(ei, w, num_supernodes, degree_norm, edge_weight_norm, batch_pooled, num_graphs,
                         sorted_rows=out_sorted, count=count if padded else None)
    return ei, w, count


def sparse_connect(
    edge_index: Tensor,
    edge_weight: Optional[Tensor] = None,
    node_index: Optional[Tensor] = None,
    cluster_index: Optional[Tensor] = None,
    num_nodes: Optional[int] = None,
    num_supernodes: Optional[int] = None,
    remove_self_loops: bool = True,
    reduce_op: str = "sum",
    edge_weight_norm: bool = False,
    batch_pooled: Optional[Tensor] = None,
    degree_norm: bool = False,
    num_graphs: Optional[int] = None,
    csr: Optional[Tuple[Tensor, Tensor]] = None,
) -> Tuple[Tensor, Optional[Tensor]]:
    """Drop-in for ``tgp.connect.base_conn.sparse_connect`` (base_conn.py:57-112).

    Branch choice, output order and filters follow the reference: kept-node path when
    ``len(node_index) < num_nodes`` (input order kept, endpoints relabelled to their position in
    ``node_index``), cluster path when ``len(cluster_index) == num_nodes`` (lexicographic order,
    duplicates combined with ``reduce_op`` in original order), else ``RuntimeError``.
    One host read per call (the output edge count; ``num_graphs`` avoids a second one with
    ``edge_weight_norm``).
    """
    _require_cuda(edge_index)
    to_coo = edge_index.is_sparse
    if to_coo:
        coo = edge_index.coalesce() if not edge_index.is_coalesced() else edge_index
        edge_index, edge_weight = coo.indices().contiguous(), coo.values()
    else:
        _validate_edge_index(edge_index)
    ei, w, _ = _sparse_connect_core(edge_index, edge_weight, node_index, cluster_index, num_nodes, num_supernodes,
                                    remove_self_loops, reduce_op, edge_weight_norm, batch_pooled, degree_norm,
                                    num_graphs, False, csr)
    if to_coo:  # tgp/connect/base_conn.py:107-110 -> connectivity_to_torch_coo
        if w is None:
            w = torch.ones(ei.size(1), device=ei.device)
        return torch.sparse_coo_tensor(ei, w, (num_supernodes, num_supernodes)).coalesce(), None
    return ei, w


def sparse_connect_padded(
    edge_index: Tensor,
    edge_weight: Optional[Tensor] = None,
    node_index: Optional[Tensor] = None,
    cluster_index: Optional[Tensor] = None,
    num_nodes: Optional[int] = None,
    num_supernodes: Optional[int] = None,
    remove_self_loops: bool = True,
    reduce_op: str = "sum",
    edge_weight_norm: bool = False,
    batch_pooled: Optional[Tensor] = None,
    degree_norm: bool = False,
    num_graphs: Optional[int] = None,
    csr: Optional[Tuple[Tensor, Tensor]] = None,
) -> Tuple[Tensor, Optional[Tensor], Tensor]:
    """``sparse_connect`` without any host read: returns ``(edge_index [2, E], edge_weight [E], count)`` where only
    the first ``count`` (a device int64) columns are valid.  Every kernel bounds itself by the device-side count, so
    the whole call can be captured in a CUDA graph (``tgp_b200.GraphedStep``) -- the form for small, launch-bound
    batches; ``num_nodes`` and (with ``edge_weight_norm``) ``num_graphs`` must be given."""
    _require_cuda(edge_index)
    _validate_edge_index(edge_index)
    if num_nodes is None or (edge_weight_norm and num_graphs is None):
        raise ValueError("sparse_connect_padded needs num_nodes (and num_graphs with edge_weight_norm): no host reads")
    return _sparse_connect_core(edge_index, edge_weight, node_index, cluster_index, num_nodes, num_supernodes,
                                remove_self_loops, reduce_op, edge_weight_norm, batch_pooled, degree_norm, num_graphs,
                                True, csr)


# --------------------------------------------------------------------------- #
# Dense reduce + connect + losses
# --------------------------------------------------------------------------- #
LOSS_NONE, LOSS_MINCUT, LOSS_DIFFPOOL, LOSS_DMON = 0, 1, 2, 3


def dense_flags(remove_self_loops: bool, degree_norm: bool, adj_transpose: bool, edge_weight_norm: bool) -> int:
    return (
        (L.REMOVE_SELF_LOOPS if remove_self_loops else 0)
        | (L.DEGREE_NORM if degree_norm else 0)
        | (L.ADJ_TRANSPOSE if adj_transpose else 0)
        | (L.EDGE_WEIGHT_NORM if edge_weight_norm else 0)
    )


def dense_pool(
    x: Optional[Tensor],
    adj: Optional[Tensor],
    s: Tensor,
    *,
    remove_self_loops: bool = False,
    degree_norm: bool = False,
    adj_transpose: bool = False,
    edge_weight_norm: bool = False,
    loss_kind: int = LOSS_NONE,
    link_div: float = 1.0,
    ent_div: float = 1.0,
    graph_nodes: Optional[Tensor] = None,
):
    """Fused ``(S^T X, postprocess(S^T A S), losses[4])`` for batched dense inputs.

    ``losses`` = ``[mincut, ortho, link, entropy]`` (unused entries are 0); with ``loss_kind=LOSS_DMON`` it is
    ``[spectral, ortho, cluster, 0]``.  ``graph_nodes`` ([B], on the device): the number of valid nodes of each graph,
    which DMoN's cluster loss divides by (``None``: every graph has N nodes).
    """
    _require_cuda(x, adj, s, graph_nodes)
    if s.dim() != 3:
        raise ValueError("dense_pool expects s of shape [B, N, K]")
    if loss_kind == LOSS_DMON and adj is None:
        raise ValueError("dense_pool: the DMoN losses need adj")
    if graph_nodes is not None:
        if graph_nodes.shape != (s.size(0),):
            raise ValueError(f"dense_pool: graph_nodes must have shape [B] = [{s.size(0)}], got {list(graph_nodes.shape)}")
        graph_nodes = graph_nodes.to(torch.float32).contiguous()
    s = s.contiguous()
    x = None if x is None else x.contiguous()
    adj = None if adj is None else adj.contiguous()
    if x is not None and x.dtype != s.dtype or adj is not None and adj.dtype != s.dtype:
        raise RuntimeError("tgp_b200.dense_pool: x, adj and s must share one dtype")
    flags = dense_flags(remove_self_loops, degree_norm, adj_transpose, edge_weight_norm)
    x_pool, adj_pool, losses, _ = _T.stas_fused(x, adj, s, flags, loss_kind, float(link_div), float(ent_div),
                                                graph_nodes)
    return (x_pool if x is not None else None), (adj_pool if adj is not None else None), losses


def acc_losses(adj: Tensor, s: Tensor) -> Tensor:
    """``[total variation, balance]`` losses of Asymmetric Cheeger Cut pooling (TVGNN), batch means, from the RAW
    ``adj`` [B, N, N] and ``s`` [B, N, K] (padded rows zero), differentiable in both:

    * total variation: ``sum_ij A_ij ||S_i - S_j||_1 / (2 nnz(A_b))`` (self loops count; an edgeless graph gives NaN);
    * balance: ``1 - sum_ik f(S_ik - q_k) / (N (K - 1))`` with ``q_k`` the entry of rank ``N // K`` of column ``k`` in
      a stable descending sort over the N (padded) rows and ``f(d) = (K - 1) d`` for ``d >= 0``, ``-d`` otherwise.

    No ``[B, N, N, K]`` tensor is formed.  ``K < 2`` raises ``ValueError``."""
    _require_cuda(adj, s)
    if s.dim() == 3 and s.size(-1) < 2:
        raise ValueError(f"acc_losses needs K >= 2 clusters, got K = {s.size(-1)}")
    losses, _, _ = _T.acc_losses(adj.contiguous(), s.contiguous())
    return losses


HOSC_FIRST, HOSC_MOTIF, HOSC_ORTHO = 1, 2, 4


def hosc_losses(adj: Tensor, s: Tensor, alpha: float, hosc_ortho: bool, graph_nodes: Optional[Tensor] = None,
                eps: float = 1e-8) -> Tensor:
    """``[L1, L2, O]`` losses of HOSC pooling (higher-order spectral clustering), batch means, from the RAW ``adj``
    [B, N, N] and ``s`` [B, N, K] (padded rows zero), differentiable in both:

    * first-order cut ``L1 = -(1/K) sum_k n_k / m_k`` with ``n_k = (S^T A S)_kk``, ``m_k = sum_i d_i S_ik^2 + eps``,
      ``d = A 1``;
    * motif cut ``L2``: the same of the triangle-motif adjacency ``A_M = (A A) * A``;
    * ``O = (sqrt(K) - sum_k ||S_:k|| / sqrt(n_b)) / (sqrt(K) - 1)``, ``n_b = graph_nodes[b]`` (N when absent).

    The HOSC loss is ``(1 - alpha) L1 + alpha L2``.  Only the terms it needs are computed: ``L1`` is 0 when
    ``alpha == 1``, ``L2`` is 0 (and no ``A A`` product runs) when ``alpha == 0``, ``O`` is 0 unless ``hosc_ortho``.
    ``K < 2`` raises ``ValueError``."""
    _require_cuda(adj, s)
    if s.dim() == 3 and s.size(-1) < 2:
        raise ValueError(f"hosc_losses needs K >= 2 clusters, got K = {s.size(-1)}")
    alpha = float(alpha)
    terms = (HOSC_FIRST if alpha != 1.0 else 0) | (HOSC_MOTIF if alpha != 0.0 else 0) | (HOSC_ORTHO if hosc_ortho else 0)
    if graph_nodes is not None:
        graph_nodes = graph_nodes.to(torch.float32).contiguous()
    losses, _ = _T.hosc_losses(adj.contiguous(), s.contiguous(), graph_nodes, terms, float(eps))
    return losses


# --------------------------------------------------------------------------- #
# Dense -> block-diagonal sparse output, dense pre-processing
# --------------------------------------------------------------------------- #
class _BlockDiag(torch.autograd.Function):
    @staticmethod
    def forward(ctx, adj_pool, out_mask, eps):
        B, K = adj_pool.size(0), adj_pool.size(1)
        dev = adj_pool.device
        lib = L.load()
        ws = L.workspace(lib.tgpb200_block_diag_workspace_bytes(B, K), dev)
        counts = torch.zeros(2, dtype=torch.long, device=dev)
        m8 = None if out_mask is None else out_mask.to(torch.uint8).contiguous()
        dt = L.dtype_code(adj_pool.dtype)
        L.call("tgpb200_block_diag_count", L.ptr(adj_pool), L.ptr(m8), B, K, dt, eps, L.ptr(counts[1:]), L.ptr(counts[:1]),
               L.ptr(ws), ws.numel(), L.stream())
        n_out = int(counts[0].item())
        ei = torch.empty((2, n_out), dtype=torch.long, device=dev)
        w = torch.empty(n_out, dtype=adj_pool.dtype, device=dev)
        src = torch.empty(max(n_out, 1), dtype=torch.int32, device=dev)
        if n_out > 0:
            L.call("tgpb200_block_diag_emit", L.ptr(adj_pool), L.ptr(m8), B, K, dt, eps, L.ptr(ei[0]), L.ptr(ei[1]),
                   L.ptr(w), L.ptr(src), L.ptr(ws), ws.numel(), L.stream())
        ctx.mark_non_differentiable(ei)
        ctx.save_for_backward(src)
        ctx.shape, ctx.n_out = adj_pool.shape, n_out
        return ei, w

    @staticmethod
    def backward(ctx, _gei, gw):
        (src,) = ctx.saved_tensors
        gadj = torch.empty(ctx.shape, dtype=gw.dtype, device=gw.device)
        L.call("tgpb200_block_diag_bwd", L.ptr(gw.contiguous()), L.ptr(src), ctx.n_out, gadj.numel(),
               L.dtype_code(gw.dtype), L.ptr(gadj), L.stream())
        return gadj, None, None


def dense_to_block_diag(adj_pool: Tensor, out_mask: Optional[Tensor] = None) -> Tuple[Tensor, Tensor]:
    """tgp/utils/ops.py:53-82 (+ the masking / compact renumbering of tgp/src.py:526-552 when ``out_mask``
    [B, K] is given): entries with ``|a| > eps`` in row-major (b, i, j) order as a block-diagonal edge list."""
    _require_cuda(adj_pool, out_mask)
    if adj_pool.dim() == 2:
        adj_pool = adj_pool.unsqueeze(0)
    if adj_pool.dim() != 3:
        raise ValueError("adj_pool must have shape [B, K, K] or [K, K].")
    return _BlockDiag.apply(adj_pool.contiguous(), out_mask, EPS)


def finalize_sparse_output(x_pool: Tensor, adj_pool: Tensor, batch: Optional[Tensor], batch_pooled: Optional[Tensor],
                           out_mask: Optional[Tensor]):
    """DenseSRCPooling._finalize_sparse_output (tgp/src.py:500-557) given ``so.out_mask``."""
    B, K = adj_pool.size(0), adj_pool.size(1)
    x_flat = x_pool.reshape(-1, x_pool.size(-1))
    if batch_pooled is None and batch is not None and batch.numel() > 0:
        batch_pooled = torch.arange(int(batch.max().item()) + 1, device=x_pool.device).repeat_interleave(K)
    if batch_pooled is None and B > 1:
        batch_pooled = torch.arange(B, device=x_pool.device).repeat_interleave(K)
    if batch_pooled is None and out_mask is not None:
        batch_pooled = torch.zeros(B * K, dtype=torch.long, device=x_pool.device)
    edge_index, edge_weight = dense_to_block_diag(adj_pool, out_mask)
    if out_mask is not None:
        valid = out_mask.reshape(-1)
        x_flat = x_flat[valid]
        batch_pooled = batch_pooled[valid]
    return x_flat, edge_index, edge_weight, batch_pooled


def graph_ptr(batch: Tensor, num_graphs: int) -> Tensor:
    ptr = torch.empty(num_graphs + 1, dtype=torch.int32, device=batch.device)
    ws = L.workspace(L.load().tgpb200_graph_ptr_workspace_bytes(num_graphs), batch.device)
    L.call("tgpb200_graph_ptr", L.ptr(batch.contiguous()), batch.numel(), num_graphs, L.ptr(ptr), L.ptr(ws), ws.numel(),
           L.stream())
    return ptr


class _ToDenseBatch(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, batch, ptr, B, Nmax):
        N, F = x.shape
        out = torch.empty((B, Nmax, F), dtype=x.dtype, device=x.device)
        mask = torch.empty((B, Nmax), dtype=torch.uint8, device=x.device)
        L.call("tgpb200_to_dense_batch", L.ptr(x), L.ptr(batch), L.ptr(ptr), N, F, B, Nmax, L.dtype_code(x.dtype),
               L.ptr(out), L.ptr(mask), L.stream())
        ctx.save_for_backward(batch, ptr)
        ctx.Nmax = Nmax
        ctx.mark_non_differentiable(mask)
        return out, mask

    @staticmethod
    def backward(ctx, g, _gm):
        batch, ptr = ctx.saved_tensors
        n = batch.numel()
        idx = batch * ctx.Nmax + (torch.arange(n, device=batch.device) - ptr.long()[batch])
        return g.reshape(-1, g.size(-1))[idx], None, None, None, None


def to_dense_batch(x: Tensor, batch: Tensor, num_graphs: Optional[int] = None, max_num_nodes: Optional[int] = None):
    """PyG to_dense_batch (tgp/src.py:448-450): ``[N, F]`` + sorted ``batch`` -> zero-padded ``[B, Nmax, F]`` and a
    bool mask ``[B, Nmax]``."""
    _require_cuda(x, batch)
    B = num_graphs if num_graphs is not None else (int(batch.max().item()) + 1 if batch.numel() else 1)
    ptr = graph_ptr(batch, B)
    if max_num_nodes is None:
        max_num_nodes = int((ptr[1:] - ptr[:-1]).max().item())
    out, mask = _ToDenseBatch.apply(x.contiguous(), batch.contiguous(), ptr, B, max_num_nodes)
    return out, mask.bool()


def to_dense_adj(edge_index: Tensor, batch: Optional[Tensor], edge_weight: Optional[Tensor] = None,
                 num_graphs: Optional[int] = None, max_num_nodes: Optional[int] = None, transpose: bool = False) -> Tensor:
    """PyG to_dense_adj (tgp/src.py:434-443): ``[B, Nmax, Nmax]`` fp32, duplicates summed, default weight 1."""
    _require_cuda(edge_index, batch, edge_weight)
    dev = edge_index.device
    if batch is None:
        n = int(edge_index.max().item()) + 1 if edge_index.numel() else 0
        batch = torch.zeros(n, dtype=torch.long, device=dev)
    B = num_graphs if num_graphs is not None else (int(batch.max().item()) + 1 if batch.numel() else 1)
    ptr = graph_ptr(batch, B)
    if max_num_nodes is None:
        max_num_nodes = int((ptr[1:] - ptr[:-1]).max().item()) if batch.numel() else 0
    adj = torch.empty((B, max_num_nodes, max_num_nodes), dtype=torch.float32, device=dev)
    w = _as_f32_weight(edge_weight)
    ei = edge_index.contiguous()
    L.call("tgpb200_to_dense_adj", L.ptr(ei[0]), L.ptr(ei[1]), L.ptr(None if w is None else w.detach()), L.ptr(batch.contiguous()),
           L.ptr(ptr), ei.size(1), B, max_num_nodes, int(transpose), L.ptr(adj), L.stream())
    if w is not None and w.requires_grad:  # d adj / d w is a gather; keep it in autograd with an index_put view
        b = batch[ei[0]]
        lr, lc = ei[0] - ptr.long()[b], ei[1] - ptr.long()[b]
        if transpose:
            lr, lc = lc, lr
        adj = adj.detach() + torch.zeros_like(adj).index_put((b, lr, lc), w - w.detach(), accumulate=True)
    return adj
