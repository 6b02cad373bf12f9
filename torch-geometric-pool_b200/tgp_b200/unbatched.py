"""Unbatched dense mode (``batched=False``): sparse adjacency + dense ``[N, K]`` assignment, no ``[B, N, N]`` tensor.

Mirror of ``DenseConnect._dense_connect_unbatched`` (tgp/connect/dense_conn.py:141-208) and of the sparse loss
twins ``sparse_mincut_loss`` / ``unbatched_orthogonality_loss`` / ``sparse_link_pred_loss``
(tgp/utils/losses.py:126-215, 319-389, 711-777).  The reference loops over the graphs of the batch in Python
(one ``torch.sparse.mm`` + one matmul per graph); here the whole batch is

* one SpMM ``W = A S`` (``[N, K]``): the segment-reduce kernel keyed by edge row, gathering rows of ``S``
  (deterministic, edge order inside a row), and
* one batched tensor-core product ``S_g^T W_g`` over the graphs padded to ``[B, Nmax, K]`` -- the padding is
  ``O(B Nmax K)``, never ``O(B Nmax^2)``, which is what the unbatched mode exists to avoid.

The losses reuse ``W`` (``tr(S^T A S) = sum_i <S_i, W_i>``), so they cost no extra pass over the edges and no
``[E, K]`` temporaries.

HOSC's motif cut needs ``A_M = (A A) . A`` on A's pattern: ``hosc_losses_unbatched`` coalesces the edge list into the
padded ``[B, Nmax]`` node layout and runs ``torch.ops.tgp_b200.hosc_losses_sparse`` (csrc/hosc_sparse.cu), whose
per-edge list intersection builds the triangle weights from the edge list; memory stays ``O(E + B Nmax K)``.
"""
from __future__ import annotations

import math
from typing import Dict, Optional, Tuple

import torch
from torch import Tensor

from . import _lib as L
from . import functional as F_
from . import ops as O

EPS = 1e-8


class _SpMM(torch.autograd.Function):
    """``out[i] = sum_{e: row_e = i} w_e x[col_e]`` (``A x`` for the COO adjacency); backward = SpMM with the
    transposed adjacency plus one row dot product per edge for the weights."""

    @staticmethod
    def forward(ctx, x, weight, row, col, num_nodes):
        E, F = row.numel(), x.size(1)
        order, ptr = F_.build_csr(row, num_nodes)
        out = torch.empty((num_nodes, F), dtype=x.dtype, device=x.device)
        dt = L.dtype_code(x.dtype)
        L.call("tgpb200_segment_reduce_fwd", L.ptr(x), L.ptr(col), L.ptr(weight), L.ptr(order), L.ptr(ptr), x.size(0), E,
               num_nodes, F, L.SUM, dt, dt, L.ptr(out), L.stream())
        ctx.save_for_backward(x, weight, row, col)
        ctx.N = num_nodes
        return out

    @staticmethod
    def backward(ctx, g):
        x, weight, row, col = ctx.saved_tensors
        E, F = row.numel(), x.size(1)
        g = g.contiguous()
        gx = None
        if ctx.needs_input_grad[0]:
            order, ptr = F_.build_csr(col, x.size(0))
            gx = torch.empty_like(x)
            dt = L.dtype_code(g.dtype)
            L.call("tgpb200_segment_reduce_fwd", L.ptr(g), L.ptr(row), L.ptr(weight), L.ptr(order), L.ptr(ptr), ctx.N, E,
                   x.size(0), F, L.SUM, dt, dt, L.ptr(gx), L.stream())
        gw = None
        if weight is not None and ctx.needs_input_grad[1]:
            gw = (g[row].float() * x[col].float()).sum(-1)
        return gx, gw, None, None, None


def spmm(edge_index: Tensor, edge_weight: Optional[Tensor], x: Tensor, num_nodes: Optional[int] = None) -> Tensor:
    """``A x`` for a COO adjacency (duplicates add up), differentiable in ``x`` and ``edge_weight``."""
    F_._require_cuda(edge_index, edge_weight, x)
    F_._validate_edge_index(edge_index)
    n = x.size(0) if num_nodes is None else num_nodes
    w = F_._as_f32_weight(edge_weight)
    ei = edge_index.contiguous()
    if ei.size(1) == 0:
        return x.new_zeros((n, x.size(1)))
    return _SpMM.apply(x.contiguous(), w, ei[0], ei[1], n)


class _BmmTN(torch.autograd.Function):
    """``a^T b`` per batch item: ``[B, N, K1]^T [B, N, K2] -> [B, K1, K2]`` (contraction over the nodes)."""

    @staticmethod
    def forward(ctx, a, b):
        B, N, K1 = a.shape
        K2 = b.size(-1)
        out = torch.empty((B, K1, K2), dtype=a.dtype, device=a.device)
        L.call("tgpb200_bmm", L.ptr(a), L.ptr(b), L.ptr(out), B, K1, K2, N, N * K1, K1, 1, N * K2, K2, 1,
               L.dtype_code(a.dtype), L.stream())
        ctx.save_for_backward(a, b)
        return out

    @staticmethod
    def backward(ctx, g):
        a, b = ctx.saved_tensors
        B, N, K1 = a.shape
        K2 = b.size(-1)
        g = g.contiguous()
        dt = L.dtype_code(a.dtype)
        ga = torch.empty_like(a)  # b g^T  [N, K1]
        L.call("tgpb200_bmm", L.ptr(b), L.ptr(g), L.ptr(ga), B, N, K1, K2, N * K2, K2, 0, K1 * K2, K2, 0, dt, L.stream())
        gb = torch.empty_like(b)  # a g    [N, K2]
        L.call("tgpb200_bmm", L.ptr(a), L.ptr(g), L.ptr(gb), B, N, K2, K1, N * K1, K1, 0, K1 * K2, K2, 1, dt, L.stream())
        return ga, gb


def _graphs_of(batch: Optional[Tensor], num_nodes: int, num_graphs: Optional[int], dev) -> Tuple[Tensor, int]:
    if batch is None:
        return torch.zeros(num_nodes, dtype=torch.long, device=dev), 1
    if num_graphs is None:  # the reference's own sync (losses.py:187, dense_conn.py:329): pass num_graphs to avoid it
        num_graphs = int(batch.max().item()) + 1 if batch.numel() else 1
    return batch, num_graphs


def _per_graph_sum(v: Tensor, batch: Tensor, num_graphs: int) -> Tensor:
    """Deterministic per-graph sums of a node vector (segment-reduce kernel in readout mode)."""
    nodes = torch.arange(v.numel(), device=v.device)
    return F_.segment_reduce(v.view(-1, 1).float(), nodes, batch, None, num_graphs, "sum",
                             csr=F_.build_csr(batch, num_graphs)).view(-1)


def dense_connect_unbatched(edge_index: Tensor, edge_weight: Optional[Tensor], batch: Optional[Tensor], s: Tensor,
                            num_graphs: Optional[int] = None, return_aux: bool = False):
    """Raw ``S^T A S`` ``[B, K, K]`` from a sparse adjacency and ``S [N, K]`` (dense_conn.py:141-208)."""
    N, K = s.shape
    batch, B = _graphs_of(batch, N, num_graphs, s.device)
    w_as = spmm(edge_index, edge_weight, s, N)  # A S
    s3, _ = F_.to_dense_batch(s, batch, B)
    w3, _ = F_.to_dense_batch(w_as, batch, B, s3.size(1))
    adj_pool = _BmmTN.apply(s3.contiguous(), w3.contiguous())
    return (adj_pool, w_as, s3, batch, B) if return_aux else adj_pool


def sparse_mincut_loss(edge_index: Tensor, S: Tensor, edge_weight: Optional[Tensor] = None,
                       batch: Optional[Tensor] = None, batch_reduction: str = "mean",
                       num_graphs: Optional[int] = None, _as: Optional[Tensor] = None) -> Tensor:
    """tgp/utils/losses.py:126-215: ``-tr(S^T A S) / (sum_i d_i |S_i|^2 + eps)`` per graph."""
    N = S.size(0)
    batch, B = _graphs_of(batch, N, num_graphs, S.device)
    w_as = _as if _as is not None else spmm(edge_index, edge_weight, S, N)
    deg = spmm(edge_index, edge_weight, torch.ones(N, 1, dtype=S.dtype, device=S.device), N).view(-1)
    num = _per_graph_sum((S * w_as).sum(-1), batch, B)
    den = _per_graph_sum(deg * (S * S).sum(-1), batch, B)
    loss = -(num / (den + EPS))
    return loss.mean(0) if batch_reduction == "mean" else loss.sum(0)


def unbatched_orthogonality_loss(S: Tensor, batch: Optional[Tensor] = None, batch_reduction: str = "mean",
                                 num_graphs: Optional[int] = None, _s3: Optional[Tensor] = None) -> Tensor:
    """tgp/utils/losses.py:319-389: per graph ``|| S_g^T S_g / ||.||_F - I / sqrt(K) ||_F`` (one batched product
    instead of the reference's loop over graphs)."""
    K = S.size(1)
    batch, B = _graphs_of(batch, S.size(0), num_graphs, S.device)
    s3 = _s3 if _s3 is not None else F_.to_dense_batch(S, batch, B)[0].contiguous()
    sts = _BmmTN.apply(s3, s3).float()
    sts = sts / torch.linalg.matrix_norm(sts, keepdim=True)
    loss = torch.linalg.matrix_norm(sts - torch.eye(K, device=S.device) / math.sqrt(K))
    return loss.mean(0) if batch_reduction == "mean" else loss.sum(0)


def sparse_link_pred_loss(S: Tensor, edge_index: Tensor, edge_weight: Optional[Tensor] = None,
                          batch: Optional[Tensor] = None, normalize_loss: bool = True,
                          num_graphs: Optional[int] = None, _as: Optional[Tensor] = None,
                          _s3: Optional[Tensor] = None) -> Tensor:
    """tgp/utils/losses.py:711-777.  The reference's ``sum_e (w - ss)^2 - sum_e ss^2`` equals
    ``sum_e w^2 - 2 sum_i <S_i, (A S)_i>`` term by term, so the edges are visited once (inside the SpMM) and no
    ``[E, K]`` gather is made; ``sum_g ||S_g^T S_g||_F^2`` comes from one batched product."""
    N = S.size(0)
    batch, B = _graphs_of(batch, N, num_graphs, S.device)
    w_as = _as if _as is not None else spmm(edge_index, edge_weight, S, N)
    w = F_._as_f32_weight(edge_weight)
    sum_w2 = (w * w).sum() if w is not None else torch.tensor(float(edge_index.size(1)), device=S.device)
    s3 = _s3 if _s3 is not None else F_.to_dense_batch(S, batch, B)[0].contiguous()
    sts = _BmmTN.apply(s3, s3).float()
    sq = sum_w2 - 2.0 * (S.float() * w_as.float()).sum() + (sts * sts).sum()
    link = torch.sqrt(torch.clamp(sq, min=0.0))
    if normalize_loss:
        counts = torch.bincount(batch, minlength=B).to(link.dtype)
        link = link / (counts * counts).sum().clamp(min=1.0)
    return link


def mincut_pool_unbatched(x: Tensor, edge_index: Tensor, edge_weight: Optional[Tensor], s: Tensor,
                          batch: Optional[Tensor] = None, num_graphs: Optional[int] = None,
                          cut_loss_coeff: float = 1.0, ortho_loss_coeff: float = 1.0, remove_self_loops: bool = True,
                          degree_norm: bool = True, edge_weight_norm: bool = False) -> Tuple[Tensor, Tensor, Dict]:
    """Unbatched MinCutPooling after select (tgp/poolers/mincut.py:260-289): reduce, connect and both losses from ONE
    SpMM and two batched products.  Returns ``(x_pool [B, K, F], adj_pool [B, K, K], losses)``."""
    from .connect import postprocess_adj_pool_dense

    raw, w_as, s3, b, B = dense_connect_unbatched(edge_index, edge_weight, batch, s, num_graphs, return_aux=True)
    x3, _ = F_.to_dense_batch(x, b, B, s3.size(1))
    x_pool = _BmmTN.apply(s3.contiguous(), x3.contiguous())
    loss = {"cut_loss": sparse_mincut_loss(edge_index, s, edge_weight, b, num_graphs=B, _as=w_as) * cut_loss_coeff,
            "ortho_loss": unbatched_orthogonality_loss(s, b, num_graphs=B, _s3=s3.contiguous()) * ortho_loss_coeff}
    adj_pool = postprocess_adj_pool_dense(raw, remove_self_loops=remove_self_loops, degree_norm=degree_norm,
                                          adj_transpose=False, edge_weight_norm=edge_weight_norm)
    return x_pool, adj_pool, loss


def _hosc_sparse(edge_index: Tensor, edge_weight: Optional[Tensor], s: Tensor, batch: Optional[Tensor], alpha: float,
                 hosc_ortho: bool, num_graphs: Optional[int], max_num_nodes: Optional[int], eps: float):
    """(losses [3], as1 = [A S | A 1 | 0..] [B, Nmax, K1] fp32, s3 [B, Nmax, K], batch, B, Nmax) of the sparse HOSC
    op.  One ``remap_coalesce`` maps node i of graph b to row ``b Nmax + (i - ptr[b])`` of the padded layout and sums
    duplicates (``to_dense_adj``); it keeps self loops and every run, zero-weight ones included (they still have a
    gradient), and carries the edge gradient back to the input edges."""
    F_._require_cuda(edge_index, edge_weight, s, batch)
    F_._validate_edge_index(edge_index)
    if s.dim() != 2:
        raise ValueError(f"hosc_losses_unbatched expects s of shape [N, K], got {tuple(s.shape)}")
    N, K = s.shape
    if K < 2:
        raise ValueError(f"hosc_losses_unbatched needs K >= 2 clusters, got K = {K}")
    dev = s.device
    batch, B = _graphs_of(batch, N, num_graphs, dev)
    batch = batch.contiguous()
    ptr = F_.graph_ptr(batch, B)
    counts = ptr[1:] - ptr[:-1]
    if max_num_nodes is None:
        max_num_nodes = int(counts.max().item()) if N > 0 else 1
    nmax = max(int(max_num_nodes), 1)
    R = B * nmax
    slot = batch * nmax + (torch.arange(N, device=dev) - ptr.long()[batch])
    ei = edge_index.contiguous()
    w = F_._as_f32_weight(edge_weight)
    if w is None:
        w = torch.ones(ei.size(1), dtype=torch.float32, device=dev)
    need_grad = w.requires_grad and torch.is_grad_enabled()
    csr = F_.build_csr(slot, R) if ei.size(1) > 0 and F_.rows_sorted(ei) else (None, None)
    # eps = -1 keeps every run: the filter drops |w| <= eps, and |w| >= 0 > -1
    ei_c, w_c, _, _, _, _ = O.remap_coalesce(ei[0], ei[1], w, slot, csr[0], csr[1], N, R, L.SUM, 0, -1.0, False,
                                             need_grad)
    row, col = ei_c[0], ei_c[1]
    _, row_ptr = F_.build_csr(row, R)
    col_order, col_ptr = F_.build_csr(col, R)  # stable: ascending row inside every column
    s3, _ = F_.to_dense_batch(s, batch, B, nmax)
    s3 = s3.contiguous()
    alpha = float(alpha)
    terms = ((F_.HOSC_FIRST if alpha != 1.0 else 0) | (F_.HOSC_MOTIF if alpha != 0.0 else 0)
             | (F_.HOSC_ORTHO if hosc_ortho else 0))
    losses, as1, _ = O._T.hosc_losses_sparse(row, col, w_c, row_ptr, col_ptr, col_order, s3, counts.float(), terms,
                                             float(eps))
    return losses, as1, s3, batch, B, nmax


def hosc_losses_unbatched(edge_index: Tensor, edge_weight: Optional[Tensor], s: Tensor, batch: Optional[Tensor] = None,
                          alpha: float = 0.5, hosc_ortho: bool = False, num_graphs: Optional[int] = None,
                          max_num_nodes: Optional[int] = None, eps: float = EPS) -> Tensor:
    """``[L1, L2, O]`` of HOSC pooling from a sparse adjacency and ``s [N, K]``: the values of
    ``functional.hosc_losses(to_dense_adj(edge_index, batch, edge_weight), to_dense_batch(s, batch)[0])`` with
    ``n_b`` each graph's own node count, without any ``[B, Nmax, Nmax]`` tensor.  Duplicates add up, self loops count,
    directed edges are taken as given.  ``L1`` is 0 when ``alpha == 1``, ``L2`` is 0 (and no motif kernel runs) when
    ``alpha == 0``, ``O`` is 0 unless ``hosc_ortho``.  Differentiable in ``s`` and ``edge_weight``; ``K < 2`` raises
    ``ValueError``."""
    return _hosc_sparse(edge_index, edge_weight, s, batch, alpha, hosc_ortho, num_graphs, max_num_nodes, eps)[0]


def hosc_pool_unbatched(x: Tensor, edge_index: Tensor, edge_weight: Optional[Tensor], s: Tensor,
                        batch: Optional[Tensor] = None, num_graphs: Optional[int] = None, mu: float = 0.1,
                        alpha: float = 0.5, hosc_ortho: bool = False, remove_self_loops: bool = True,
                        degree_norm: bool = True, edge_weight_norm: bool = False) -> Tuple[Tensor, Tensor, Dict]:
    """Unbatched HOSC pooling after select: ``x_pool = S^T X`` [B, K, F], ``adj_pool`` = post-processed ``S^T A S``
    [B, K, K] and ``{"hosc_loss": (1 - alpha) L1 + alpha L2, "ortho_loss": mu * O}`` (MinCut's orthogonality term
    without ``hosc_ortho``).  The connect's ``A S`` is the first K columns of the loss op's ``[A S | A 1]``: the
    adjacency is multiplied by ``S`` once."""
    from .connect import postprocess_adj_pool_dense

    losses, as1, s3, b, B, nmax = _hosc_sparse(edge_index, edge_weight, s, batch, alpha, hosc_ortho, num_graphs, None,
                                               EPS)
    K = s.size(1)
    raw = _BmmTN.apply(s3, as1[..., :K].to(s.dtype).contiguous())
    x3, _ = F_.to_dense_batch(x, b, B, nmax)
    x_pool = _BmmTN.apply(s3, x3.contiguous())
    ortho = losses[2] if hosc_ortho else unbatched_orthogonality_loss(s, b, num_graphs=B, _s3=s3)
    loss = {"hosc_loss": (1.0 - alpha) * losses[0] + alpha * losses[1], "ortho_loss": mu * ortho}
    adj_pool = postprocess_adj_pool_dense(raw, remove_self_loops=remove_self_loops, degree_norm=degree_norm,
                                          adj_transpose=False, edge_weight_norm=edge_weight_norm)
    return x_pool, adj_pool, loss
