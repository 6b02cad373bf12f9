"""CPU reference of batched HOSC pooling (higher-order spectral clustering, Duval & Malliaros, CIKM 2022: the
first-order and triangle-motif normalised cuts of ``dense_hoscpool`` and its orthogonality terms), written on top of
the restated reference path in ``oracle/ref_path.py`` the way ``dmon_oracle.py`` and ``acc_oracle.py`` are: the losses
from the RAW ``adj`` and ``S``, the pooled outputs from ``S^T X`` and the connector's post-processing of ``S^T A S``.
No golden vector from the reference's own classes exists for these formulas: parity is pinned to this restatement."""
import math
from typing import Dict, Optional, Tuple

import torch
from torch import Tensor

from oracle.ref_path import (OracleSelectOutput, _batch_reduce, base_reduce, dense_connect, orthogonality_loss,
                             postprocess_adj_pool_dense)

EPS = 1e-8  # tgp's global eps, the value the MinCut path uses


def motif_adjacency(adj: Tensor) -> Tensor:
    """Triangle-motif adjacency ``A_M = (A A) . A``: A_M[i, j] weighs the triangles through the edge (i, j)."""
    return torch.matmul(adj, adj) * adj


def cut_loss(adj: Tensor, S: Tensor, eps: float = EPS, batch_reduction: str = "mean") -> Tensor:
    """mean_b -(1/K) sum_k n_k / m_k with n_k = (S^T A S)_kk, m_k = sum_i d_i S_ik^2 + eps, d = A 1.  An all-zero
    ``adj`` (e.g. the motif adjacency of a graph without triangles) gives 0."""
    d = adj.sum(-1)
    n = torch.einsum("bik,bij,bjk->bk", S, adj, S)
    m = torch.einsum("bi,bik->bk", d, S * S) + eps
    return _batch_reduce(-(n / m).sum(-1) / S.size(-1), batch_reduction)


def hosc_ortho_loss(S: Tensor, mask: Optional[Tensor] = None, batch_reduction: str = "mean") -> Tensor:
    """mean_b (sqrt(K) - sum_k ||S_:k||_2 / sqrt(n_b)) / (sqrt(K) - 1), n_b = mask.sum(1) (N without a mask)."""
    K = S.size(-1)
    n = mask.sum(1).to(S.dtype) if mask is not None else torch.full((S.size(0),), S.size(1), dtype=S.dtype)
    norms = torch.norm(S, dim=-2).sum(-1)
    return _batch_reduce((math.sqrt(K) - norms / torch.sqrt(n.to(S.device))) / (math.sqrt(K) - 1), batch_reduction)


def hosc_losses(adj: Tensor, S: Tensor, mask: Optional[Tensor] = None, eps: float = EPS) -> Tensor:
    """[L1, L2, O]: the first-order cut, the motif cut and the HOSC orthogonality term."""
    return torch.stack([cut_loss(adj, S, eps), cut_loss(motif_adjacency(adj), S, eps), hosc_ortho_loss(S, mask)])


def hosc_pool(
    x: Tensor,
    adj: Tensor,
    s: Tensor,
    mask: Optional[Tensor] = None,
    mu: float = 0.1,
    alpha: float = 0.5,
    hosc_ortho: bool = False,
    remove_self_loops: bool = True,
    degree_norm: bool = True,
    adj_transpose: bool = True,
    edge_weight_norm: bool = False,
    eps: float = EPS,
) -> Tuple[Tensor, Tensor, Dict[str, Tensor]]:
    """HOSCPooling.forward batched path after select: ``S^T X``, ``postprocess(S^T A S)``, the HOSC loss
    ``(1 - alpha) L1 + alpha L2`` of the raw inputs and ``mu`` times the orthogonality term (tgp's
    ``orthogonality_loss``, or HOSC's own with ``hosc_ortho``)."""
    so = OracleSelectOutput(s=s)
    x_pool, _ = base_reduce(x, so)
    adj_pool = dense_connect(adj, s)
    l1 = cut_loss(adj, s, eps)
    l2 = cut_loss(motif_adjacency(adj), s, eps)
    ortho = hosc_ortho_loss(s, mask) if hosc_ortho else orthogonality_loss(s, "mean")
    loss = {"hosc_loss": (1 - alpha) * l1 + alpha * l2, "ortho_loss": mu * ortho}
    adj_pool = postprocess_adj_pool_dense(
        adj_pool,
        remove_self_loops=remove_self_loops,
        degree_norm=degree_norm,
        adj_transpose=adj_transpose,
        edge_weight_norm=edge_weight_norm,
    )
    return x_pool, adj_pool, loss
