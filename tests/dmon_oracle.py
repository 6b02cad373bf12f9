"""CPU reference of batched DMoN pooling (PyG's ``DMoNPooling`` losses, as tgp's ``spectral_loss`` / ``cluster_loss``
restate them), written on top of the restated reference path in ``oracle/ref_path.py`` the way its ``mincut_pool`` is:
losses from the RAW ``S^T A S``, then the connector's post-processing.  No golden vector from the reference's own
classes exists for these formulas: parity is pinned to this restatement."""
import math
from typing import Dict, Optional, Tuple

import torch
from torch import Tensor

from oracle.ref_path import (OracleSelectOutput, _batch_reduce, base_reduce, dense_connect, orthogonality_loss,
                             postprocess_adj_pool_dense)


def spectral_loss(adj: Tensor, S: Tensor, adj_pooled: Tensor, batch_reduction: str = "mean") -> Tensor:
    """mean_b -(tr(S^T A S) - ||S^T d||^2 / 2m) / 2m with d = A 1 (self loops included) and 2m = sum_i d_i; the trace
    comes from the RAW ``adj_pooled``.  A graph with 2m = 0 gives NaN."""
    d = adj.sum(-1)
    m2 = d.sum(-1)
    tr = torch.einsum("ijj->i", adj_pooled)
    c = torch.matmul(S.transpose(-2, -1), d.unsqueeze(-1)).squeeze(-1)
    return _batch_reduce(-(tr - (c * c).sum(-1) / m2) / m2, batch_reduction)


def cluster_loss(S: Tensor, mask: Optional[Tensor] = None, batch_reduction: str = "mean") -> Tensor:
    """mean_b ||S_b^T 1|| sqrt(K) / n_b - 1, n_b = mask.sum(1) (N without a mask); padded rows of S are zero."""
    n = mask.sum(1).to(S.dtype) if mask is not None else torch.full((S.size(0),), S.size(1), dtype=S.dtype)
    e = S.sum(-2)
    return _batch_reduce(torch.norm(e, dim=-1) * math.sqrt(S.size(-1)) / n - 1, batch_reduction)


def dmon_pool(
    x: Tensor,
    adj: Tensor,
    s: Tensor,
    mask: Optional[Tensor] = None,
    spectral_loss_coeff: float = 1.0,
    cluster_loss_coeff: float = 1.0,
    ortho_loss_coeff: float = 1.0,
    remove_self_loops: bool = True,
    degree_norm: bool = True,
    adj_transpose: bool = True,
    edge_weight_norm: bool = False,
) -> Tuple[Tensor, Tensor, Dict[str, Tensor]]:
    """DMoNPooling.forward batched path after select, written like ``mincut_pool``: the losses come from the RAW
    ``S^T A S`` (spectral_loss, cluster_loss, orthogonality_loss), then the connector's post-processing."""
    so = OracleSelectOutput(s=s)
    x_pool, _ = base_reduce(x, so)
    adj_pool = dense_connect(adj, s)
    loss = {
        "spectral_loss": spectral_loss(adj, s, adj_pool, "mean") * spectral_loss_coeff,
        "cluster_loss": cluster_loss(s, mask, "mean") * cluster_loss_coeff,
        "ortho_loss": orthogonality_loss(s, "mean") * ortho_loss_coeff,
    }
    adj_pool = postprocess_adj_pool_dense(
        adj_pool,
        remove_self_loops=remove_self_loops,
        degree_norm=degree_norm,
        adj_transpose=adj_transpose,
        edge_weight_norm=edge_weight_norm,
    )
    return x_pool, adj_pool, loss
