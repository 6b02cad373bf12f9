"""CPU reference of batched Asymmetric Cheeger Cut pooling (TVGNN's total-variation and asymmetric-norm balance
losses, as tgp's ``totvar_loss`` / ``asym_norm_loss`` are restated here), written on top of the restated reference
path in ``oracle/ref_path.py`` the way ``dmon_oracle.py`` is: the losses from the RAW ``adj`` and ``S``, the pooled
outputs from ``S^T X`` and the connector's post-processing of ``S^T A S``.  No golden vector from the reference's own
classes exists for these formulas: parity is pinned to this restatement."""
from typing import Dict, Tuple

import torch
from torch import Tensor

from oracle.ref_path import OracleSelectOutput, _batch_reduce, base_reduce, dense_connect, postprocess_adj_pool_dense


def totvar_loss(S: Tensor, adj: Tensor, batch_reduction: str = "mean") -> Tensor:
    """mean_b sum_ij A_ij ||S_i - S_j||_1 / (2 nnz(A_b)); self loops count in nnz, an edgeless graph gives NaN."""
    l1 = torch.sum(torch.abs(S[..., None, :] - S[:, None, ...]), dim=-1)  # [B, N, N]
    loss = torch.sum(adj * l1, dim=(-1, -2))
    n_edges = torch.count_nonzero(adj, dim=(-1, -2))
    return _batch_reduce(loss / (2 * n_edges), batch_reduction)


def quantile(S: Tensor) -> Tuple[Tensor, Tensor]:
    """(value, node) [B, K] that a stable descending sort of every column puts at position N // K (padded N)."""
    idx = S.size(-2) // S.size(-1)
    val, order = torch.sort(S, dim=-2, descending=True, stable=True)
    return val[:, idx, :], order[:, idx, :]


def asym_norm_loss(S: Tensor, batch_reduction: str = "mean") -> Tensor:
    """mean_b 1 - sum_ik f(S_ik - q_k) / (N (K - 1)), f(d) = (K - 1) d for d >= 0 and -d below."""
    B, N, K = S.shape
    idx = N // K
    quant = torch.sort(S, dim=-2, descending=True, stable=True)[0][:, idx, :]
    d = S - quant[:, None, :]
    loss = (d >= 0) * (K - 1) * d + (d < 0) * -d
    return _batch_reduce(1 - loss.sum((-1, -2)) / (N * (K - 1)), batch_reduction)


def acc_pool(
    x: Tensor,
    adj: Tensor,
    s: Tensor,
    totvar_coeff: float = 1.0,
    balance_coeff: float = 1.0,
    remove_self_loops: bool = True,
    degree_norm: bool = True,
    adj_transpose: bool = True,
    edge_weight_norm: bool = False,
) -> Tuple[Tensor, Tensor, Dict[str, Tensor]]:
    """AsymCheegerCutPooling.forward batched path after select: ``S^T X``, ``postprocess(S^T A S)`` and the two
    losses of the raw inputs."""
    so = OracleSelectOutput(s=s)
    x_pool, _ = base_reduce(x, so)
    adj_pool = dense_connect(adj, s)
    loss = {
        "total_variation_loss": totvar_loss(s, adj, "mean") * totvar_coeff,
        "balance_loss": asym_norm_loss(s, "mean") * balance_coeff,
    }
    adj_pool = postprocess_adj_pool_dense(
        adj_pool,
        remove_self_loops=remove_self_loops,
        degree_norm=degree_norm,
        adj_transpose=adj_transpose,
        edge_weight_norm=edge_weight_norm,
    )
    return x_pool, adj_pool, loss
