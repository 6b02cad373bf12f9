"""Pooler-level orchestration of the path (what the pooler ``forward``s do after ``select``).

``mincut_pool`` / ``diff_pool`` / ``dmon_pool`` run reduce + connect + auxiliary losses + post-processing as ONE
fused forward and ONE fused backward; ``acc_pool`` adds the Asymmetric Cheeger Cut losses (their own kernels) to the
loss-free fused call, ``hosc_pool`` the HOSC cut losses (their own products and kernels); ``topk_pool`` / ``cluster_pool`` chain the sparse reduce and the sparse connect.  ``patch_pooler`` installs the B200 operators on a reference pooler object.
"""
from __future__ import annotations

from typing import Dict, Optional, Tuple

import torch
from torch import Tensor

from . import functional as F_
from .connect import B200DenseConnect, B200SparseConnect
from .reduce import B200Reduce


def mincut_pool(
    x: Tensor,
    adj: Tensor,
    s: Tensor,
    cut_loss_coeff: float = 1.0,
    ortho_loss_coeff: float = 1.0,
    remove_self_loops: bool = True,
    degree_norm: bool = True,
    adj_transpose: bool = True,
    edge_weight_norm: bool = False,
) -> Tuple[Tensor, Tensor, Dict[str, Tensor]]:
    """MinCutPooling.forward batched path after select (tgp/poolers/mincut.py:219-237, 291-310)."""
    x_pool, adj_pool, losses = F_.dense_pool(
        x, adj, s, remove_self_loops=remove_self_loops, degree_norm=degree_norm, adj_transpose=adj_transpose,
        edge_weight_norm=edge_weight_norm, loss_kind=F_.LOSS_MINCUT,
    )
    loss = {"cut_loss": losses[0] * cut_loss_coeff, "ortho_loss": losses[1] * ortho_loss_coeff}
    return x_pool, adj_pool, loss


def diff_pool(
    x: Tensor,
    adj: Tensor,
    s: Tensor,
    num_nodes: Optional[int] = None,
    link_loss_coeff: float = 1.0,
    ent_loss_coeff: float = 1.0,
    normalize_loss: bool = False,
    remove_self_loops: bool = True,
    degree_norm: bool = True,
    adj_transpose: bool = True,
    edge_weight_norm: bool = False,
) -> Tuple[Tensor, Tensor, Dict[str, Tensor]]:
    """DiffPool.forward batched path after select (tgp/poolers/diffpool.py:208-218, 262-284)."""
    if num_nodes is None:
        num_nodes = s.size(0) * s.size(1)
    x_pool, adj_pool, losses = F_.dense_pool(
        x, adj, s, remove_self_loops=remove_self_loops, degree_norm=degree_norm, adj_transpose=adj_transpose,
        edge_weight_norm=edge_weight_norm, loss_kind=F_.LOSS_DIFFPOOL,
        link_div=float(adj.numel()) if normalize_loss else 1.0, ent_div=float(num_nodes),
    )
    loss = {"link_loss": losses[2] * link_loss_coeff, "entropy_loss": losses[3] * ent_loss_coeff}
    return x_pool, adj_pool, loss


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
    """DMoNPooling.forward batched path after select: ``S^T X``, ``postprocess(S^T A S)`` and the spectral, cluster
    and orthogonality losses of PyG's ``DMoNPooling`` (restated in ``tests/dmon_oracle.py``), all from the raw product.
    ``mask`` [B, N] gives the valid node count of each graph (the cluster loss divides by it); it stays on the device.
    No activation is applied to the pooled features."""
    graph_nodes = None if mask is None else mask.sum(1).to(torch.float32)
    x_pool, adj_pool, losses = F_.dense_pool(
        x, adj, s, remove_self_loops=remove_self_loops, degree_norm=degree_norm, adj_transpose=adj_transpose,
        edge_weight_norm=edge_weight_norm, loss_kind=F_.LOSS_DMON, graph_nodes=graph_nodes,
    )
    loss = {"spectral_loss": losses[0] * spectral_loss_coeff, "cluster_loss": losses[2] * cluster_loss_coeff,
            "ortho_loss": losses[1] * ortho_loss_coeff}
    return x_pool, adj_pool, loss


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
    """AsymCheegerCutPooling.forward batched path after select: ``S^T X`` and ``postprocess(S^T A S)`` from the fused
    dense path (no loss there), and the total-variation and balance losses of Asymmetric Cheeger Cut pooling
    (restated in ``tests/acc_oracle.py``) from ``functional.acc_losses`` on the raw ``adj``."""
    x_pool, adj_pool, _ = F_.dense_pool(
        x, adj, s, remove_self_loops=remove_self_loops, degree_norm=degree_norm, adj_transpose=adj_transpose,
        edge_weight_norm=edge_weight_norm, loss_kind=F_.LOSS_NONE,
    )
    losses = F_.acc_losses(adj, s)
    tv_key, bal_key = _ACC_KEYS
    return x_pool, adj_pool, {tv_key: losses[0] * totvar_coeff, bal_key: losses[1] * balance_coeff}


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
) -> Tuple[Tensor, Tensor, Dict[str, Tensor]]:
    """HOSCPooling.forward batched path after select: ``S^T X`` and ``postprocess(S^T A S)`` from the fused dense path,
    the HOSC loss ``(1 - alpha) L1 + alpha L2`` (first-order and triangle-motif cuts, restated in
    ``tests/hosc_oracle.py``) from ``functional.hosc_losses`` on the raw ``adj``, and ``mu`` times the orthogonality
    term: MinCut's ``orthogonality_loss`` from the fused call, or with ``hosc_ortho`` HOSC's column-norm term, whose
    ``n_b`` is the valid node count of ``mask`` [B, N] (it stays on the device)."""
    graph_nodes = None if mask is None else mask.sum(1).to(torch.float32)
    x_pool, adj_pool, dl = F_.dense_pool(
        x, adj, s, remove_self_loops=remove_self_loops, degree_norm=degree_norm, adj_transpose=adj_transpose,
        edge_weight_norm=edge_weight_norm, loss_kind=F_.LOSS_NONE if hosc_ortho else F_.LOSS_MINCUT,
    )
    losses = F_.hosc_losses(adj, s, alpha, hosc_ortho, graph_nodes=graph_nodes)
    hosc = (1.0 - alpha) * losses[0] + alpha * losses[1]
    ortho = losses[2] if hosc_ortho else dl[1]
    return x_pool, adj_pool, {"hosc_loss": hosc, "ortho_loss": mu * ortho}


def sparse_pool(
    x: Tensor,
    edge_index: Tensor,
    so,
    edge_weight: Optional[Tensor] = None,
    batch: Optional[Tensor] = None,
    reduce_op: str = "sum",
    multiplier: float = 1.0,
    connect_op: str = "sum",
    remove_self_loops: bool = True,
    degree_norm: bool = False,
    edge_weight_norm: bool = False,
):
    """TopkPooling / GraclusPooling forward after select (tgp/poolers/topk.py:171-190,
    tgp/poolers/graclus.py:91-156): reduce, then connect."""
    x_pool, batch_pool = B200Reduce(reduce_op)(x, so, batch=batch)
    if multiplier != 1:
        x_pool = multiplier * x_pool
    conn = B200SparseConnect(connect_op, remove_self_loops, edge_weight_norm, degree_norm)
    ei, ew = conn(edge_index, so, edge_weight=edge_weight, batch_pooled=batch_pool)
    return x_pool, ei, ew, batch_pool


def sparse_pool_padded(
    x: Tensor,
    edge_index: Tensor,
    so,
    edge_weight: Optional[Tensor] = None,
    batch: Optional[Tensor] = None,
    reduce_op: str = "sum",
    connect_op: str = "sum",
    remove_self_loops: bool = True,
    degree_norm: bool = False,
    edge_weight_norm: bool = False,
    num_graphs: Optional[int] = None,
):
    """``sparse_pool`` with NO host read: the coarse edge list comes back padded to the input edge count together
    with the device-side count of valid edges, ``(x_pool, edge_index [2, E], edge_weight [E], batch_pool, count)``.
    Nothing in the call synchronises, so a whole forward + backward step on static tensors can be captured with
    ``tgp_b200.GraphedStep`` (small batches are launch-bound: ~40 launches and a host read per step otherwise)."""
    x_pool = F_.segment_reduce(x, so.node_index, so.cluster_index, so.weight, so.num_supernodes, reduce_op,
                               csr=F_.csr_of(so))
    batch_pool = None if batch is None else F_.reduce_batch_sparse(so, batch)
    ei, ew, count = F_.sparse_connect_padded(
        edge_index, edge_weight, node_index=so.node_index, cluster_index=so.cluster_index, num_nodes=so.num_nodes,
        num_supernodes=so.num_supernodes, remove_self_loops=remove_self_loops, reduce_op=connect_op,
        edge_weight_norm=edge_weight_norm, batch_pooled=batch_pool, degree_norm=degree_norm, num_graphs=num_graphs,
        csr=F_.csr_of(so) if len(so.cluster_index) == so.num_nodes else None)
    return x_pool, ei, ew, batch_pool, count


class PoolingOutput:
    """Stand-in for ``tgp.src.PoolingOutput`` when tgp itself is not importable (same attribute names)."""

    def __init__(self, x=None, edge_index=None, edge_weight=None, batch=None, so=None, loss=None):
        self.x, self.edge_index, self.edge_weight, self.batch, self.so, self.loss = x, edge_index, edge_weight, batch, so, loss

    def __iter__(self):
        return iter((self.x, self.edge_index, self.edge_weight, self.batch, self.so, self.loss))


def _pooling_output_cls():
    try:
        from tgp.src import PoolingOutput as Ref  # the user's pipeline expects the reference type

        return Ref
    except Exception:
        return PoolingOutput


# the loss keys of AsymCheegerCutPooling (total variation, balance)
_ACC_KEYS = ("total_variation_loss", "balance_loss")
_AGGR_TO_OP = {"SumAggregation": "sum", "MeanAggregation": "mean", "MaxAggregation": "max", "MinAggregation": "min"}


def _reduce_op_of(reducer) -> Optional[str]:
    """The segment operation a reference reducer performs: ``BaseReduce`` -> sum, ``AggrReduce`` with a PyG
    Sum / Mean / Max / Min aggregation -> that op; ``None`` for anything else (learned or order-statistic
    aggregators have no kernel here and must stay in place)."""
    name = type(reducer).__name__
    if name == "B200Reduce":
        return reducer.reduce_op
    if name == "BaseReduce":
        return "sum"
    if name == "AggrReduce":
        aggr = getattr(reducer, "aggr", None) or getattr(reducer, "operator", None)
        return _AGGR_TO_OP.get(type(aggr).__name__)
    return None


def _diff_forward(pooler, x, adj, s, mask, flags):
    x_pool, adj_pool, loss = diff_pool(x, adj, s, num_nodes=1, link_loss_coeff=pooler.link_loss_coeff,
                                       ent_loss_coeff=1.0, normalize_loss=pooler.normalize_loss, **flags)
    n_valid = mask.sum() if mask is not None else s.size(0) * s.size(1)  # stays on the device: no sync
    loss["entropy_loss"] = loss["entropy_loss"] / n_valid * pooler.ent_loss_coeff
    return x_pool, adj_pool, loss


# The dense poolers with a fused forward, by reference class name: (the attributes the fused forward reads that must
# exist for it to replace the reference's, ``(pooler, x, adj, s, mask, flags) -> (x_pool, adj_pool, loss)``).
# MinCutPooling and DiffPool require none: a missing attribute raises instead of falling back.
_FUSED_DENSE = {
    "MinCutPooling": (
        (), lambda p, x, adj, s, mask, flags: mincut_pool(x, adj, s, p.cut_loss_coeff, p.ortho_loss_coeff, **flags)),
    "DiffPool": ((), _diff_forward),
    "DMoNPooling": (
        ("spectral_loss_coeff", "cluster_loss_coeff", "ortho_loss_coeff"),
        lambda p, x, adj, s, mask, flags: dmon_pool(x, adj, s, mask, p.spectral_loss_coeff, p.cluster_loss_coeff,
                                                    p.ortho_loss_coeff, **flags)),
    "AsymCheegerCutPooling": (
        ("totvar_coeff", "balance_coeff"),
        lambda p, x, adj, s, mask, flags: acc_pool(x, adj, s, p.totvar_coeff, p.balance_coeff, **flags)),
    "HOSCPooling": (
        ("mu", "alpha", "hosc_ortho"),
        lambda p, x, adj, s, mask, flags: hosc_pool(x, adj, s, mask, p.mu, p.alpha, p.hosc_ortho, **flags)),
}


def _fused_dense_forward(pooler, pool):
    """``forward`` of a batched pooler of ``_FUSED_DENSE`` (tgp/poolers/mincut.py:210-258,
    tgp/poolers/diffpool.py:200-237) with reduce + connect + auxiliary losses + post-processing as ONE fused
    forward / backward through ``pool``, its entry's function; select, input densification, lifting and the unbatched
    mode stay the reference's."""
    ref_forward = pooler.forward
    Out = _pooling_output_cls()

    def forward(x, adj=None, edge_weight=None, so=None, mask=None, batch=None, batch_pooled=None, lifting=False,
                **kwargs):
        if lifting or not getattr(pooler, "batched", True):
            return ref_forward(x=x, adj=adj, edge_weight=edge_weight, so=so, mask=mask, batch=batch,
                               batch_pooled=batch_pooled, lifting=lifting, **kwargs)
        x, adj, mask = pooler._ensure_batched_inputs(x=x, edge_index=adj, edge_weight=edge_weight, batch=batch,
                                                     mask=mask)
        so = pooler.select(x=x, mask=mask)
        c = pooler.connector
        flags = dict(remove_self_loops=c.remove_self_loops, degree_norm=c.degree_norm, adj_transpose=c.adj_transpose,
                     edge_weight_norm=c.edge_weight_norm)
        x_pool, adj_pool, loss = pool(pooler, x, adj, so.s, mask, flags)
        batch_pooled = B200Reduce.reduce_batch(so, batch)
        if getattr(pooler, "sparse_output", False):
            xs, ei, ew, bp = pooler._finalize_sparse_output(x_pool=x_pool, adj_pool=adj_pool, batch=batch,
                                                            batch_pooled=batch_pooled, so=so)
            return Out(x=xs, edge_index=ei, edge_weight=ew, batch=bp, so=so, loss=loss)
        return Out(x=x_pool, edge_index=adj_pool, so=so, loss=loss)

    return forward


def patch_pooler(pooler, reduce_op: Optional[str] = None, fuse_dense: bool = True):
    """Install the B200 operators on a reference ``tgp`` pooler, in place.

    * ``pooler.connector`` (and ``preconnector``): ``SparseConnect`` / ``DenseConnect`` -> the B200 operator with the
      same ctor attributes (the poolers read them, tgp/poolers/mincut.py:233-236);
    * ``pooler.reducer``: ``BaseReduce`` / ``AggrReduce(sum | mean | max | min)`` -> ``B200Reduce`` with the SAME
      reduction; any other reducer (learned / order-statistic aggregators) is left in place.  ``reduce_op`` overrides;
    * ``fuse_dense``: a batched pooler whose class is in ``_FUSED_DENSE`` also gets the fused forward (reduce +
      connect + losses + post-processing on the device kernels) -- without it the patched pooler still calls the
      reference's torch loss functions.  A pooler lacking one of the attributes its entry requires keeps the
      reference forward.
    """
    for attr in ("connector", "preconnector"):
        conn = getattr(pooler, attr, None)
        if conn is None:
            continue
        name = type(conn).__name__
        if name == "SparseConnect":
            setattr(pooler, attr, B200SparseConnect(conn.reduce_op, conn.remove_self_loops, conn.edge_weight_norm,
                                                    conn.degree_norm))
        elif name == "DenseConnect":
            setattr(pooler, attr, B200DenseConnect(conn.remove_self_loops, conn.degree_norm, conn.adj_transpose,
                                                   conn.edge_weight_norm, conn.sparse_output))
    reducer = getattr(pooler, "reducer", None)
    if reducer is not None:
        op = reduce_op if reduce_op is not None else _reduce_op_of(reducer)
        if op is not None:
            pooler.reducer = B200Reduce(op)
    required, pool = _FUSED_DENSE.get(type(pooler).__name__, (None, None))
    if (fuse_dense and pool is not None and all(hasattr(pooler, a) for a in required)
            and type(getattr(pooler, "connector", None)).__name__ == "B200DenseConnect"):
        pooler.forward = _fused_dense_forward(pooler, pool)
    return pooler
