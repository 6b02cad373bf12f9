"""Pooler-level orchestration of the path (what the pooler ``forward``s do after ``select``).

``mincut_pool`` / ``diff_pool`` / ``dmon_pool`` run reduce + connect + auxiliary losses + post-processing as ONE
fused forward and ONE fused backward; ``topk_pool`` / ``cluster_pool`` chain the sparse reduce and
the sparse connect.  ``patch_pooler`` installs the B200 operators on a reference pooler object.
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


_DMON_COEFFS = ("spectral_loss_coeff", "cluster_loss_coeff", "ortho_loss_coeff")
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


def _fused_dense_forward(pooler, kind: str):
    """``forward`` of a batched ``MinCutPooling`` / ``DiffPool`` / ``DMoNPooling`` (tgp/poolers/mincut.py:210-258,
    tgp/poolers/diffpool.py:200-237) with reduce + connect + auxiliary losses + post-processing as ONE fused
    forward / backward; select, input densification, lifting and the unbatched mode stay the reference's."""
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
        if kind == "mincut":
            x_pool, adj_pool, loss = mincut_pool(x, adj, so.s, pooler.cut_loss_coeff, pooler.ortho_loss_coeff, **flags)
        elif kind == "dmon":
            x_pool, adj_pool, loss = dmon_pool(x, adj, so.s, mask, pooler.spectral_loss_coeff, pooler.cluster_loss_coeff,
                                               pooler.ortho_loss_coeff, **flags)
        else:
            x_pool, adj_pool, loss = diff_pool(x, adj, so.s, num_nodes=1, link_loss_coeff=pooler.link_loss_coeff,
                                               ent_loss_coeff=1.0, normalize_loss=pooler.normalize_loss, **flags)
            n_valid = mask.sum() if mask is not None else so.s.size(0) * so.s.size(1)  # stays on the device: no sync
            loss["entropy_loss"] = loss["entropy_loss"] / n_valid * pooler.ent_loss_coeff
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
    * ``fuse_dense``: a batched ``MinCutPooling`` / ``DiffPool`` / ``DMoNPooling`` also gets the fused forward
      (reduce + connect + losses + post-processing in one kernel chain) -- without it the patched pooler still calls
      the reference's torch loss functions.  A ``DMoNPooling`` lacking one of ``spectral_loss_coeff``,
      ``cluster_loss_coeff``, ``ortho_loss_coeff`` keeps the reference forward.
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
    kind = {"MinCutPooling": "mincut", "DiffPool": "diff", "DMoNPooling": "dmon"}.get(type(pooler).__name__)
    if kind == "dmon" and not all(hasattr(pooler, a) for a in _DMON_COEFFS):
        kind = None
    if fuse_dense and kind is not None and type(getattr(pooler, "connector", None)).__name__ == "B200DenseConnect":
        pooler.forward = _fused_dense_forward(pooler, kind)
    return pooler
