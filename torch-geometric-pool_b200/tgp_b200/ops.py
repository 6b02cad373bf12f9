"""``torch.ops.tgp_b200.*``: the operators of the Reduce + Connect path as torch custom ops (SURVEY 8b).

* ``stas_fused`` / ``stas_fused_bwd``, ``segment_reduce`` / ``segment_reduce_bwd``, ``build_csr`` are C++ dispatcher
  ops (``csrc/torch_ops.cpp`` -> ``libtgp_b200_ops.so``: allocate with the caching allocator, take the current stream,
  call the C ABI of ``libtgp_b200.so``);
* ``filter_relabel_edges``, ``remap_coalesce``, ``degree_norm``, ``weight_norm`` (+ their ``*_bwd``) are
  ``torch.library.custom_op`` operators over the same C ABI (their host logic -- plan / count read-backs, capacity
  vs exact outputs -- is Python).

Every forward op has a fake (meta) kernel and an autograd formula registered with ``torch.library.register_autograd``;
the backward formulas are themselves ops.  There is no CPU kernel: CPU tensors fail in the dispatcher ("no kernel for
CPU"), a missing library fails at import.
"""
from __future__ import annotations

import os
from typing import Optional, Tuple

import torch
from torch import Tensor

from . import _lib as L

_OPS_PATH = os.path.join(os.path.dirname(os.path.abspath(__file__)), "libtgp_b200_ops.so")
EPS = 1e-8
PLAN_SYNC_MIN_EDGES = 1 << 20  # larger row-sorted inputs read the bucket plan back to size the launches exactly


def _load_ops() -> None:
    L.load()  # libtgp_b200.so first: the ops library resolves its C-ABI symbols against it
    if not os.path.isfile(_OPS_PATH):
        raise RuntimeError(
            f"tgp_b200: {_OPS_PATH} not found. Build it with `bash torch-geometric-pool_b200/csrc/build.sh` "
            "(or __graft_entry__.build()). There is no CPU / eager fallback.")
    torch.ops.load_library(_OPS_PATH)


_load_ops()
_T = torch.ops.tgp_b200


# --------------------------------------------------------------------------------------------------------------
# stas_fused: (x_pool, adj_pool, losses[4], saved) = fused S^T X, postprocess(S^T A S), auxiliary losses
# --------------------------------------------------------------------------------------------------------------
@torch.library.register_fake("tgp_b200::stas_fused")
def _stas_fused_fake(x, adj, s, flags, loss_kind, link_div, ent_div, graph_nodes=None):
    B, N, K = s.shape
    F = x.size(-1) if x is not None else 0
    saved = L.load().tgpb200_dense_pool_saved_bytes(B, N, K)
    return (s.new_empty((B if x is not None else 0, K, F)), s.new_empty((B if adj is not None else 0, K, K)),
            s.new_empty((4,), dtype=torch.float32), s.new_empty((max(saved, 256),), dtype=torch.uint8))


@torch.library.register_fake("tgp_b200::stas_fused_bwd")
def _stas_fused_bwd_fake(x, adj, s, saved, gx_pool, gadj_pool, glosses, flags, loss_kind, link_div, ent_div, need_gadj,
                         graph_nodes=None):
    gx = torch.empty_like(x) if x is not None else s.new_empty((0,))
    ga = torch.empty_like(adj) if (adj is not None and need_gadj) else s.new_empty((0,))
    return gx, ga, torch.empty_like(s)


def _stas_setup(ctx, inputs, output):
    x, adj, s, flags, loss_kind, link_div, ent_div, graph_nodes = inputs
    ctx.save_for_backward(x, adj, s, output[3], graph_nodes)
    ctx.cfg = (flags, loss_kind, link_div, ent_div)
    ctx.set_materialize_grads(False)


def _stas_backward(ctx, gx_pool, gadj_pool, glosses, _gsaved):
    x, adj, s, saved, graph_nodes = ctx.saved_tensors
    need_adj = adj is not None and ctx.needs_input_grad[1]
    gx, ga, gs = _T.stas_fused_bwd(x, adj, s, saved, gx_pool, gadj_pool, glosses, *ctx.cfg, need_adj, graph_nodes)
    # one entry per argument the call passed (the dispatcher drops trailing arguments left at their default)
    rest = (None,) * (len(ctx.needs_input_grad) - 3)
    return ((gx if x is not None else None), (ga if need_adj else None), gs) + rest


torch.library.register_autograd("tgp_b200::stas_fused", _stas_backward, setup_context=_stas_setup)


# --------------------------------------------------------------------------------------------------------------
# build_csr, segment_reduce
# --------------------------------------------------------------------------------------------------------------
@torch.library.register_fake("tgp_b200::build_csr")
def _build_csr_fake(cluster_index, num_clusters):
    return (cluster_index.new_empty((max(cluster_index.numel(), 1),), dtype=torch.int32),
            cluster_index.new_empty((num_clusters + 1,), dtype=torch.int32))


@torch.library.register_fake("tgp_b200::segment_reduce")
def _segment_reduce_fake(x, node_index, cluster_index, weight, order, ptr, num_clusters, op):
    return x.new_empty((num_clusters, x.size(1)))


@torch.library.register_fake("tgp_b200::segment_reduce_bwd")
def _segment_reduce_bwd_fake(x, node_index, cluster_index, weight, order, ptr, x_pool, grad, num_clusters, op,
                             need_weight_grad):
    nw = node_index.numel() if (weight is not None and need_weight_grad) else 0
    return torch.empty_like(x), x.new_empty((nw,), dtype=torch.float32)


def _segred_setup(ctx, inputs, output):
    x, node_index, cluster_index, weight, order, ptr, num_clusters, op = inputs
    ctx.save_for_backward(x, node_index, cluster_index, weight, order, ptr, output)
    ctx.cfg = (num_clusters, op)


def _segred_backward(ctx, g):
    x, node_index, cluster_index, weight, order, ptr, out = ctx.saved_tensors
    need_w = weight is not None and ctx.needs_input_grad[3]
    gx, gw = _T.segment_reduce_bwd(x, node_index, cluster_index, weight, order, ptr, out, g, *ctx.cfg, need_w)
    return gx, None, None, (gw if need_w else None), None, None, None, None


torch.library.register_autograd("tgp_b200::segment_reduce", _segred_backward, setup_context=_segred_setup)


# --------------------------------------------------------------------------------------------------------------
# filter_relabel_edges: kept-node branch + self-loop / tiny-weight filters (one order-preserving compaction)
#   padded = False: exact-size outputs (one host read of the survivor count)
#   padded = True : capacity-E outputs plus the device-side count, no host read (CUDA-graph capturable)
# returns (edge_index [2, n], weight [n] or [0], src_edge [n] or [0], count [1])
# --------------------------------------------------------------------------------------------------------------
@torch.library.custom_op("tgp_b200::filter_relabel_edges", mutates_args=(), device_types="cuda")
def filter_relabel_edges(row: Tensor, col: Tensor, edge_weight: Optional[Tensor], node_index: Tensor, num_nodes: int,
                         flags: int, eps: float, padded: bool, need_src: bool) -> Tuple[Tensor, Tensor, Tensor, Tensor]:
    E, dev = row.numel(), row.device
    lib = L.load()
    ws = L.workspace(lib.tgpb200_filter_relabel_onepass_workspace_bytes(E, num_nodes), dev)
    count = torch.empty(1, dtype=torch.long, device=dev)
    cap = max(E, 1)
    ei_c = torch.empty((2, cap), dtype=torch.long, device=dev)
    w_c = None if edge_weight is None else torch.empty(cap, dtype=torch.float32, device=dev)
    src_c = torch.empty(cap, dtype=torch.int32, device=dev) if need_src else None
    L.call("tgpb200_filter_relabel_onepass", L.ptr(row), L.ptr(col), L.ptr(edge_weight), E, L.ptr(node_index),
           node_index.numel(), num_nodes, flags, eps, L.ptr(ei_c[0]), L.ptr(ei_c[1]), L.ptr(w_c), L.ptr(src_c),
           L.ptr(count), L.ptr(ws), ws.numel(), L.stream())
    empty_f = torch.empty(0, dtype=torch.float32, device=dev)
    empty_i = torch.empty(0, dtype=torch.int32, device=dev)
    if padded:
        return (ei_c[:, :E].clone() if E == 0 else ei_c, w_c if w_c is not None else empty_f,
                src_c if src_c is not None else empty_i, count)
    n_out = int(count.item())  # the one device->host word: sizes the exact, contiguous outputs
    return (ei_c[:, :n_out].contiguous(), w_c[:n_out].clone() if w_c is not None else empty_f,
            src_c[:max(n_out, 1)].clone() if src_c is not None else empty_i, count)


@filter_relabel_edges.register_fake
def _filter_relabel_fake(row, col, edge_weight, node_index, num_nodes, flags, eps, padded, need_src):
    n = max(row.numel(), 1) if padded else torch.library.get_ctx().new_dynamic_size()
    return (row.new_empty((2, n)), row.new_empty((n if edge_weight is not None else 0,), dtype=torch.float32),
            row.new_empty((n if need_src else 0,), dtype=torch.int32), row.new_empty((1,)))


@torch.library.custom_op("tgp_b200::filter_relabel_edges_bwd", mutates_args=(), device_types="cuda")
def filter_relabel_edges_bwd(grad_out: Tensor, src_edge: Tensor, count: Optional[Tensor], num_out: int,
                             num_edges: int) -> Tensor:
    gin = torch.empty(num_edges, dtype=torch.float32, device=grad_out.device)
    L.call("tgpb200_filter_relabel_bwd", L.ptr(grad_out.contiguous()), L.ptr(src_edge), num_out, L.ptr(count), num_edges,
           L.ptr(gin), L.stream())
    return gin


@filter_relabel_edges_bwd.register_fake
def _filter_relabel_bwd_fake(grad_out, src_edge, count, num_out, num_edges):
    return grad_out.new_empty((num_edges,), dtype=torch.float32)


def _fr_setup(ctx, inputs, output):
    row, col, edge_weight, node_index, num_nodes, flags, eps, padded, need_src = inputs
    ei, w, src, count = output
    ctx.save_for_backward(src, count if padded else None)
    ctx.E, ctx.n_out = row.numel(), (row.numel() if padded else ei.size(1))


def _fr_backward(ctx, _gei, gw, _gsrc, _gcount):
    src, count = ctx.saved_tensors
    if gw is None or src.numel() == 0:
        return (None,) * 9
    return None, None, filter_relabel_edges_bwd(gw, src, count, ctx.n_out, ctx.E), None, None, None, None, None, None


torch.library.register_autograd("tgp_b200::filter_relabel_edges", _fr_backward, setup_context=_fr_setup)


# --------------------------------------------------------------------------------------------------------------
# remap_coalesce: cluster branch.  Row-sorted edge lists (order / ptr = cluster CSR given) take the row-bucketed
# coalesce, other inputs the generic remap -> global stable radix sort -> in-order combine; identical results.
# returns (edge_index [2, n], weight [n] or [0], edge_slot [E] or [0], run_len [n] or [0], run_aux [n] or [0], count)
# --------------------------------------------------------------------------------------------------------------
@torch.library.custom_op("tgp_b200::remap_coalesce", mutates_args=(), device_types="cuda")
def remap_coalesce(row: Tensor, col: Tensor, edge_weight: Optional[Tensor], cluster_index: Tensor,
                   order: Optional[Tensor], ptr: Optional[Tensor], num_nodes: int, num_clusters: int, op: int,
                   flags: int, eps: float, padded: bool,
                   need_slots: bool) -> Tuple[Tensor, Tensor, Tensor, Tensor, Tensor, Tensor]:
    E, dev = row.numel(), row.device
    lib = L.load()
    weighted = edge_weight is not None
    need_grad = weighted and need_slots
    count = torch.empty(1, dtype=torch.long, device=dev)
    bucketed = order is not None and E > 0 and E + num_nodes < 2 ** 31 - 1
    virt_cap = -1
    if bucketed:
        ws = L.workspace(lib.tgpb200_bucket_coalesce_workspace_bytes(E, num_nodes, num_clusters), dev)
        plan = torch.empty(4, dtype=torch.long, device=dev)
        L.call("tgpb200_bucket_coalesce_plan", L.ptr(row), E, L.ptr(cluster_index), L.ptr(order), L.ptr(ptr),
               num_nodes, num_clusters, L.ptr(plan), L.ptr(ws), ws.numel(), L.stream())
        hub_cap = -1
        if not padded and E >= PLAN_SYNC_MIN_EDGES:
            virt_cap, hub_cap = plan[:2].tolist()  # one host read: exact launch sizes for large graphs
        L.call("tgpb200_bucket_coalesce_count", L.ptr(row), L.ptr(col), L.ptr(edge_weight), E, L.ptr(cluster_index),
               L.ptr(order), L.ptr(ptr), num_nodes, num_clusters, op, flags, eps, virt_cap, hub_cap, int(need_grad),
               L.ptr(count), L.ptr(ws), ws.numel(), L.stream())
    else:
        ws = L.workspace(lib.tgpb200_remap_coalesce_workspace_bytes(E, num_clusters), dev)
        L.call("tgpb200_remap_coalesce_count", L.ptr(row), L.ptr(col), L.ptr(edge_weight), E, L.ptr(cluster_index),
               num_nodes, num_clusters, op, flags, eps, L.ptr(count), L.ptr(ws), ws.numel(), L.stream())
    n_out = E if padded else int(count.item())
    ei = torch.empty((2, n_out), dtype=torch.long, device=dev)
    w_out = torch.empty(n_out if weighted else 0, dtype=torch.float32, device=dev)
    slot = torch.empty(max(E, 1) if need_grad else 0, dtype=torch.int32, device=dev)
    run_len = torch.empty(max(n_out, 1) if need_grad else 0, dtype=torch.int32, device=dev)
    run_aux = torch.empty(max(n_out, 1) if (need_grad and bucketed and op == L.MUL) else 0, dtype=torch.float32,
                          device=dev)
    opt = lambda t: L.ptr(t) if t.numel() > 0 else None  # noqa: E731
    if n_out > 0 and bucketed:
        L.call("tgpb200_bucket_coalesce_emit", E, num_nodes, num_clusters, int(weighted), virt_cap, L.ptr(ei[0]),
               L.ptr(ei[1]), opt(w_out), opt(slot), opt(run_len), opt(run_aux), L.ptr(ws), ws.numel(), L.stream())
    elif n_out > 0:
        L.call("tgpb200_remap_coalesce_emit", E, num_clusters, int(weighted), flags, eps, L.ptr(ei[0]), L.ptr(ei[1]),
               opt(w_out), opt(slot), opt(run_len), L.ptr(ws), ws.numel(), L.stream())
    elif slot.numel() > 0:
        slot.fill_(-1)
    return ei, w_out, slot, run_len, run_aux, count


@remap_coalesce.register_fake
def _remap_coalesce_fake(row, col, edge_weight, cluster_index, order, ptr, num_nodes, num_clusters, op, flags, eps,
                         padded, need_slots):
    E = row.numel()
    n = E if padded else torch.library.get_ctx().new_dynamic_size()
    weighted = edge_weight is not None
    g = weighted and need_slots
    return (row.new_empty((2, n)), row.new_empty((n if weighted else 0,), dtype=torch.float32),
            row.new_empty((max(E, 1) if g else 0,), dtype=torch.int32),
            row.new_empty((n if g else 0,), dtype=torch.int32),
            row.new_empty((n if (g and order is not None and op == L.MUL) else 0,), dtype=torch.float32),
            row.new_empty((1,)))


@torch.library.custom_op("tgp_b200::remap_coalesce_bwd", mutates_args=(), device_types="cuda")
def remap_coalesce_bwd(edge_weight: Tensor, out_weight: Tensor, grad_out: Tensor, edge_slot: Tensor, run_len: Tensor,
                       run_aux: Tensor, num_out: int, op: int) -> Tensor:
    E = edge_weight.numel()
    gin = torch.empty(E, dtype=torch.float32, device=grad_out.device)
    ws = L.workspace(L.load().tgpb200_coalesce_bwd_workspace_bytes(E, num_out, op), grad_out.device)
    L.call("tgpb200_coalesce_bwd", L.ptr(edge_weight), L.ptr(out_weight), L.ptr(grad_out.contiguous()),
           L.ptr(edge_slot), L.ptr(run_len), L.ptr(run_aux) if run_aux.numel() > 0 else None, E, num_out, op,
           L.ptr(gin), L.ptr(ws), ws.numel(), L.stream())
    return gin


@remap_coalesce_bwd.register_fake
def _remap_coalesce_bwd_fake(edge_weight, out_weight, grad_out, edge_slot, run_len, run_aux, num_out, op):
    return torch.empty_like(edge_weight, dtype=torch.float32)


def _rc_setup(ctx, inputs, output):
    edge_weight, op = inputs[2], inputs[8]
    ei, w_out, slot, run_len, run_aux, count = output
    ctx.save_for_backward(edge_weight, w_out, slot, run_len, run_aux)
    ctx.op, ctx.n_out = op, ei.size(1)


def _rc_backward(ctx, _gei, gw, _gslot, _grl, _gra, _gcount):
    w, w_out, slot, run_len, run_aux = ctx.saved_tensors
    if gw is None or w is None or slot.numel() == 0:
        return (None,) * 13
    gin = remap_coalesce_bwd(w, w_out, gw, slot, run_len, run_aux, ctx.n_out, ctx.op)
    return (None, None, gin) + (None,) * 10


torch.library.register_autograd("tgp_b200::remap_coalesce", _rc_backward, setup_context=_rc_setup)


# --------------------------------------------------------------------------------------------------------------
# degree_norm / weight_norm (postprocess_adj_pool_sparse, tgp/utils/ops.py:383-417); deterministic sums.
# `count` (optional device int64) bounds the valid edges of a padded list.
# --------------------------------------------------------------------------------------------------------------
def _norm_ws(E: int, K: int, dev) -> Tensor:
    return L.workspace(L.load().tgpb200_edge_norm_workspace_bytes(E, K), dev)


@torch.library.custom_op("tgp_b200::degree_norm", mutates_args=(), device_types="cuda")
def degree_norm(w: Optional[Tensor], row: Tensor, col: Tensor, num_clusters: int, eps: float, sorted_rows: bool,
                count: Optional[Tensor]) -> Tuple[Tensor, Tensor]:
    E, dev = row.numel(), row.device
    deg = torch.empty(max(num_clusters, 1), dtype=torch.float32, device=dev)
    out = torch.empty(E, dtype=torch.float32, device=dev)
    ws = _norm_ws(E, num_clusters, dev)
    L.call("tgpb200_degree_norm_fwd", L.ptr(row), L.ptr(col), L.ptr(w), E, L.ptr(count), num_clusters, eps,
           int(sorted_rows), L.ptr(deg), L.ptr(out), L.ptr(ws), ws.numel(), L.stream())
    return out, deg


@degree_norm.register_fake
def _degree_norm_fake(w, row, col, num_clusters, eps, sorted_rows, count):
    return (row.new_empty((row.numel(),), dtype=torch.float32),
            row.new_empty((max(num_clusters, 1),), dtype=torch.float32))


@torch.library.custom_op("tgp_b200::degree_norm_bwd", mutates_args=(), device_types="cuda")
def degree_norm_bwd(w: Tensor, row: Tensor, col: Tensor, deg: Tensor, grad_out: Tensor, num_clusters: int, eps: float,
                    sorted_rows: bool, count: Optional[Tensor]) -> Tensor:
    E, dev = row.numel(), row.device
    gd = torch.empty(max(num_clusters, 1), dtype=torch.float32, device=dev)
    gw = torch.empty(E, dtype=torch.float32, device=dev)
    ws = _norm_ws(E, num_clusters, dev)
    L.call("tgpb200_degree_norm_bwd", L.ptr(row), L.ptr(col), L.ptr(w), L.ptr(deg), L.ptr(grad_out.contiguous()), E,
           L.ptr(count), num_clusters, eps, int(sorted_rows), L.ptr(gd), L.ptr(gw), L.ptr(ws), ws.numel(), L.stream())
    return gw


@degree_norm_bwd.register_fake
def _degree_norm_bwd_fake(w, row, col, deg, grad_out, num_clusters, eps, sorted_rows, count):
    return torch.empty_like(grad_out)


def _dn_setup(ctx, inputs, output):
    w, row, col, num_clusters, eps, sorted_rows, count = inputs
    ctx.save_for_backward(w, row, col, output[1], count)
    ctx.cfg = (num_clusters, eps, sorted_rows)


def _dn_backward(ctx, g, _gdeg):
    w, row, col, deg, count = ctx.saved_tensors
    if w is None or g is None:
        return (None,) * 7
    return (degree_norm_bwd(w, row, col, deg, g, *ctx.cfg, count),) + (None,) * 6


torch.library.register_autograd("tgp_b200::degree_norm", _dn_backward, setup_context=_dn_setup)


@torch.library.custom_op("tgp_b200::weight_norm", mutates_args=(), device_types="cuda")
def weight_norm(w: Tensor, row: Tensor, batch_pooled: Tensor, num_clusters: int, num_graphs: int, sorted_rows: bool,
                count: Optional[Tensor]) -> Tuple[Tensor, Tensor, Tensor]:
    E, dev = row.numel(), row.device
    mx = torch.empty(max(num_graphs, 1), dtype=torch.float32, device=dev)
    arg = torch.empty(max(num_graphs, 1), dtype=torch.int32, device=dev)
    out = torch.empty(E, dtype=torch.float32, device=dev)
    L.call("tgpb200_weight_norm_fwd", L.ptr(row), L.ptr(w), L.ptr(batch_pooled), E, L.ptr(count), num_graphs, L.ptr(mx),
           L.ptr(arg), L.ptr(out), L.stream())
    return out, mx, arg


@weight_norm.register_fake
def _weight_norm_fake(w, row, batch_pooled, num_clusters, num_graphs, sorted_rows, count):
    g = max(num_graphs, 1)
    return torch.empty_like(w), w.new_empty((g,)), w.new_empty((g,), dtype=torch.int32)


@torch.library.custom_op("tgp_b200::weight_norm_bwd", mutates_args=(), device_types="cuda")
def weight_norm_bwd(w: Tensor, row: Tensor, batch_pooled: Tensor, mx: Tensor, arg: Tensor, grad_out: Tensor,
                    num_clusters: int, num_graphs: int, sorted_rows: bool, count: Optional[Tensor]) -> Tensor:
    E, dev = row.numel(), row.device
    acc = torch.empty(max(num_graphs, 1), dtype=torch.float32, device=dev)
    gw = torch.empty(E, dtype=torch.float32, device=dev)
    ws = _norm_ws(E, max(num_clusters, num_graphs), dev)
    L.call("tgpb200_weight_norm_bwd", L.ptr(row), L.ptr(w), L.ptr(batch_pooled), L.ptr(mx), L.ptr(arg),
           L.ptr(grad_out.contiguous()), E, L.ptr(count), num_clusters, num_graphs, int(sorted_rows), L.ptr(acc),
           L.ptr(gw), L.ptr(ws), ws.numel(), L.stream())
    return gw


@weight_norm_bwd.register_fake
def _weight_norm_bwd_fake(w, row, batch_pooled, mx, arg, grad_out, num_clusters, num_graphs, sorted_rows, count):
    return torch.empty_like(grad_out)


def _wn_setup(ctx, inputs, output):
    w, row, batch_pooled, num_clusters, num_graphs, sorted_rows, count = inputs
    ctx.save_for_backward(w, row, batch_pooled, output[1], output[2], count)
    ctx.cfg = (num_clusters, num_graphs, sorted_rows)


def _wn_backward(ctx, g, _gmx, _garg):
    w, row, batch_pooled, mx, arg, count = ctx.saved_tensors
    if g is None:
        return (None,) * 7
    return (weight_norm_bwd(w, row, batch_pooled, mx, arg, g, *ctx.cfg, count),) + (None,) * 6


torch.library.register_autograd("tgp_b200::weight_norm", _wn_backward, setup_context=_wn_setup)

OP_NAMES = ("stas_fused", "stas_fused_bwd", "build_csr", "segment_reduce", "segment_reduce_bwd", "filter_relabel_edges",
            "filter_relabel_edges_bwd", "remap_coalesce", "remap_coalesce_bwd", "degree_norm", "degree_norm_bwd",
            "weight_norm", "weight_norm_bwd")
