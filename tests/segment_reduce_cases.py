"""Cases, launch rules and float64 oracle of the sparse segment reduce (``csrc/sparse_reduce.cu``).

The host side of the segment reduce picks one of six kernels from the shape alone.  ``expected_paths`` restates those
rules in plain Python so that a test can say which kernel each case runs, and ``CASES`` puts every rule on both sides
of its threshold:

* forward (``launch_fwd``): 16-byte chunks when F is a multiple of the vector width W (4 for fp32, 8 for bf16) and the
  bases of ``x`` and ``out`` are 16-byte aligned; with chunks, rows of more than 16 chunks go to the row kernels,
  ``rows<8,1>`` when ``nnz <= K + K/4`` (about one member per cluster, TopK) and ``rows<4,2>`` otherwise;
* backward (``launch_bwd``): a node's first entry comes from a binary search of ``node_index`` when
  ``0 < N <= 32768`` and ``nnz <= 32768``, from the inverse map of ``k_first_entry`` otherwise; sum / mean without a
  weight gradient on aligned 16-byte chunks run ``bwd_rows<8>``, the rest the generic kernel with chunks (``vec``) or
  element by element (``scalar``); max / min count the ties first (``k_count_ties``).

``oracle`` computes what the reference computes (``R.base_reduce`` / ``R.aggr_reduce`` and their autograd) in
float64, together with the sum of the absolute values of the terms of every output element, which the component-wise
bounds of the GPU tests scale with.  Max / min compare the products in the precision the reference multiplies in:
float32 products for fp32 inputs, products rounded to bf16 for bf16 inputs; the gradient of a cluster is split evenly
among the members whose product equals the extreme.
"""
from __future__ import annotations

import zlib
from typing import Dict, NamedTuple, Optional, Tuple

import torch
from torch import Tensor

VEC = {"fp32": 4, "bf16": 8}          # elements per 16-byte chunk
DTYPES = {"fp32": torch.float32, "bf16": torch.bfloat16}
SEARCH_LIMIT = 32768                  # launch_bwd: binary search up to this N and nnz, inverse map above
OPS = ("sum", "mean", "max", "min")
FWD_PATHS = ("scalar", "vec", "rows41", "rows81")
BWD_PATHS = ("rows8", "vec", "scalar")
FIRST_PATHS = ("search", "map")
# widths on both sides of each forward rule: not a multiple of W; 16 chunks (generic kernel with chunks); 17 chunks
# (the first width with 32 lanes per row: row kernels); 32 chunks; several passes of the feature loop, the last partial
WIDTHS = {"fp32": (3, 64, 68, 128, 520), "bf16": (12, 128, 136, 256, 1032)}


class Case(NamedTuple):
    dtype: str                 # "fp32" / "bf16"
    op: str
    F: int
    N: int
    K: int                     # not a multiple of 8 unless a consumer shape asks for it
    layout: str                # "topk", "hard", "readout", "soft"
    nnz: int
    weights: str = "w"         # "none", "w" (weighted, no weight gradient), "wgrad"
    twice: bool = False        # also run twice and compare bitwise (C4 / C5-shaped)
    seed: int = 0

    @property
    def id(self) -> str:
        return (f"{self.dtype}-{self.op}-F{self.F}-N{self.N}-K{self.K}-{self.layout}{self.nnz}-{self.weights}"
                + ("-twice" if self.twice else ""))


def topk(dtype, op, F, N, K, extra=0, weights="w", **kw) -> Case:
    """A subset of K + extra of the N nodes, every cluster with one member, ``extra`` clusters with a second one."""
    return Case(dtype, op, F, N, K, "topk", K + extra, weights, **kw)


def hard(dtype, op, F, N, K, weights="w", **kw) -> Case:
    """Every node in one of the first K - 3 clusters (the last three stay empty)."""
    return Case(dtype, op, F, N, K, "hard", N, weights, **kw)


def readout(dtype, op, F, N, K, weights="none", **kw) -> Case:
    """Every node; cluster 0 holds about 85 % of them (one cluster of thousands of members, as in a readout)."""
    return Case(dtype, op, F, N, K, "readout", N, weights, **kw)


def soft(dtype, op, F, N, K, nnz, weights="w", **kw) -> Case:
    """``nnz`` distinct (node, cluster) pairs, every node in nnz / N clusters (rounded down or up)."""
    return Case(dtype, op, F, N, K, "soft", nnz, weights, **kw)


def _cases():
    cs = []
    for dt in ("fp32", "bf16"):
        rw, wide = WIDTHS[dt][3], WIDTHS[dt][4]      # row-kernel widths: 32 chunks; several passes
        narrow, chunked = WIDTHS[dt][0], WIDTHS[dt][1]
        for op in OPS:
            # every forward width rule on both sides; N % 8 = 3, K % 8 = 1 (partial warps of the row kernels)
            for F in WIDTHS[dt]:
                cs.append(hard(dt, op, F, 1003, 257, weights="w"))
            for F in (narrow, chunked, wide):  # the weight gradient: generic backward whatever the op
                cs.append(hard(dt, op, F, 1003, 257, weights="wgrad", seed=1))
            # nnz against K + K/4 (rows<8,1> / rows<4,2>) at both row widths
            cs.append(topk(dt, op, wide, 5003, 2001, extra=2001 // 4))
            cs.append(topk(dt, op, wide, 5003, 2001, extra=2001 // 4 + 1))
            cs.append(soft(dt, op, rw, 1003, 257, 2998, weights="wgrad" if op == "sum" else "w"))
            cs.append(readout(dt, op, rw, 2500, 5))
        cs.append(topk(dt, "sum", rw, 5003, 2001, weights="wgrad"))
        cs.append(topk(dt, "mean", rw, 5003, 2001, weights="none"))
        cs.append(topk(dt, "max", rw, 5003, 2001, extra=7, weights="w"))
        cs.append(topk(dt, "min", rw, 5003, 2001, extra=7, weights="wgrad"))
        # N and nnz around 32768: search at the limit, the inverse map one above (F <= 128)
        f = 128
        cs.append(topk(dt, "sum", f, 32768, 16001, extra=7))
        cs.append(topk(dt, "max", f, 32768, 16001, extra=7, weights="wgrad"))
        cs.append(topk(dt, "sum", f, 32769, 16001, extra=7))
        cs.append(topk(dt, "max", f, 32769, 16001, extra=7, weights="wgrad"))
        cs.append(soft(dt, "mean", f, 5000, 1001, 32768))
        cs.append(soft(dt, "mean", f, 5000, 1001, 32769))
        cs.append(soft(dt, "min", narrow, 5000, 1001, 32769, weights="none"))
        cs.append(soft(dt, "sum", chunked, 5000, 1001, 32769, weights="wgrad"))
    # C4-shaped (matching-style clusters, K ~ 0.55 N, mean) and C5-shaped (TopK 50 %, weighted sum), both on the map
    cs.append(hard("fp32", "mean", 128, 40000, 22003, weights="none", twice=True))
    cs.append(topk("fp32", "sum", 128, 70001, 35001, weights="w", twice=True))
    cs.append(topk("fp32", "sum", 128, 70001, 35001, weights="wgrad", twice=True))
    cs.append(topk("bf16", "sum", 128, 70001, 35001, weights="w", twice=True))
    return cs


CASES = _cases()


# --------------------------------------------------------------------------- #
# the launch rules of launch_fwd / launch_bwd
# --------------------------------------------------------------------------- #
def expected_paths(case: Case, aligned: bool = True) -> Tuple[str, str, str]:
    """(forward kernel, backward kernel, how the backward finds a node's first entry) that the library runs."""
    W = VEC[case.dtype]
    vec = case.F % W == 0 and aligned
    chunks = -(-case.F // W)
    lpr = 1
    while lpr < 32 and lpr < chunks:
        lpr <<= 1
    if vec and lpr == 32:
        fwd = "rows81" if case.nnz <= case.K + case.K // 4 else "rows41"
    else:
        fwd = "vec" if vec else "scalar"
    if vec and case.weights != "wgrad" and case.op in ("sum", "mean"):
        bwd = "rows8"
    else:
        bwd = "vec" if vec else "scalar"
    first = "search" if 0 < case.N <= SEARCH_LIMIT and case.nnz <= SEARCH_LIMIT else "map"
    return fwd, bwd, first


# --------------------------------------------------------------------------- #
# inputs
# --------------------------------------------------------------------------- #
def _index(case: Case, g: torch.Generator) -> Tuple[Tensor, Tensor]:
    """(node_index ascending, cluster_index) of the case's layout."""
    N, K, nnz = case.N, case.K, case.nnz
    if case.layout == "topk":
        node = torch.sort(torch.randperm(N, generator=g)[:nnz]).values
        cl = torch.cat([torch.arange(K), torch.randint(0, K, (nnz - K,), generator=g)])
        return node, cl[torch.randperm(nnz, generator=g)]
    if case.layout == "hard":
        return torch.arange(N), torch.randint(0, K - 3, (N,), generator=g)
    if case.layout == "readout":
        big = torch.rand(N, generator=g) < 0.85
        return torch.arange(N), torch.where(big, torch.zeros(N, dtype=torch.long), torch.randint(1, K, (N,), generator=g))
    if case.layout == "soft":
        j = torch.arange(nnz)
        node = j * N // nnz                                   # ascending; every node gets floor / ceil(nnz / N) entries
        first = torch.searchsorted(node, node, right=False)  # position of the node's first entry
        base = torch.randint(0, K, (N,), generator=g)
        cl = (base[node] + (j - first)) % K                   # distinct clusters per node (entries per node < K)
        key = torch.sort(node * K + cl).values                # coalesced order: (node, cluster) lexicographic
        return key // K, key % K
    raise ValueError(case.layout)


def _exact_ties(case: Case, x: Tensor, w: Optional[Tensor], node: Tensor, cl: Tensor, g: torch.Generator):
    """Max / min: copy the (row, weight) of one member of a cluster onto another member of the same cluster, for a few
    clusters with several members.  bf16 weighted cases also get ties that appear only after rounding: products
    4 (1 + 2^-7)^2 and 4 (1 + 2^-6) differ in float32 and round to the same bf16, and lead their clusters."""
    counts = torch.bincount(cl, minlength=case.K)
    multi = torch.nonzero(counts >= 2).flatten()
    if multi.numel() == 0:
        return
    sign = 1.0 if case.op == "max" else -1.0
    pick = multi[torch.randperm(multi.numel(), generator=g)[:16]]
    for i, c in enumerate(pick.tolist()):
        ent = torch.nonzero(cl == c).flatten()
        e0, e1 = int(ent[0]), int(ent[1])
        n0, n1 = int(node[e0]), int(node[e1])
        if n0 == n1:
            continue
        if case.dtype == "bf16" and w is not None and i % 2 == 1:
            x[n0] = sign * 4 * (1 + 2 ** -7)
            x[n1] = sign * 4 * (1 + 2 ** -6)
            w[e0], w[e1] = 1 + 2 ** -7, 1.0
        else:
            x[n1] = x[n0]
            if w is not None:
                w[e1] = w[e0]


def inputs(case: Case) -> Dict[str, Optional[Tensor]]:
    """CPU inputs in the case's dtype: x [N, F], node_index, cluster_index, weight [nnz] (or None), cotangent g [K, F]."""
    g = torch.Generator().manual_seed(zlib.crc32(case.id.encode()) + case.seed)
    node, cl = _index(case, g)
    x = torch.randn(case.N, case.F, generator=g)
    w = None if case.weights == "none" else torch.rand(case.nnz, generator=g) + 0.5
    dt = DTYPES[case.dtype]
    x = x.to(dt).float()
    w = None if w is None else w.to(dt).float()
    if case.op in ("max", "min"):
        _exact_ties(case, x, w, node, cl, g)
    cot = torch.randn(case.K, case.F, generator=g).to(dt)
    return {"x": x.to(dt), "node": node, "cluster": cl, "w": None if w is None else w.to(dt), "g": cot}


# --------------------------------------------------------------------------- #
# oracle
# --------------------------------------------------------------------------- #
def _products(x: Tensor, w: Optional[Tensor], node: Tensor, dtype: str) -> Tuple[Tensor, Tensor]:
    """(exact products in float64, products as the reference compares them for max / min)."""
    xs = x.double()[node]
    p = xs if w is None else xs * w.double()[:, None]
    if dtype == "fp32":
        pr = (x.float()[node] if w is None else x.float()[node] * w.float()[:, None]).double()
    else:  # a product of two bf16 values is exact in float32; the reference rounds it to bf16
        pr = p.float().bfloat16().double()
    return p, pr


def oracle(case: Case, x: Tensor, w: Optional[Tensor], node: Tensor, cl: Tensor, g: Tensor) -> Dict[str, Tensor]:
    """Float64 forward, dX and dW of ``op_{i in c} w_i x[node_i]`` with cotangent ``g``, and the sums of |terms|.

    Keys: ``out``, ``out_terms``, ``dx``, ``dx_terms``, ``dw``, ``dw_terms`` (``dw`` None without weights)."""
    K, F = case.K, x.size(1)
    p, pr = _products(x, w, node, case.dtype)
    idx = cl[:, None].expand(-1, F)
    cnt = torch.bincount(cl, minlength=K).double()
    gg = g.double()
    if case.op in ("sum", "mean"):
        out = torch.zeros(K, F, dtype=torch.float64).index_add_(0, cl, p)
        terms = torch.zeros(K, F, dtype=torch.float64).index_add_(0, cl, p.abs())
        coef = (1.0 / cnt.clamp(min=1))[cl][:, None] if case.op == "mean" else torch.ones(cl.numel(), 1, dtype=torch.float64)
        if case.op == "mean":
            out, terms = out / cnt.clamp(min=1)[:, None], terms / cnt.clamp(min=1)[:, None]
        gs = gg[cl] * coef                        # d out[c] / d p_i
    else:
        red = "amax" if case.op == "max" else "amin"
        ext = torch.zeros(K, F, dtype=torch.float64).scatter_reduce_(0, idx, pr, red, include_self=False)
        hit = (pr == ext[cl]).double()
        ties = torch.zeros(K, F, dtype=torch.float64).index_add_(0, cl, hit)
        gs = hit * gg[cl] / ties[cl].clamp(min=1)
        out, terms = ext, ext.abs()
    wi = torch.ones(cl.numel(), dtype=torch.float64) if w is None else w.double()
    dx = torch.zeros(case.N, F, dtype=torch.float64).index_add_(0, node, gs * wi[:, None])
    dx_terms = torch.zeros(case.N, F, dtype=torch.float64).index_add_(0, node, (gs * wi[:, None]).abs())
    res = {"out": out, "out_terms": terms, "dx": dx, "dx_terms": dx_terms, "dw": None, "dw_terms": None}
    if w is not None:
        xs = x.double()[node]
        res["dw"] = (xs * gs).sum(1)
        res["dw_terms"] = (xs * gs).abs().sum(1)
    return res


def reference_fp32_forward(case: Case, x: Tensor, w: Optional[Tensor], node: Tensor, cl: Tensor) -> Tensor:
    """The reference's own float32 forward (sequential CPU scatter in member order): what fp32 sum / max / min of the
    kernels reproduce bit for bit."""
    from oracle import ref_path as R

    vals = torch.ones(case.nnz) if w is None else w.float()
    so = R.OracleSelectOutput(s=torch.sparse_coo_tensor(torch.stack([node, cl]), vals, (case.N, case.K),
                                                        is_coalesced=True))
    with torch.no_grad():
        if case.op == "sum":
            return R.base_reduce(x.float(), so)[0]
        return R.aggr_reduce(x.float(), so, case.op)[0]
