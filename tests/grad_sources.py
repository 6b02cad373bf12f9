"""Per-source gradient checks of the dense poolers (MinCut, DiffPool, DMoN) against the float64 oracle.

A combined objective ``x_pool.gx + adj_pool.ga + sum(losses)`` hides the loss terms: the ``X Gx^T`` part of ``dS`` is
orders of magnitude larger than the cut, orthogonality, link, entropy, spectral or cluster parts, so a bound scaled by
the combined gradient accepts a loss term that is largely wrong or missing.  The helpers here take the gradient apart:

* ``hetero_batch``: graphs that differ from one another (density 0.02 .. 0.4, 0/1 and weighted entries, one
  non-symmetric graph, one scaled by 8, ragged valid-node counts, and a last graph with a hard one-hot assignment that
  leaves cluster K-1 empty), so that a per-graph coefficient read from the wrong graph shows;
* ``oracle``: the float64 reference gradient of ONE source (``gx``, ``ga`` or one loss with a non-unit coefficient),
  cached per (case, source) so that every device path of a case reuses it;
* ``assert_per_graph``: ``|got_b - ref_b| <= tau * max|ref_b|`` for every graph b of every gradient, with ``tau`` 1e-4
  for fp32 and 2e-2 for bf16 (the oracle then runs on the bf16-rounded operands).
"""
import functools
from typing import Dict, NamedTuple, Optional, Tuple

import torch
from torch import Tensor

import dmon_oracle as D
from oracle import ref_path as R

FP32_TAU, BF16_TAU = 1e-4, 2e-2
EPS = 1e-8

# loss_kind of dense_pool and the index of each loss in its losses[4]
FAMILIES = {
    "plain": (0, {}),
    "mincut": (1, {"cut": 0, "ortho": 1}),
    "diff": (2, {"link": 2, "entropy": 3}),
    "dmon": (3, {"spectral": 0, "ortho": 1, "cluster": 2}),
}
# non-unit, of both signs: a coefficient dropped or applied twice shows
LOSS_COEF = {"cut": 1.7, "ortho": -0.6, "link": -1.3, "entropy": 0.45, "spectral": -0.8, "cluster": 1.25}
# the poolers' defaults, and max-normalisation with row-sum degrees
FLAGSETS = (
    dict(remove_self_loops=True, degree_norm=True, adj_transpose=True, edge_weight_norm=False),
    dict(remove_self_loops=True, degree_norm=True, adj_transpose=False, edge_weight_norm=True),
)
GRADS = ("dS", "dX", "dA")

# Every path the dense backward can take, forced only by shape, dtype and the existing switches:
# (id, bf16, environment, families, shapes (B, N, K, F))
_FUSED_SHAPES = ((5, 256, 64, 128), (5, 200, 48, 100), (150, 64, 8, 16))
PATHS = (
    # fp32 k_dense_bwd_fused, element-wise terms in its epilogue (K <= 64, F <= 128, N, K, F multiples of 4)
    ("fp32-fused", False, {}, ("mincut", "diff"), _FUSED_SHAPES),
    # fp32 product chain, element-wise terms in the engine's ew_* hook
    ("fp32-chain", False, {"TGPB200_BWD_FUSED": "0"}, ("mincut", "diff"), _FUSED_SHAPES),
    # fp32 outside the fused envelope (K = 128; F = 256)
    ("fp32-wide", False, {}, ("mincut", "diff"), ((3, 256, 128, 64), (3, 128, 32, 256))),
    # fp32 FP32-pipe products, k_ds_elementwise and the scalar k_da_elementwise (K or N not a multiple of 4)
    ("fp32-pipe", False, {}, ("mincut", "diff"), ((4, 72, 6, 36), (4, 99, 16, 33))),
    # bf16 engine chain and the 128-bit k_da_elementwise_vec
    ("bf16", True, {}, ("mincut", "diff"), ((4, 256, 64, 128), (2, 256, 256, 256))),
    # bf16 with N not a multiple of 8: scalar k_da_elementwise
    ("bf16-scalar", True, {}, ("mincut", "diff"), ((4, 100, 16, 32),)),
    # DMoN: d_i u_k + v_k in the fused epilogue / k_ds_elementwise, the row term of k_dmon_bwd in dA
    ("dmon-fp32-fused", False, {}, ("dmon",), ((5, 256, 64, 128), (5, 200, 48, 100))),
    ("dmon-fp32-chain", False, {"TGPB200_BWD_FUSED": "0"}, ("dmon",), ((5, 256, 64, 128), (5, 200, 48, 100))),
    ("dmon-bf16", True, {}, ("dmon",), ((4, 256, 64, 128), (4, 100, 16, 32))),
    # the per-graph kernels split over the largest cluster of row strips
    ("fp32-strip64", False, {"TGPB200_STRIP_ELEMS": "64"}, ("mincut", "diff", "dmon"), ((5, 256, 64, 128),)),
    # loss_kind 0: the plain connect (no P, no element-wise terms)
    ("fp32-plain", False, {}, ("plain",), ((5, 256, 64, 128), (4, 99, 16, 33))),
)


def path_cases():
    """(path id, environment, Case) for every path, family, shape and flag set."""
    return [(pid, env, Case(fam, shape, fl, bf16))
            for pid, bf16, env, fams, shapes in PATHS for fam in fams for shape in shapes for fl in range(len(FLAGSETS))]


class Case(NamedTuple):
    family: str
    shape: Tuple[int, int, int, int]  # B, N, K, F
    flags: int = 0                    # index into FLAGSETS
    bf16: bool = False
    seed: int = 0

    @property
    def loss_kind(self) -> int:
        return FAMILIES[self.family][0]

    @property
    def sources(self) -> Tuple[str, ...]:
        return ("gx", "ga") + tuple(FAMILIES[self.family][1])

    @property
    def kw(self) -> dict:
        return FLAGSETS[self.flags]

    @property
    def tau(self) -> float:
        return BF16_TAU if self.bf16 else FP32_TAU

    @property
    def ent_div(self) -> float:
        return float(self.shape[0] * self.shape[1])


def hetero_batch(B: int, N: int, K: int, F: int, seed: int = 0):
    """(x, a, s, n) in float32: graph b has n[b] valid nodes (rows of x and s, rows and columns of a beyond are 0).
    Graph 0 is non-symmetric, graph 1 % B is scaled by 8, odd graphs and the last one are weighted, the last graph has
    a hard one-hot assignment with cluster K-1 empty (pooled degree 0: the clamp of the degree normalisation; s = 0:
    the entropy's log(eps))."""
    g = torch.Generator().manual_seed(1000 * seed + 7 * B + N + 3 * K + F)
    n = torch.tensor([N - (13 * b) % max(1, N // 4) for b in range(B)])
    mask = torch.arange(N)[None, :] < n[:, None]
    dens = torch.linspace(0.02, 0.4, B) if B > 1 else torch.tensor([0.1])
    a = torch.zeros(B, N, N)
    for b in range(B):
        e = (torch.rand(N, N, generator=g) < dens[b]).float()
        if b % 2 == 1 or b == B - 1:
            e = e * (torch.rand(N, N, generator=g) + 0.5)
        if b != 0:
            e = torch.triu(e, 1)
            e = e + e.t()
        a[b] = e * (8.0 if b == 1 % B else 1.0)
    a = a * (mask[:, :, None] & mask[:, None, :])
    # peaked soft assignments (the temperature varies by graph); the last graph hard, cluster K-1 left empty
    temp = torch.linspace(1.0, 3.0, B)[:, None, None]
    s = torch.softmax(temp * torch.randn(B, N, K, generator=g), -1)
    s[-1] = torch.nn.functional.one_hot(torch.randint(0, max(K - 1, 1), (N,), generator=g), K).float()
    s = s * mask[..., None]
    x = torch.randn(B, N, F, generator=g) * mask[..., None]
    return x, a, s, n


@functools.lru_cache(maxsize=None)
def inputs(case: Case):
    """hetero_batch of the case (bf16-rounded for a bf16 case) and the cotangents gx [B, K, F], ga [B, K, K]."""
    B, N, K, F = case.shape
    x, a, s, n = hetero_batch(B, N, K, F, case.seed)
    g = torch.Generator().manual_seed(99 + case.seed)
    gx, ga = torch.randn(B, K, F, generator=g), torch.randn(B, K, K, generator=g)
    if case.bf16:
        x, a, s, gx, ga = (t.bfloat16().float() for t in (x, a, s, gx, ga))
    return x, a, s, n, gx, ga


def reference_outputs(case: Case, x: Tensor, a: Tensor, s: Tensor, n: Tensor):
    """(x_pool, adj_pool, {loss name: value}) of the restated reference in the dtype of the inputs."""
    kw = case.kw
    if case.family in ("plain", "mincut"):
        xp, ap, loss = R.mincut_pool(x, a, s, **kw)
        return xp, ap, {"cut": loss["cut_loss"], "ortho": loss["ortho_loss"]}
    if case.family == "diff":
        xp, ap, loss = R.diff_pool(x, a, s, num_nodes=int(case.ent_div), normalize_loss=False, **kw)
        return xp, ap, {"link": loss["link_loss"], "entropy": loss["entropy_loss"]}
    mask = torch.arange(s.size(1))[None, :] < n[:, None]
    xp, ap, loss = D.dmon_pool(x, a, s, mask, **kw)
    return xp, ap, {"spectral": loss["spectral_loss"], "ortho": loss["ortho_loss"], "cluster": loss["cluster_loss"]}


def reference_grads(case: Case, sources, dtype=torch.float64) -> Dict[str, Tensor]:
    """{dS, dX, dA} of the sum of ``sources`` (each with its cotangent / coefficient), computed in ``dtype``."""
    x, a, s, n, gx, ga = inputs(case)
    x, a, s = (t.to(dtype).requires_grad_(True) for t in (x, a, s))
    xp, ap, loss = reference_outputs(case, x, a, s, n)
    obj = 0.0
    for src in sources:
        if src == "gx":
            obj = obj + (xp * gx.to(dtype)).sum()
        elif src == "ga":
            obj = obj + (ap * ga.to(dtype)).sum()
        else:
            obj = obj + LOSS_COEF[src] * loss[src]
    grads = torch.autograd.grad(obj, (s, x, a), allow_unused=True)
    return {k: (torch.zeros_like(t) if gr is None else gr.detach())
            for k, gr, t in zip(GRADS, grads, (s, x, a))}


@functools.lru_cache(maxsize=None)
def oracle(case: Case, source: str) -> Dict[str, Tensor]:
    """Float64 reference gradients of one source (cached: callers must not modify them)."""
    return reference_grads(case, (source,))


def assert_per_graph(got: Tensor, ref: Tensor, tau: float, name: str) -> None:
    """|got_b - ref_b| <= tau * max|ref_b| for every graph b; a graph whose reference is identically zero is bounded by
    tau times the batch scale of this gradient (max|ref| over the batch), so a gradient that is zero for every graph
    must be exactly zero.  NaN / Inf in ``got`` fail."""
    got, ref = got.detach().double().cpu(), ref.detach().double().cpu()
    assert got.shape == ref.shape, f"{name}: shape {tuple(got.shape)} != {tuple(ref.shape)}"
    B = ref.size(0)
    err = (got - ref).abs().reshape(B, -1).amax(1)
    scale = ref.abs().reshape(B, -1).amax(1)
    bound = tau * torch.where(scale > 0, scale, scale.max())
    bad = ~(err <= bound)
    if bool(bad.any()):
        worst = int(torch.nan_to_num(err / bound.clamp_min(1e-300), nan=float("inf")).argmax())
        raise AssertionError(f"{name}: graphs {bad.nonzero().flatten().tolist()} beyond {tau} * max|ref_b|; graph "
                             f"{worst}: err {float(err[worst]):.3e}, max|ref_b| {float(scale[worst]):.3e}")


def symmetrised(t: Tensor) -> Tensor:
    """Max-normalisation routes one gradient term to "the" arg-max; a symmetric adjacency ties (r, c) with (c, r) and
    the pick depends on rounding noise, so only the symmetric part of dA is defined."""
    return 0.5 * (t + t.transpose(1, 2))


def check_grads(case: Case, got: Dict[str, Optional[Tensor]], ref: Dict[str, Tensor], label: str,
                tau: Optional[float] = None) -> None:
    """assert_per_graph on every gradient in ``got`` (an entry left None is not checked)."""
    tau = case.tau if tau is None else tau
    for k in GRADS:
        if got.get(k) is None:
            continue
        g_, r_ = got[k], ref[k]
        if k == "dA" and case.kw["edge_weight_norm"]:
            g_, r_ = symmetrised(g_.double().cpu()), symmetrised(r_)
        assert_per_graph(g_, r_, tau, f"{label} {k}")
