"""B200: every launch path of the sparse segment reduce against the float64 oracle, aligned and unaligned.

Cases, launch rules and oracle: ``segment_reduce_cases``.  Bars (DESIGN.md section 2):

* fp32 forward: sum, max and min bit-identical to the reference's sequential float32 CPU reduce; mean
  ``|err| <= 1e-5 * sum|terms|`` against float64;
* fp32 backward: dX and the weight gradient ``|err| <= 1e-5 * sum|terms|`` against float64 (the terms of the weight
  gradient are the products of its row dot product); max / min split the gradient evenly among tied products;
* bf16: ``2e-2 * max|ref|`` per output against float64 on the bf16-rounded inputs; max / min forward exactly the
  extreme of the bf16-rounded products;
* unaligned: ``x`` and the cotangent as contiguous views one element off a 16-byte boundary take the scalar kernels,
  which do the same arithmetic in the same order: ``x_pool`` and dX bitwise equal to the aligned run, the weight
  gradient at the oracle bar.

The consumers of the kernels (sparse lift, unbatched SpMM, readout) run at row-kernel widths, and the dense poolers
take unaligned inputs and cotangents one at a time (the fallbacks behind their alignment guards).
"""
import pytest
import torch

import grad_sources as G
import segment_reduce_cases as S
import tgp_b200 as T
from tgp_b200 import functional as F_
from tgp_b200 import unbatched as U

pytestmark = pytest.mark.gpu
DEV = "cuda"


def unaligned(t: torch.Tensor) -> torch.Tensor:
    """A contiguous copy of ``t`` on the device whose data starts one element after a 16-byte boundary."""
    buf = torch.empty(t.numel() + 1, dtype=t.dtype, device=DEV)
    v = buf[1:].view(t.shape)
    v.copy_(t)
    assert v.is_contiguous() and v.data_ptr() % 16 != 0
    return v


def close_cw(got, ref, cond, name, rtol=1e-5):
    """|got - ref| <= rtol * cond element-wise (cond: sum of the absolute values of the terms)."""
    err = (got.double().cpu() - ref).abs()
    bound = rtol * cond + 1e-30
    bad = ~(err <= bound)
    assert not bool(bad.any()), f"{name}: {int(bad.sum())} elements beyond {rtol} * sum|terms|, worst ratio " \
                                f"{float(torch.nan_to_num(err / bound, nan=float('inf')).max()):.3f}"


def close_bf16(got, ref, name):
    got = got.double().cpu()
    scale = float(ref.abs().max()) if ref.numel() else 0.0
    err = float((got - ref).abs().max()) if ref.numel() else 0.0
    assert bool(torch.isfinite(got).all()), f"{name}: not finite"
    assert err <= 2e-2 * scale, f"{name}: max error {err:.3e} beyond 2e-2 * max|ref| = {2e-2 * scale:.3e}"


def run(case, inp, x_unaligned=False, g_unaligned=False):
    """Device (x_pool, dX, dW) through F_.segment_reduce and autograd."""
    node, cl = inp["node"].to(DEV), inp["cluster"].to(DEV)
    if x_unaligned:
        buf = torch.zeros(inp["x"].numel() + 1, dtype=inp["x"].dtype, device=DEV)
        buf[1:].copy_(inp["x"].flatten())
        buf.requires_grad_(True)
        x = buf[1:].view(inp["x"].shape)
        assert x.data_ptr() % 16 != 0
    else:
        buf = x = inp["x"].to(DEV).requires_grad_(True)
    w = None
    if inp["w"] is not None:
        w = inp["w"].to(DEV).requires_grad_(case.weights == "wgrad")
    out = F_.segment_reduce(x, node, cl, w, case.K, case.op)
    g = inp["g"].to(DEV)
    seen = []
    out.register_hook(lambda t: seen.append(t.data_ptr() % 16))
    if g_unaligned:  # the cotangent of x_pool after a concatenation: contiguous, one element off
        z = out.new_zeros(1)
        torch.cat([z, out.flatten()]).backward(torch.cat([z, g.flatten()]))
        assert seen and seen[0] != 0, "the cotangent reached the reduce aligned"
    else:
        out.backward(g)
    dx = buf.grad[1:].view(inp["x"].shape) if x_unaligned else buf.grad
    dw = w.grad if case.weights == "wgrad" else None
    torch.cuda.synchronize()
    return out.detach().cpu(), dx.cpu(), (None if dw is None else dw.cpu())


def check_against_oracle(case, inp, got, label):
    out, dx, dw = got
    ref = S.oracle(case, inp["x"], inp["w"], inp["node"], inp["cluster"], inp["g"])
    if case.dtype == "fp32":
        if case.op == "mean":
            close_cw(out, ref["out"], ref["out_terms"], f"{label} x_pool")
        else:
            exp = S.reference_fp32_forward(case, inp["x"], inp["w"], inp["node"], inp["cluster"])
            assert torch.equal(out, exp), f"{label} x_pool: fp32 {case.op} is not bit-identical to the reference " \
                                          f"({int((out != exp).sum())} elements differ)"
        close_cw(dx, ref["dx"], ref["dx_terms"], f"{label} dX")
        if dw is not None:
            close_cw(dw, ref["dw"], ref["dw_terms"], f"{label} dW")
    else:
        if case.op in ("max", "min"):
            exp = ref["out"].float().bfloat16()
            assert torch.equal(out, exp), f"{label} x_pool: bf16 {case.op} is not the extreme of the rounded products"
        else:
            close_bf16(out, ref["out"], f"{label} x_pool")
        close_bf16(dx, ref["dx"], f"{label} dX")
        if dw is not None:
            close_bf16(dw, ref["dw"], f"{label} dW")
    unselected = torch.ones(case.N, dtype=torch.bool)
    unselected[inp["node"]] = False
    assert not bool(dx[unselected].any()), f"{label}: rows of unselected nodes are not exactly zero"


@pytest.mark.parametrize("case", S.CASES, ids=[c.id for c in S.CASES])
def test_segment_reduce_path(case):
    inp = S.inputs(case)
    fwd, bwd, first = S.expected_paths(case)
    label = f"{case.id} [{fwd}/{bwd}/{first}]"
    got = run(case, inp)
    check_against_oracle(case, inp, got, label)
    # the same call with x and the cotangent one element off: scalar kernels, same arithmetic in the same order
    gu = run(case, inp, x_unaligned=True, g_unaligned=True)
    assert torch.equal(gu[0], got[0]), f"{label}: unaligned x_pool differs from the aligned run"
    assert torch.equal(gu[1], got[1]), f"{label}: unaligned dX differs from the aligned run"
    check_against_oracle(case, inp, gu, label + " unaligned")
    if case.twice:
        again = run(case, inp)
        for a, b, n in zip(got, again, ("x_pool", "dX", "dW")):
            assert (a is None and b is None) or torch.equal(a, b), f"{label}: {n} differs between two runs"


@pytest.mark.parametrize("dtype,op,weights", [("fp32", "sum", "w"), ("fp32", "max", "wgrad"), ("bf16", "mean", "w")])
def test_inverse_map_matches_search(dtype, op, weights):
    """N = 30 000 finds each node's first entry by binary search; padded with unselected nodes to N = 40 000 the
    backward builds the inverse map instead.  dX of the original nodes is bitwise the same, the padding rows zero."""
    case = S.topk(dtype, op, 128, 30000, 15001, extra=9, weights=weights)
    big = case._replace(N=40000)
    assert S.expected_paths(case)[2] == "search" and S.expected_paths(big)[2] == "map"
    inp = S.inputs(case)
    pad = dict(inp)
    pad["x"] = torch.cat([inp["x"], torch.randn(10000, 128, generator=torch.Generator().manual_seed(1)).to(inp["x"].dtype)])
    small, large = run(case, inp), run(big, pad)
    assert torch.equal(small[0], large[0])
    assert torch.equal(large[1][:30000], small[1]), "dX through the inverse map differs from dX through the search"
    assert not bool(large[1][30000:].any()), "padding rows of dX are not exactly zero"
    if small[2] is not None:
        assert torch.equal(small[2], large[2])
    check_against_oracle(big, pad, large, f"{case.id} padded")


# --------------------------------------------------------------------------- #
# consumers at row-kernel widths
# --------------------------------------------------------------------------- #
def _lift_oracle(x_pool, w, node, cl, g, N):
    xp, w64, g64 = x_pool.double(), w.double(), g.double()
    terms = xp[cl] * w64[:, None]
    out = torch.zeros(N, xp.size(1), dtype=torch.float64).index_add_(0, node, terms)
    out_t = torch.zeros_like(out).index_add_(0, node, terms.abs())
    gt = g64[node] * w64[:, None]
    dxp = torch.zeros_like(xp).index_add_(0, cl, gt)
    dxp_t = torch.zeros_like(xp).index_add_(0, cl, gt.abs())
    dw = (xp[cl] * g64[node]).sum(1)
    dw_t = (xp[cl] * g64[node]).abs().sum(1)
    return out, out_t, dxp, dxp_t, dw, dw_t


@pytest.mark.parametrize("dtype,F", [("fp32", 128), ("bf16", 256)])
def test_sparse_lift_row_kernel(dtype, F):
    """B200Lift with a TopK-style sparse S: one member per output row, a rows<8,1> call of the forward."""
    dt = S.DTYPES[dtype]
    N, K = 9003, 4001
    g_ = torch.Generator().manual_seed(F)
    node = torch.sort(torch.randperm(N, generator=g_)[:K]).values
    cl = torch.randperm(K, generator=g_)
    w = (torch.rand(K, generator=g_) + 0.5).to(dt)
    x_pool = torch.randn(K, F, generator=g_).to(dt)
    g = torch.randn(N, F, generator=g_).to(dt)
    ref = _lift_oracle(x_pool, w, node, cl, g, N)
    idx = torch.stack([node, cl]).to(DEV)

    def lift(g_unaligned):
        xp = x_pool.to(DEV).requires_grad_(True)
        wd = w.to(DEV).requires_grad_(True)
        so = T.SelectOutput(s=torch.sparse_coo_tensor(idx, wd, (N, K), is_coalesced=True))
        out = T.B200Lift()(xp, so)
        if g_unaligned:
            z = out.new_zeros(1)
            torch.cat([z, out.flatten()]).backward(torch.cat([z, g.to(DEV).flatten()]))
        else:
            out.backward(g.to(DEV))
        return out.detach().cpu(), xp.grad.cpu(), wd.grad.cpu()

    got = lift(False)
    for t, r, c, n in zip(got, ref[0::2], ref[1::2], ("x_lift", "dx_pool", "dW")):
        if dtype == "fp32":
            close_cw(t, r, c, f"lift {n}")
        else:
            close_bf16(t, r, f"lift bf16 {n}")
    gu = lift(True)
    assert torch.equal(gu[0], got[0]) and torch.equal(gu[1], got[1]), "unaligned cotangent changed the lift"
    if dtype == "fp32":
        close_cw(gu[2], ref[4], ref[5], "lift dW (unaligned cotangent)")
    else:
        close_bf16(gu[2], ref[4], "lift bf16 dW (unaligned cotangent)")


def test_unbatched_spmm_row_kernel():
    """unbatched.spmm (A x) at F = 128: forward and dX are segment-reduce forward calls at the row-kernel width."""
    N, E, F = 6001, 24007, 128
    g_ = torch.Generator().manual_seed(11)
    ei = torch.randint(0, N, (2, E), generator=g_)
    w = torch.rand(E, generator=g_) + 0.5
    x = torch.randn(N, F, generator=g_)
    g = torch.randn(N, F, generator=g_)
    row, col = ei[0], ei[1]
    x64, w64, g64 = x.double(), w.double(), g.double()
    t = x64[col] * w64[:, None]
    ref_out = torch.zeros(N, F, dtype=torch.float64).index_add_(0, row, t)
    ref_out_t = torch.zeros(N, F, dtype=torch.float64).index_add_(0, row, t.abs())
    tg = g64[row] * w64[:, None]
    ref_dx = torch.zeros(N, F, dtype=torch.float64).index_add_(0, col, tg)
    ref_dx_t = torch.zeros(N, F, dtype=torch.float64).index_add_(0, col, tg.abs())
    ref_dw = (g64[row] * x64[col]).sum(1)
    ref_dw_t = (g64[row] * x64[col]).abs().sum(1)

    def spmm(unal):
        xd = unaligned(x) if unal else x.to(DEV)
        xd.requires_grad_(True)
        wd = w.to(DEV).requires_grad_(True)
        out = U.spmm(ei.to(DEV), wd, xd, N)
        if unal:
            z = out.new_zeros(1)
            torch.cat([z, out.flatten()]).backward(torch.cat([z, g.to(DEV).flatten()]))
        else:
            out.backward(g.to(DEV))
        return out.detach().cpu(), xd.grad.cpu(), wd.grad.cpu()

    got = spmm(False)
    close_cw(got[0], ref_out, ref_out_t, "spmm out")
    close_cw(got[1], ref_dx, ref_dx_t, "spmm dX")
    close_cw(got[2], ref_dw, ref_dw_t, "spmm dW")
    gu = spmm(True)
    assert torch.equal(gu[0], got[0]) and torch.equal(gu[1], got[1]), "unaligned x / cotangent changed the SpMM"
    close_cw(gu[2], ref_dw, ref_dw_t, "spmm dW (unaligned)")


@pytest.mark.parametrize("op", S.OPS)
def test_readout_row_kernel(op):
    """B200Reduce(op)(x, None, batch=...) over four graphs of about 2000 nodes at F = 128."""
    sizes = [1999, 2003, 2011, 1987]
    N, F = sum(sizes), 128
    batch = torch.repeat_interleave(torch.arange(4), torch.tensor(sizes))
    case = S.Case("fp32", op, F, N, 4, "readout", N, "none")
    g_ = torch.Generator().manual_seed(5)
    x = torch.randn(N, F, generator=g_)
    if op in ("max", "min"):
        x[1000] = x[10]  # an exact tie inside graph 0
    g = torch.randn(4, F, generator=g_)
    inp = {"x": x, "w": None, "node": torch.arange(N), "cluster": batch, "g": g}

    def readout(unal):
        xd = unaligned(x) if unal else x.to(DEV)
        xd.requires_grad_(True)
        out, gb = T.B200Reduce(op)(xd, None, batch=batch.to(DEV))
        assert torch.equal(gb.cpu(), torch.arange(4))
        if unal:
            z = out.new_zeros(1)
            torch.cat([z, out.flatten()]).backward(torch.cat([z, g.to(DEV).flatten()]))
        else:
            out.backward(g.to(DEV))
        return out.detach().cpu(), xd.grad.cpu(), None

    got = readout(False)
    check_against_oracle(case, inp, got, f"readout {op}")
    gu = readout(True)
    assert torch.equal(gu[0], got[0]) and torch.equal(gu[1], got[1]), "unaligned x / cotangent changed the readout"


# --------------------------------------------------------------------------- #
# dense poolers, unaligned inputs and cotangents (the fallbacks behind the alignment guards)
# --------------------------------------------------------------------------- #
_DENSE = [(fam, shape, bf16) for fam in ("mincut", "diff", "dmon") for bf16 in (False, True)
          for shape in ((3, 256, 64, 128), (5, 200, 48, 100))]
_WHICH = ("x", "adj", "s", "g_x_pool", "g_adj_pool", "g_losses")


@pytest.mark.parametrize("family,shape,bf16", _DENSE,
                         ids=[f"{f}-{'x'.join(map(str, s))}-{'bf16' if b else 'fp32'}" for f, s, b in _DENSE])
def test_dense_pool_unaligned(family, shape, bf16):
    """x, adj and s one element off a 16-byte boundary, one at a time; then the cotangents of x_pool, adj_pool and the
    losses.  The combined gradient of every run is held to the per-graph bars of ``grad_sources``."""
    case = G.Case(family, shape, 0, bf16)
    x, a, s, n, gx, ga = G.inputs(case)
    ref = G.reference_grads(case, case.sources)
    dt = torch.bfloat16 if bf16 else torch.float32
    gl = torch.zeros(4)
    for src, idx in G.FAMILIES[family][1].items():
        gl[idx] = G.LOSS_COEF[src]
    for which in _WHICH:
        leaves = {k: t.to(DEV, dt) for k, t in (("x", x), ("adj", a), ("s", s))}
        if which in leaves:
            leaves[which] = unaligned(leaves[which])
        for t in leaves.values():
            t.requires_grad_(True)
        gn = n.float().to(DEV) if family == "dmon" else None
        xp, ap, losses = F_.dense_pool(leaves["x"], leaves["adj"], leaves["s"], loss_kind=case.loss_kind,
                                       ent_div=case.ent_div, graph_nodes=gn, **case.kw)
        outs = [xp, ap, losses]
        cots = [gx.to(DEV, dt), ga.to(DEV, dt), gl.to(DEV)]
        k = _WHICH.index(which) - 3
        if k >= 0:  # route this output's cotangent through a concatenation: one element off
            z = outs[k].new_zeros(1)
            outs[k] = torch.cat([z, outs[k].flatten()])
            cots[k] = torch.cat([z, cots[k].flatten()])
        torch.autograd.backward(outs, cots)
        torch.cuda.synchronize()
        got = {"dS": leaves["s"].grad, "dX": leaves["x"].grad, "dA": leaves["adj"].grad}
        for key, t in got.items():
            assert bool(torch.isfinite(t.float()).all()), f"{which} unaligned: {key} not finite"
        G.check_grads(case, got, ref, f"{family} {shape} {'bf16' if bf16 else 'fp32'} {which} unaligned")
