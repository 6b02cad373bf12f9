"""CPU checks of the segment-reduce case table (``segment_reduce_cases``): every launch path of the forward and the
backward is reached by some case for every dtype and op, every launch rule is run on both sides of its threshold, and
the float64 oracle reproduces the reference's own reduce and autograd (the even split of the gradient among ties
included).  ``pytest -rP`` prints which cases reach each path."""
import itertools

import pytest
import torch

import segment_reduce_cases as S
from oracle import ref_path as R

_PATHS = {c: S.expected_paths(c) for c in S.CASES}


def _combos():
    out = []
    for dt, op in itertools.product(S.DTYPES, S.OPS):
        out += [("fwd", p, dt, op) for p in S.FWD_PATHS]
        out += [("bwd", p, dt, op) for p in S.BWD_PATHS if not (p == "rows8" and op in ("max", "min"))]
        out += [("first", p, dt, op) for p in S.FIRST_PATHS]
    return out


def _reaching(kind, path, dt, op):
    k = {"fwd": 0, "bwd": 1, "first": 2}[kind]
    return [c for c, p in _PATHS.items() if p[k] == path and c.dtype == dt and c.op == op]


@pytest.mark.parametrize("kind,path,dt,op", _combos(), ids=["-".join(c) for c in _combos()])
def test_launch_path_reached(kind, path, dt, op):
    cases = _reaching(kind, path, dt, op)
    print(f"{kind} {path} {dt} {op}: " + ", ".join(c.id for c in cases))
    assert cases, f"no case runs the {kind} path {path} for {dt} {op}"


def test_thresholds_on_both_sides():
    for dt in S.DTYPES:
        W = S.VEC[dt]
        cs = [c for c in S.CASES if c.dtype == dt]
        Fs = {c.F for c in cs}
        assert any(F % W for F in Fs) and any(F % W == 0 for F in Fs), "F a multiple of the vector width and not"
        assert 16 * W in Fs and 17 * W in Fs, "16 chunks (generic kernel) and 17 (row kernels)"
        assert any(F % W == 0 and F > 32 * W and F % (32 * W) for F in Fs), "several passes, the last partial"
        rows = [c for c in cs if _PATHS[c][0] in ("rows41", "rows81")]
        assert any(c.nnz == c.K + c.K // 4 for c in rows), "nnz == K + K/4 (rows<8,1>)"
        assert any(c.nnz == c.K + c.K // 4 + 1 for c in rows), "nnz == K + K/4 + 1 (rows<4,2>)"
        assert any(c.K % 8 and c.N % 8 for c in rows), "partial last warp of the row kernels"
        assert any(c.N == S.SEARCH_LIMIT and _PATHS[c][2] == "search" for c in cs)
        assert any(c.N == S.SEARCH_LIMIT + 1 and _PATHS[c][2] == "map" for c in cs)
        assert any(c.N < S.SEARCH_LIMIT and c.nnz == S.SEARCH_LIMIT and _PATHS[c][2] == "search" for c in cs)
        assert any(c.N < S.SEARCH_LIMIT and c.nnz == S.SEARCH_LIMIT + 1 and _PATHS[c][2] == "map" for c in cs)
        for w in ("none", "w", "wgrad"):
            assert any(c.weights == w for c in cs), w
        for lay in ("topk", "hard", "readout", "soft"):
            assert any(c.layout == lay for c in cs), lay


def test_unaligned_inputs_take_the_scalar_kernels():
    for c in S.CASES:
        assert S.expected_paths(c, aligned=False)[:2] == ("scalar", "scalar")


@pytest.mark.parametrize("layout", ["hard", "readout", "soft", "topk"])
def test_layouts(layout):
    c = next(c for c in S.CASES if c.layout == layout)
    inp = S.inputs(c)
    node, cl = inp["node"], inp["cluster"]
    assert node.numel() == cl.numel() == c.nnz
    assert bool((node[1:] >= node[:-1]).all()), "node_index ascending"
    assert int(cl.min()) >= 0 and int(cl.max()) < c.K
    counts = torch.bincount(cl, minlength=c.K)
    if layout == "hard":
        assert not bool(counts[-3:].any()), "last clusters empty"
    if layout == "readout":
        assert int(counts.max()) > 2000
    if layout == "soft":
        assert torch.unique(node * c.K + cl).numel() == c.nnz, "distinct (node, cluster) pairs"
        assert int(torch.bincount(node).max()) > 1, "nodes in several clusters"
    if layout == "topk":
        assert torch.unique(node).numel() == c.nnz < c.N and bool(counts.all())


def _small_cases():
    out = []
    for op in S.OPS:
        out.append(S.hard("fp32", op, 5, 61, 13, weights="wgrad"))
        out.append(S.topk("fp32", op, 8, 61, 13, extra=4, weights="wgrad"))
        out.append(S.soft("fp32", op, 4, 29, 11, 70, weights="wgrad"))
        out.append(S.readout("fp32", op, 6, 50, 3))
    return out


@pytest.mark.parametrize("case", _small_cases(), ids=[c.id for c in _small_cases()])
def test_oracle_matches_reference_autograd(case):
    """float64 reference (R.base_reduce / R.aggr_reduce + autograd) against the oracle; max / min cases hold exact ties,
    whose gradient the reference splits evenly."""
    inp = S.inputs(case)
    x, w, node, cl, g = (inp[k] for k in ("x", "w", "node", "cluster", "g"))
    ref = S.oracle(case, x, w, node, cl, g)
    x64 = x.double().requires_grad_(True)
    w64 = None if w is None else w.double().requires_grad_(True)
    vals = w64 if w64 is not None else torch.ones(case.nnz, dtype=torch.float64)
    # (node, cluster) pairs are already in coalesced order: the COO takes them as they are
    so = R.OracleSelectOutput(s=torch.sparse_coo_tensor(torch.stack([node, cl]), vals, (case.N, case.K),
                                                        is_coalesced=True))
    out = R.base_reduce(x64, so)[0] if case.op == "sum" else R.aggr_reduce(x64, so, case.op)[0]
    (out * g.double()).sum().backward()
    kw = dict(rtol=1e-12, atol=1e-12)
    if case.op in ("sum", "mean"):
        torch.testing.assert_close(ref["out"], out.detach(), **kw)
    else:  # the extreme of the float32 products, as the reference computes it on float32 inputs
        assert torch.equal(ref["out"], S.reference_fp32_forward(case, x, w, node, cl).double())
        torch.testing.assert_close(ref["out"], out.detach(), rtol=1e-7, atol=0.0)
    torch.testing.assert_close(ref["dx"], x64.grad, **kw)
    if w64 is not None:
        torch.testing.assert_close(ref["dw"], w64.grad, **kw)
    assert bool((ref["out_terms"] >= ref["out"].abs() - 1e-12).all())
    if case.op in ("max", "min") and case.layout != "readout":
        _, p = S._products(x, w, node, "fp32")
        ext = ref["out"][cl]
        assert bool(((p == ext).sum(0) > 0).any())
        hit = torch.zeros(case.K, case.F, dtype=torch.float64).index_add_(0, cl, (p == ext).double())
        assert bool((hit > 1).any()), "the case holds exact ties"


@pytest.mark.parametrize("op", ["max", "min"])
def test_oracle_bf16_ties_after_rounding(op):
    """bf16: the reference multiplies in bf16 and compares the rounded products; the oracle does the same, so products
    that differ in float32 but round to the same bf16 share the gradient."""
    case = S.topk("bf16", op, 8, 97, 23, extra=20, weights="wgrad")
    inp = S.inputs(case)
    x, w, node, cl, g = (inp[k] for k in ("x", "w", "node", "cluster", "g"))
    p, pr = S._products(x, w, node, "bf16")
    ext = torch.zeros(case.K, case.F, dtype=torch.float64).scatter_reduce_(
        0, cl[:, None].expand(-1, case.F), pr, "amax" if op == "max" else "amin", include_self=False)
    rounding_tie = (pr == ext[cl]) & (p != ext[cl])
    assert bool(rounding_tie.any()), "the case holds ties that appear only after rounding"
    ref = S.oracle(case, x, w, node, cl, g)
    xb, wb = x.clone().requires_grad_(True), w.clone().requires_grad_(True)
    so = R.OracleSelectOutput(s=torch.sparse_coo_tensor(torch.stack([node, cl]), wb, (case.N, case.K), is_coalesced=True))
    out = R.aggr_reduce(xb, so, op)[0]
    (out.float() * g.float()).sum().backward()
    assert torch.equal(out.float().double(), ref["out"].float().bfloat16().double())
    torch.testing.assert_close(xb.grad.double(), ref["dx"], rtol=2e-2, atol=2e-2 * float(ref["dx"].abs().max()))
    torch.testing.assert_close(wb.grad.double(), ref["dw"], rtol=2e-2, atol=2e-2 * float(ref["dw"].abs().max()))
