"""B200: every launch path of the sparse connect against the float64 oracle, unpadded, padded and unaligned.

Cases, launch rules and oracle: ``sparse_connect_cases``.  Bars (DESIGN.md section 2):

* ``edge_index``, edge order and count bit-exact; max / min coalesced weights exactly the float32 extreme;
* coalesced sum / mean / mul without normalisation: ``|err| <= (L + 1) 2^-24 sum|terms|`` per output edge, L its
  number of members.  A sequential float32 sum of L terms errs by at most ``(L - 1) u sum|terms|`` (u = 2^-24, first
  order), the mean's division and the product's L - 1 roundings add at most ``u`` per operation, and the whole-block
  runs of ``k_hub_long_runs`` (double partials, one rounding) stay below ``u sum|terms|``;
* normalised weights and every weight gradient: ``|err| <= 1e-5 sum|terms|`` component-wise, no global atol.  The
  max-weight normalisation's arg is checked through it: a wrong tied edge is off by ``acc / m^2``;
* padded calls (``sparse_connect_padded``, capacity launches, device-side count): the first ``count`` entries and the
  weight gradient bitwise equal to the unpadded call;
* unaligned inputs: ``edge_index`` and ``edge_weight`` one element off a 16-byte boundary (the scalar branch of
  ``k_fine_row_spans``) give bitwise the same outputs and gradient;
* the C4- and C5-shaped cases give the same bits on a second run.
"""
import functools

import pytest
import torch

import sparse_connect_cases as S
import tgp_b200 as T
from tgp_b200 import functional as F_

pytestmark = pytest.mark.gpu
DEV = "cuda"
U = 2.0 ** -24


@functools.lru_cache(maxsize=None)
def _data(case):
    inp = S.inputs(case)
    return inp, S.oracle(case, inp)


def _select(case, inp):
    if case.branch == "kept":
        node = inp["node_index"].to(DEV)
        return T.SelectOutput(node_index=node, num_nodes=case.N, cluster_index=torch.arange(node.numel(), device=DEV),
                              num_supernodes=node.numel())
    return T.SelectOutput(cluster_index=inp["cluster"].to(DEV), num_nodes=case.N, num_supernodes=case.K)


def _on_device(t, unaligned):
    if not unaligned:
        return t.to(DEV)
    buf = torch.zeros(t.numel() + 1, dtype=t.dtype, device=DEV)
    buf[1:].copy_(t.flatten())
    v = buf[1:].view(t.shape)
    assert v.is_contiguous() and v.data_ptr() % 16 != 0
    return v


def run(case, inp, ref, padded=False, unaligned=False):
    """Device (edge_index, weights, weight gradient) of one call, on the CPU; padded calls cut to their count."""
    ei = _on_device(inp["edge_index"], unaligned)
    w = leaf = None
    if inp["w"] is not None:
        if unaligned:
            leaf = torch.zeros(inp["w"].numel() + 1, device=DEV)
            leaf[1:].copy_(inp["w"])
            leaf.requires_grad_(True)
            w = leaf[1:]
            assert w.data_ptr() % 16 != 0
        else:
            leaf = w = inp["w"].to(DEV).requires_grad_(True)
    so = _select(case, inp)
    bp = inp["batch_pooled"].to(DEV)
    if padded:
        csr = F_.csr_of(so) if case.branch == "cluster" else None
        eo, wo, count = F_.sparse_connect_padded(
            ei, w, node_index=so.node_index, cluster_index=so.cluster_index, num_nodes=case.N,
            num_supernodes=so.num_supernodes, remove_self_loops=case.rsl, reduce_op=case.op,
            edge_weight_norm=case.ewn, batch_pooled=bp, degree_norm=case.dn, num_graphs=case.G, csr=csr)
        n = int(count.item())
        eo = eo[:, :n]
    else:
        eo, wo = T.B200SparseConnect(case.op, case.rsl, case.ewn, case.dn)(ei, so, edge_weight=w, batch_pooled=bp)
        n = eo.size(1)
    dw = None
    if wo is not None and leaf is not None:
        g = ref["g"].float().to(DEV)
        if padded:
            g = torch.cat([g, torch.zeros(wo.numel() - n, device=DEV)])
        (wo * g).sum().backward()
        dw = leaf.grad[1:] if unaligned else leaf.grad
        dw = dw.cpu()
    torch.cuda.synchronize()
    return eo.cpu(), (None if wo is None else wo.detach()[:n].cpu()), dw


def close_cw(got, ref, cond, name, rtol):
    err = (got.double() - ref).abs()
    bound = rtol * cond + 1e-30
    bad = ~(err <= bound)
    assert not bool(bad.any()), f"{name}: {int(bad.sum())} of {err.numel()} elements beyond the bound, worst ratio " \
                                f"{float(torch.nan_to_num(err / bound, nan=float('inf')).max()):.3f}"


def check(case, ref, got, label):
    eo, wo, dw = got
    assert eo.shape == ref["edge_index"].shape, f"{label}: {eo.size(1)} edges, oracle {ref['edge_index'].size(1)}"
    assert torch.equal(eo, ref["edge_index"]), f"{label}: edge_index / order differ from the oracle"
    if ref["w"] is None:
        assert wo is None, f"{label}: weights where the reference has none"
        return
    assert wo is not None and wo.numel() == ref["w"].numel()
    if case.dn or case.ewn:
        close_cw(wo, ref["w"], ref["w_terms"], f"{label} normalised weights", 1e-5)
    elif case.op in ("max", "min") and case.branch == "cluster":
        assert torch.equal(wo, ref["w32"]), f"{label}: {case.op} weights are not the float32 extreme"
    else:
        L = ref["run_len"].double()
        close_cw(wo, ref["w"], (L + 1) * U * ref["w_terms"], f"{label} coalesced weights", 1.0)
    if ref["dw"] is not None:
        assert dw is not None, f"{label}: no weight gradient"
        close_cw(dw, ref["dw"], ref["dw_terms"], f"{label} weight gradient", 1e-5)


@pytest.mark.parametrize("case", S.CASES, ids=[c.id for c in S.CASES])
def test_sparse_connect_path(case):
    inp, ref = _data(case)
    paths = S.expected_paths(case, inp, ref["edge_index"].size(1))
    label = f"{case.id} {paths}"
    got = run(case, inp, ref)
    check(case, ref, got, label)
    pad = run(case, inp, ref, padded=True)
    for a, b, n in zip(got, pad, ("edge_index", "weights", "weight gradient")):
        assert (a is None and b is None) or torch.equal(a, b), f"{label}: padded {n} differs from the unpadded call"
    un = run(case, inp, ref, unaligned=True)
    for a, b, n in zip(got, un, ("edge_index", "weights", "weight gradient")):
        assert (a is None and b is None) or torch.equal(a, b), f"{label}: unaligned {n} differs from the aligned call"
    if case.twice:
        again = run(case, inp, ref)
        for a, b, n in zip(got, again, ("edge_index", "weights", "weight gradient")):
            assert (a is None and b is None) or torch.equal(a, b), f"{label}: {n} differs between two runs"
