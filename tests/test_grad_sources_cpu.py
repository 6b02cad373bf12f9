"""The per-source gradient harness of ``grad_sources.py`` on CPU: its fp32 bar is not tighter than fp32 arithmetic
allows (calibration), and it rejects small defects that a bound scaled by the combined gradient accepts (sensitivity)."""
import math

import pytest
import torch

import grad_sources as G

FP32_CASES = sorted({c for _, _, c in G.path_cases() if not c.bf16})


@pytest.mark.parametrize("case", FP32_CASES, ids=lambda c: f"{c.family}-{'x'.join(map(str, c.shape))}-flags{c.flags}")
def test_float32_oracle_passes_fp32_bar(case):
    """A float32 evaluation of the reference passes the fp32 bar against the float64 one, for every source."""
    for src in case.sources:
        got = G.reference_grads(case, (src,), torch.float32)
        G.check_grads(case, got, G.oracle(case, src), f"float32 oracle {src}")


def _rejects(case, got, ref, label):
    with pytest.raises(AssertionError):
        G.check_grads(case, got, ref, label)


SENS_CASES = [G.Case("mincut", (5, 200, 48, 100), 0), G.Case("diff", (4, 99, 16, 33), 1),
              G.Case("dmon", (5, 256, 64, 128), 0)]


@pytest.mark.parametrize("case", SENS_CASES, ids=lambda c: c.family)
def test_rejects_relative_error_in_one_source_of_one_graph(case):
    for src in case.sources:
        ref = G.oracle(case, src)
        for k in G.GRADS:
            for b in range(case.shape[0]):
                if not bool(ref[k][b].any()):
                    continue
                got = dict(ref)
                got[k] = ref[k].clone()
                got[k][b] *= 1 + 1e-3
                _rejects(case, got, ref, f"{src} {k} graph {b}")


def test_rejects_graph_using_graph0_cut_coefficient():
    """MinCut's cut loss has a coefficient per graph (1 / den_b, num_b / den_b^2); graph b >= 1 using graph 0's is
    rejected, while the same formula with each graph's own coefficients reproduces the oracle."""
    case = G.Case("mincut", (5, 200, 48, 100), 0)
    x, a, s, n, _, _ = G.inputs(case)
    a, s = a.double(), s.double()
    B = s.size(0)
    num = torch.einsum("bnk,bnm,bmk->b", s, a, s)
    deg = a.sum(-1)
    den = torch.einsum("bnk,bn,bnk->b", s, deg, s) + G.EPS
    dnum = (a + a.transpose(1, 2)) @ s
    dden = 2 * deg[..., None] * s
    coef = G.LOSS_COEF["cut"] / B

    def ds(num, den):
        return coef * (-dnum / den[:, None, None] + (num / den**2)[:, None, None] * dden)

    ref = G.oracle(case, "cut")
    G.check_grads(case, {"dS": ds(num, den)}, ref, "own coefficients")
    one = torch.zeros(B, dtype=torch.long)
    _rejects(case, {"dS": ds(num[one], den[one])}, ref, "graph 0's coefficients")


def test_rejects_dmon_cluster_term_dropped():
    """The cluster loss reaches dS as v_k = (g_c / B) sqrt(K) e_k / (n_b ||e||) on every row (e = S^T 1): the model
    matches the oracle and a dS without it is rejected."""
    case = G.Case("dmon", (5, 200, 48, 100), 1)
    x, a, s, n, _, _ = G.inputs(case)
    B, N, K, _ = case.shape
    e = s.double().sum(1)
    v = G.LOSS_COEF["cluster"] / B * math.sqrt(K) * e / (n.double()[:, None] * e.norm(dim=1, keepdim=True))
    ref = G.oracle(case, "cluster")
    G.check_grads(case, {"dS": v[:, None, :].expand(B, N, K)}, ref, "v_k")
    _rejects(case, {"dS": ref["dS"] - v[:, None, :]}, ref, "v_k dropped")


def test_rejects_entropy_without_ratio_term():
    """d/ds of -s log(s + eps) is -log(s + eps) - s / (s + eps); dropping the second term is rejected."""
    case = G.Case("diff", (5, 200, 48, 100), 0)
    s = G.inputs(case)[2].double()
    c = G.LOSS_COEF["entropy"] / case.ent_div
    ref = G.oracle(case, "entropy")
    G.check_grads(case, {"dS": c * (-torch.log(s + G.EPS) - s / (s + G.EPS))}, ref, "entropy model")
    _rejects(case, {"dS": c * -torch.log(s + G.EPS)}, ref, "without s / (s + eps)")


def test_zero_reference_graph_uses_batch_scale():
    ref = torch.zeros(3, 4, 4)
    ref[0] = 1.0
    G.assert_per_graph(ref + 0.5e-4 * (torch.arange(3) == 2).double()[:, None, None], ref, 1e-4, "within")
    with pytest.raises(AssertionError):
        G.assert_per_graph(ref + 2e-4 * (torch.arange(3) == 2).double()[:, None, None], ref, 1e-4, "beyond")
    with pytest.raises(AssertionError):
        G.assert_per_graph(ref * float("nan"), ref, 1e-4, "nan")
    # a gradient that is zero for the whole batch must come out exactly zero
    zero = torch.zeros(3, 4, 4)
    G.assert_per_graph(zero, zero, 1e-4, "zero")
    with pytest.raises(AssertionError):
        G.assert_per_graph(zero + 1e-30, zero, 1e-4, "not zero")


def test_hetero_batch_has_the_promised_structure():
    x, a, s, n = G.hetero_batch(5, 64, 8, 16)
    assert not torch.equal(a[0], a[0].t()) and all(torch.equal(a[b], a[b].t()) for b in range(1, 5))
    assert float(a[1].max()) > 4.0 and float(a[0].max()) == 1.0
    assert len(set(n.tolist())) > 1
    for b in range(5):
        assert not bool(s[b, n[b]:].any()) and not bool(x[b, n[b]:].any()) and not bool(a[b, n[b]:].any())
    last = s[-1, :n[-1]]
    assert bool(((last == 0) | (last == 1)).all()) and not bool(last[:, -1].any())
