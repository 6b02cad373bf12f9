"""CPU: the Asymmetric Cheeger Cut oracle (hand values, the closed-form gradients the kernels implement, the tie rule of
the quantile), the wiring of ``acc_pool`` / ``patch_pooler`` with the device calls replaced by the oracle, and the
shape propagation of the new ops.  No kernels are launched here."""
import pytest
import torch

import acc_oracle as A
import dropin_harness as H
from oracle import ref_path as R


def _two_triangles(w_cross=0.0):
    a = torch.zeros(1, 6, 6, dtype=torch.float64)
    for comp in ([0, 1, 2], [3, 4, 5]):
        for i in comp:
            for j in comp:
                if i != j:
                    a[0, i, j] = 1.0
    a[0, 2, 3] = a[0, 3, 2] = w_cross
    return a


def _split():
    s = torch.zeros(1, 6, 2, dtype=torch.float64)
    s[0, :3, 0] = 1.0
    s[0, 3:, 1] = 1.0
    return s


def test_hand_values():
    a, s = _two_triangles(), _split()
    assert A.totvar_loss(s, a).item() == pytest.approx(0.0, abs=1e-12)
    assert A.asym_norm_loss(s).item() == pytest.approx(0.0, abs=1e-12)
    one = torch.zeros(1, 6, 2, dtype=torch.float64)
    one[0, :, 0] = 1.0
    assert A.asym_norm_loss(one).item() == pytest.approx(1.0, abs=1e-12)
    # one symmetric edge of weight w across the split: 2 w ||e_0 - e_1||_1 / (2 nnz), nnz = 12 + 2 directions
    assert A.totvar_loss(s, _two_triangles(0.5)).item() == pytest.approx(1.0 / 14.0, abs=1e-12)


def test_edgeless_graph_gives_nan():
    s = torch.softmax(torch.randn(2, 5, 3, dtype=torch.float64), -1)
    a = torch.zeros(2, 5, 5, dtype=torch.float64)
    a[0, 0, 1] = 1.0
    loss = A.totvar_loss(s, a, "sum")
    assert torch.isnan(loss)


def test_quantile_follows_the_stable_sort():
    s = torch.tensor([[[.5, .1], [.2, .2], [.2, .3], [.2, .9], [.1, .4]]], dtype=torch.float64)
    val, node = A.quantile(s)  # N // K = 2
    assert node[0, 0].item() == 2 and val[0, 0].item() == 0.2  # the rank rule, not the lowest tied index
    assert node[0, 1].item() == 2 and val[0, 1].item() == 0.3


def closed_form(s, a, g_tv, g_bal):
    """dS, dA of g_tv * totvar + g_bal * balance as the kernels compute them."""
    B, N, K = s.shape
    c = g_tv / (2 * torch.count_nonzero(a, dim=(1, 2)).to(s.dtype) * B)
    e = g_bal / (N * (K - 1) * B)
    diff = s[:, :, None, :] - s[:, None, :, :]  # [B, i, j, k]
    ds = c[:, None, None] * torch.einsum("bij,bijk->bik", a + a.transpose(1, 2), torch.sign(diff))
    q, qi = A.quantile(s)
    fp = torch.where(s - q[:, None, :] >= 0, float(K - 1), -1.0).to(s.dtype)
    ds = ds - e * fp
    ds = ds.scatter_add(1, qi[:, None, :], e * fp.sum(1, keepdim=True))
    da = c[:, None, None] * diff.abs().sum(-1)
    return ds, da


def _masked_batch(B=3, N=12, K=3, seed=0):
    g = torch.Generator().manual_seed(seed)
    n = torch.tensor([N, N - 4, 3][:B])
    mask = torch.arange(N)[None, :] < n[:, None]
    a = torch.rand(B, N, N, generator=g, dtype=torch.float64)
    a = (a < 0.4) * (a + a.transpose(1, 2)) * (mask[:, :, None] & mask[:, None, :])
    s = torch.softmax(torch.randn(B, N, K, generator=g, dtype=torch.float64), -1) * mask[..., None]
    return a, s


def _tied_case():
    s = torch.tensor([[[.5, .1], [.2, .2], [.2, .3], [.2, .9], [.1, .4]]], dtype=torch.float64)
    a = torch.tensor([[[0, 1, 0, 1, 0], [1, 0, 1, 0, 0], [0, 1, 0, 2, 1], [1, 0, 2, 0, 0], [0, 0, 1, 0, 1]]],
                     dtype=torch.float64)
    return a, s


@pytest.mark.parametrize("case", ["ragged0", "ragged1", "ties", "bf16_ties"])
def test_closed_form_gradients_match_autograd(case):
    """Ragged batches (padded zero rows tie in both losses and the quantile can land among them), the tie column of
    the rank rule, and bf16-rounded softmax rows (many exact ties) in float64."""
    if case == "ties":
        a, s = _tied_case()
    elif case == "bf16_ties":
        a, s = _masked_batch(B=2, N=40, K=4, seed=5)
        s = s.to(torch.bfloat16).to(torch.float64)
    else:
        a, s = _masked_batch(seed=int(case[-1]))
    g_tv, g_bal = 0.7, -1.3
    a_, s_ = a.clone().requires_grad_(), s.clone().requires_grad_()
    (g_tv * A.totvar_loss(s_, a_) + g_bal * A.asym_norm_loss(s_)).backward()
    ds, da = closed_form(s, a, g_tv, g_bal)
    torch.testing.assert_close(s_.grad, ds, rtol=1e-12, atol=1e-14)
    torch.testing.assert_close(a_.grad, da, rtol=1e-12, atol=1e-14)


class AsymCheegerCutPooling(H._DenseBase):  # the restated attributes of AsymCheegerCutPooling
    totvar_coeff, balance_coeff = 0.6, 1.7


def test_acc_pool_and_patched_pooler_wiring(monkeypatch):
    """The pooler-level code with the two device calls replaced by the oracle: coefficients, loss keys and connector
    flags reach the right places, and the losses come from the raw adjacency."""
    import tgp_b200 as T
    from tgp_b200 import poolers as P

    def dense_pool(x, adj, s, *, loss_kind, **flags):
        assert loss_kind == T.functional.LOSS_NONE
        return s.transpose(1, 2) @ x, R.postprocess_adj_pool_dense(R.dense_connect(adj, s), **flags), None

    monkeypatch.setattr(P.F_, "dense_pool", dense_pool)
    monkeypatch.setattr(P.F_, "acc_losses", lambda adj, s: torch.stack([A.totvar_loss(s, adj), A.asym_norm_loss(s)]))
    a, s = _masked_batch(B=3, N=12, K=3, seed=2)
    x = torch.randn(3, 12, 5, dtype=torch.float64)
    flags = dict(remove_self_loops=True, degree_norm=True, adj_transpose=False, edge_weight_norm=True)
    pooler = AsymCheegerCutPooling(selector=lambda x, mask: R.OracleSelectOutput(s=s), reducer=H.BaseReduce(),
                                   connector=H.DenseConnect(**flags))
    T.patch_pooler(pooler)
    out = pooler(x=x, adj=a)
    xp, ap, loss = A.acc_pool(x, a, s, 0.6, 1.7, **flags)
    assert set(out.loss) == {"total_variation_loss", "balance_loss"} == set(loss)
    for k in loss:
        torch.testing.assert_close(out.loss[k], loss[k], rtol=1e-12, atol=0.0)
    torch.testing.assert_close(out.x, xp)
    torch.testing.assert_close(out.edge_index, ap)


def test_acc_ops_fake_tensor_shapes():
    from torch._subclasses.fake_tensor import FakeTensorMode

    import tgp_b200  # noqa: F401  (registers the ops and their fake kernels)
    from tgp_b200 import ops

    assert {"acc_losses", "acc_losses_bwd"} <= set(ops.OP_NAMES)
    with FakeTensorMode():
        s = torch.empty(4, 32, 8, device="cuda", dtype=torch.bfloat16)
        a = torch.empty(4, 32, 32, device="cuda", dtype=torch.bfloat16)
        losses, quant, saved = torch.ops.tgp_b200.acc_losses(a, s)
        assert losses.shape == (2,) and losses.dtype == torch.float32
        assert quant.shape == (4, 8) and quant.dtype == torch.bfloat16 and saved.dtype == torch.uint8
        ga, gs = torch.ops.tgp_b200.acc_losses_bwd(a, s, saved, losses, True)
        assert ga.shape == a.shape and gs.shape == s.shape
        ga, _ = torch.ops.tgp_b200.acc_losses_bwd(a, s, saved, losses, False)
        assert ga.numel() == 0


def test_acc_pool_is_exported_and_cpu_raises():
    import tgp_b200 as T

    assert "acc_pool" in T.__all__
    with pytest.raises(RuntimeError, match="CUDA"):
        T.acc_pool(torch.randn(1, 4, 2), torch.rand(1, 4, 4), torch.rand(1, 4, 2))
    with pytest.raises(RuntimeError, match="CUDA"):
        T.functional.acc_losses(torch.rand(1, 4, 4), torch.rand(1, 4, 2))
