"""CPU: the HOSC oracle (hand values, a float64 gradcheck, the closed-form gradients the kernels implement), the wiring
of ``hosc_pool`` / ``patch_pooler`` with the device calls replaced by the oracle, and the shape propagation of the new
ops.  No kernels are launched here."""
import math

import pytest
import torch

import dropin_harness as H
import hosc_oracle as O
from oracle import ref_path as R


def _two_triangles():
    a = torch.zeros(1, 6, 6, dtype=torch.float64)
    for comp in ([0, 1, 2], [3, 4, 5]):
        for i in comp:
            for j in comp:
                if i != j:
                    a[0, i, j] = 1.0
    s = torch.zeros(1, 6, 2, dtype=torch.float64)
    s[0, :3, 0] = 1.0
    s[0, 3:, 1] = 1.0
    return a, s


def _four_cycle():
    a = torch.zeros(1, 4, 4, dtype=torch.float64)
    for i in range(4):
        a[0, i, (i + 1) % 4] = a[0, (i + 1) % 4, i] = 1.0
    s = torch.zeros(1, 4, 2, dtype=torch.float64)
    s[0, :2, 0] = 1.0
    s[0, 2:, 1] = 1.0
    return a, s


def test_hand_values():
    a, s = _two_triangles()
    assert torch.equal(O.motif_adjacency(a), a)  # every edge lies on exactly one triangle
    l1, l2, o = O.hosc_losses(a, s, eps=0.0).tolist()
    assert l1 == pytest.approx(-1.0, abs=1e-12) and l2 == pytest.approx(-1.0, abs=1e-12)
    assert o == pytest.approx(0.0, abs=1e-12)
    a, s = _four_cycle()
    assert torch.count_nonzero(O.motif_adjacency(a)) == 0  # no triangle
    l1, l2, _ = O.hosc_losses(a, s).tolist()
    assert l1 == pytest.approx(-0.5, abs=1e-8)
    assert l2 == 0.0  # 0 / eps: no NaN


def _masked_batch(B=3, N=12, K=3, seed=0):
    g = torch.Generator().manual_seed(seed)
    n = torch.tensor([N, N - 4, 3, N - 1][:B])
    mask = torch.arange(N)[None, :] < n[:, None]
    a = torch.rand(B, N, N, generator=g, dtype=torch.float64)
    a = (a < 0.5) * (a + a.transpose(1, 2)) * (mask[:, :, None] & mask[:, None, :])
    s = torch.softmax(torch.randn(B, N, K, generator=g, dtype=torch.float64), -1) * mask[..., None]
    return a, s, mask


def test_oracle_gradcheck_float64():
    a, s, mask = _masked_batch(B=2, N=7, K=3, seed=3)
    a = a + 0.1 * torch.rand_like(a).triu(1)  # an asymmetric part: the transposes of the backward matter
    fn = lambda a_, s_: O.hosc_losses(a_, s_, mask)  # noqa: E731
    assert torch.autograd.gradcheck(fn, (a.requires_grad_(), s.requires_grad_()), eps=1e-6, atol=1e-7)


def closed_form(a, s, g, mask=None, eps=O.EPS):
    """dS, dA of g . [L1, L2, O] as the kernels compute them (dense_hosc.cu)."""
    B, N, K = s.shape
    P = a @ a
    am = P * a

    def order(adj, gk):
        d = adj.sum(-1)
        n = torch.einsum("bik,bij,bjk->bk", s, adj, s)
        m = torch.einsum("bi,bik->bk", d, s * s) + eps
        alpha, beta = -gk / (K * B * m), gk * n / (K * B * m * m)
        sa = s * alpha[:, None, :]
        ds = adj @ sa + adj.transpose(1, 2) @ sa + 2 * d[..., None] * s * beta[:, None, :]
        r = (s * s * beta[:, None, :]).sum(-1)
        return ds, sa @ s.transpose(1, 2) + r[..., None]

    ds1, e1 = order(a, g[0])
    ds2, G = order(am, g[1])
    nb = mask.sum(1).to(s.dtype) if mask is not None else torch.full((B,), float(N), dtype=s.dtype)
    norms = torch.norm(s, dim=1, keepdim=True)
    coef = -g[2] / (B * torch.sqrt(nb)[:, None, None] * (math.sqrt(K) - 1))
    ds_o = torch.where(norms > 0, coef * s / norms.clamp_min(1e-300), torch.zeros_like(s))
    Hm = G * a
    da = e1 + G * P + Hm @ a.transpose(1, 2) + a.transpose(1, 2) @ Hm
    return ds1 + ds2 + ds_o, da


@pytest.mark.parametrize("case", ["ragged0", "ragged1", "asym", "zero_column"])
def test_closed_form_gradients_match_autograd(case):
    a, s, mask = _masked_batch(B=4, N=12, K=3, seed=int(case[-1]) if case[-1].isdigit() else 5)
    if case == "asym":
        a = a * (1 + torch.rand_like(a))  # A != A^T
    if case == "zero_column":
        s[:, :, 2] = 0.0
    g = torch.tensor([0.7, -1.3, 0.9], dtype=torch.float64)
    a_, s_ = a.clone().requires_grad_(), s.clone().requires_grad_()
    (g * O.hosc_losses(a_, s_, mask)).sum().backward()
    ds, da = closed_form(a, s, g, mask)
    torch.testing.assert_close(s_.grad, ds, rtol=1e-10, atol=1e-12)
    torch.testing.assert_close(a_.grad, da, rtol=1e-10, atol=1e-12)


class HOSCPooling(H._DenseBase):  # the restated attributes of HOSCPooling
    mu, alpha, hosc_ortho = 0.3, 0.4, False


@pytest.mark.parametrize("hosc_ortho", [False, True])
def test_hosc_pool_and_patched_pooler_wiring(monkeypatch, hosc_ortho):
    """The pooler-level code with the device calls replaced by the oracle: alpha, mu, the mask, the ortho choice, the
    loss keys and the connector flags reach the right places, and the losses come from the raw adjacency."""
    import tgp_b200 as T
    from tgp_b200 import poolers as P

    def dense_pool(x, adj, s, *, loss_kind, **flags):
        assert loss_kind == (T.functional.LOSS_NONE if hosc_ortho else T.functional.LOSS_MINCUT)
        raw = R.dense_connect(adj, s)
        losses = torch.stack([R.mincut_loss(adj, s, raw), R.orthogonality_loss(s), s.new_zeros(()), s.new_zeros(())])
        return s.transpose(1, 2) @ x, R.postprocess_adj_pool_dense(raw, **flags), losses

    def hosc_losses(adj, s, alpha, hosc_ortho_, graph_nodes=None, eps=1e-8):
        assert hosc_ortho_ == hosc_ortho and eps == 1e-8
        m = torch.arange(s.size(1))[None, :] < graph_nodes[:, None]
        return O.hosc_losses(adj, s, m, eps)

    monkeypatch.setattr(P.F_, "dense_pool", dense_pool)
    monkeypatch.setattr(P.F_, "hosc_losses", hosc_losses)
    a, s, mask = _masked_batch(B=3, N=12, K=3, seed=2)
    x = torch.randn(3, 12, 5, dtype=torch.float64)
    flags = dict(remove_self_loops=True, degree_norm=True, adj_transpose=False, edge_weight_norm=True)
    pooler = HOSCPooling(selector=lambda x, mask: R.OracleSelectOutput(s=s), reducer=H.BaseReduce(),
                         connector=H.DenseConnect(**flags))
    pooler.hosc_ortho = hosc_ortho
    T.patch_pooler(pooler)
    out = pooler(x=x, adj=a, mask=mask)
    xp, ap, loss = O.hosc_pool(x, a, s, mask, 0.3, 0.4, hosc_ortho, **flags)
    assert set(out.loss) == {"hosc_loss", "ortho_loss"} == set(loss)
    for k in loss:
        torch.testing.assert_close(out.loss[k], loss[k], rtol=1e-12, atol=0.0)
    torch.testing.assert_close(out.x, xp)
    torch.testing.assert_close(out.edge_index, ap)


def test_hosc_ops_fake_tensor_shapes():
    from torch._subclasses.fake_tensor import FakeTensorMode

    import tgp_b200  # noqa: F401  (registers the ops and their fake kernels)
    from tgp_b200 import ops

    assert {"hosc_losses", "hosc_losses_bwd"} <= set(ops.OP_NAMES)
    with FakeTensorMode():
        s = torch.empty(4, 32, 8, device="cuda", dtype=torch.bfloat16)
        a = torch.empty(4, 32, 32, device="cuda", dtype=torch.bfloat16)
        n = torch.empty(4, device="cuda")
        losses, saved = torch.ops.tgp_b200.hosc_losses(a, s, n, 7, 1e-8)
        assert losses.shape == (3,) and losses.dtype == torch.float32 and saved.dtype == torch.uint8
        ga, gs = torch.ops.tgp_b200.hosc_losses_bwd(a, s, n, saved, losses, 7, True)
        assert ga.shape == a.shape and gs.shape == s.shape
        ga, _ = torch.ops.tgp_b200.hosc_losses_bwd(a, s, None, saved, losses, 1, False)
        assert ga.numel() == 0


def test_saved_bytes_hold_the_motif_adjacency_only_when_asked():
    from tgp_b200 import _lib as L

    lib = L.load()
    B, N, K = 4, 64, 8
    with_motif = lib.tgpb200_hosc_loss_saved_bytes(B, N, K, 3, L.F32)
    without = lib.tgpb200_hosc_loss_saved_bytes(B, N, K, 1, L.F32)
    assert with_motif - without == B * N * N * 4
    assert lib.tgpb200_hosc_loss_saved_bytes(B, N, K, 3, L.BF16) - without == B * N * N * 2


def test_hosc_pool_is_exported_and_cpu_raises():
    import tgp_b200 as T

    assert "hosc_pool" in T.__all__
    with pytest.raises(RuntimeError, match="CUDA"):
        T.hosc_pool(torch.randn(1, 4, 2), torch.rand(1, 4, 4), torch.rand(1, 4, 2))
    with pytest.raises(RuntimeError, match="CUDA"):
        T.functional.hosc_losses(torch.rand(1, 4, 4), torch.rand(1, 4, 2), 0.5, False)
