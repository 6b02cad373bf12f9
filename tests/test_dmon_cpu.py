"""CPU: the DMoN oracle (hand values, float64 gradcheck, the closed-form gradients the kernels implement) and the
shape propagation of the dense op's ``graph_nodes`` argument.  No kernels are launched here."""
import math

import pytest
import torch

import dmon_oracle as D
from oracle import ref_path as R


def _two_triangles():
    a = torch.zeros(1, 6, 6, dtype=torch.float64)
    for comp in ([0, 1, 2], [3, 4, 5]):
        for i in comp:
            for j in comp:
                if i != j:
                    a[0, i, j] = 1.0
    return a


def test_hand_values():
    a = _two_triangles()
    x = torch.randn(1, 6, 3, dtype=torch.float64)
    s = torch.zeros(1, 6, 2, dtype=torch.float64)
    s[0, :3, 0] = 1.0
    s[0, 3:, 1] = 1.0
    _, _, loss = D.dmon_pool(x, a, s)
    assert loss["spectral_loss"].item() == pytest.approx(-0.5, abs=1e-12)  # minus the modularity of the split
    assert loss["cluster_loss"].item() == pytest.approx(0.0, abs=1e-12)
    one = torch.zeros(1, 6, 2, dtype=torch.float64)
    one[0, :, 0] = 1.0
    _, _, loss = D.dmon_pool(x, a, one)
    assert loss["cluster_loss"].item() == pytest.approx(math.sqrt(2) - 1, abs=1e-12)
    assert loss["spectral_loss"].item() == pytest.approx(0.0, abs=1e-12)


def test_zero_degree_graph_gives_nan():
    a = torch.zeros(1, 4, 4, dtype=torch.float64)
    s = torch.softmax(torch.randn(1, 4, 2, dtype=torch.float64), -1)
    assert torch.isnan(D.spectral_loss(a, s, R.dense_connect(a, s)))


def _masked_batch(B=3, N=9, K=4, F=5, seed=0, dtype=torch.float64):
    g = torch.Generator().manual_seed(seed)
    n = torch.tensor([N, N - 3, 4][:B])
    mask = torch.arange(N).unsqueeze(0) < n.unsqueeze(1)
    a = torch.rand(B, N, N, generator=g, dtype=dtype)
    a = (a + a.transpose(1, 2)) * (mask.unsqueeze(1) & mask.unsqueeze(2))
    s = torch.softmax(torch.randn(B, N, K, generator=g, dtype=dtype), -1) * mask.unsqueeze(-1)
    x = torch.randn(B, N, F, generator=g, dtype=dtype) * mask.unsqueeze(-1)
    return x, a, s, mask


def test_gradcheck_float64():
    x, a, s, mask = _masked_batch()

    def f(x, a, s):
        xp, ap, loss = D.dmon_pool(x, a, s, mask, 0.7, 1.3, 0.9)
        return xp.sum(), ap.square().sum(), loss["spectral_loss"], loss["cluster_loss"], loss["ortho_loss"]

    assert torch.autograd.gradcheck(f, (x.requires_grad_(), a.requires_grad_(), s.requires_grad_()))


@pytest.mark.parametrize("seed", [0, 1, 2])
def test_closed_form_gradients_match_autograd(seed):
    """dS and dA of g_s * spectral + g_c * cluster from the formulas the kernels implement (the trace term as a
    diagonal Graw, d_i u_k + v_k, the row broadcast r_i) against the oracle's autograd."""
    x, a, s, mask = _masked_batch(seed=seed)
    B, N, K = s.shape
    g_s, g_c = 0.8, -1.7
    a_, s_ = a.clone().requires_grad_(), s.clone().requires_grad_()
    (g_s * D.spectral_loss(a_, s_, R.dense_connect(a_, s_)) + g_c * D.cluster_loss(s_, mask)).backward()

    gamma = g_s / B
    d = a.sum(-1)  # [B, N]
    m2 = d.sum(-1)  # 2m
    t = torch.einsum("bii->b", s.transpose(1, 2) @ a @ s)
    c = (s.transpose(1, 2) @ d.unsqueeze(-1)).squeeze(-1)  # [B, K]
    e = s.sum(1)
    n = mask.sum(1).to(s.dtype)
    graw = (-gamma / m2)[:, None, None] * torch.eye(K, dtype=s.dtype)  # c_num on the diagonal
    u = 2 * gamma * c / m2[:, None] ** 2
    v = (g_c / B) * math.sqrt(K) * e / (n * e.norm(dim=-1))[:, None]
    ds = a @ s @ graw.transpose(1, 2) + a.transpose(1, 2) @ s @ graw + d[:, :, None] * u[:, None, :] + v[:, None, :]
    r = gamma * (2 * (s @ c.unsqueeze(-1)).squeeze(-1) / m2[:, None] ** 2 + (t / m2 ** 2)[:, None]
                 - (2 * (c * c).sum(-1) / m2 ** 3)[:, None])
    da = s @ graw @ s.transpose(1, 2) + r[:, :, None]
    torch.testing.assert_close(s_.grad, ds, rtol=1e-10, atol=1e-12)
    torch.testing.assert_close(a_.grad, da, rtol=1e-10, atol=1e-12)


def test_fake_tensor_shapes_with_graph_nodes():
    from torch._subclasses.fake_tensor import FakeTensorMode

    import tgp_b200  # noqa: F401  (registers the ops and their fake kernels)

    schema = str(torch.ops.tgp_b200.stas_fused.default._schema)
    assert "Tensor? graph_nodes=None" in schema
    assert "Tensor? graph_nodes=None" in str(torch.ops.tgp_b200.stas_fused_bwd.default._schema)
    with FakeTensorMode():
        s = torch.empty(4, 32, 8, device="cuda")
        x = torch.empty(4, 32, 16, device="cuda")
        a = torch.empty(4, 32, 32, device="cuda")
        gn = torch.empty(4, device="cuda")
        xp, ap, losses, saved = torch.ops.tgp_b200.stas_fused(x, a, s, 3, 3, 1.0, 1.0, gn)
        assert xp.shape == (4, 8, 16) and ap.shape == (4, 8, 8) and losses.shape == (4,) and saved.dtype == torch.uint8
        gx, ga, gs = torch.ops.tgp_b200.stas_fused_bwd(x, a, s, saved, xp, ap, losses, 3, 3, 1.0, 1.0, True, gn)
        assert gx.shape == x.shape and ga.shape == a.shape and gs.shape == s.shape


def test_dmon_pool_is_exported_and_cpu_raises():
    import tgp_b200 as T

    assert T.functional.LOSS_DMON == 3 and "dmon_pool" in T.__all__
    with pytest.raises(RuntimeError, match="CUDA"):
        T.dmon_pool(torch.randn(1, 4, 2), torch.rand(1, 4, 4), torch.rand(1, 4, 2))
