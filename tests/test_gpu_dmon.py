"""B200: DMoN on the fused dense path (loss_kind 3) against the float64 oracle, the patched pooler, determinism,
graph replay and argument errors."""
import math

import pytest
import torch

import dense_loss_cases as C
import dmon_oracle as D
import dropin_harness as H
import tgp_b200 as T
from dense_loss_cases import DEV, FLAGSETS
from oracle import ref_path as R
from tgp_b200 import functional as F_

pytestmark = pytest.mark.gpu


class DMoNPooling(H._DenseBase):  # attributes of tgp/poolers/dmon.py
    spectral_loss_coeff, cluster_loss_coeff, ortho_loss_coeff = 0.6, 1.4, 0.8


def _oracle(x, a, s, mask, gx, ga, gl, flags):
    x64, a64, s64 = (t.double().requires_grad_(True) for t in (x, a, s))
    xp, ap, loss = D.dmon_pool(x64, a64, s64, mask, **flags)
    obj = ((xp * gx.double()).sum() + (ap * ga.double()).sum() + gl[0] * loss["spectral_loss"]
           + gl[1] * loss["ortho_loss"] + gl[2] * loss["cluster_loss"])
    obj.backward()
    losses = torch.stack([loss["spectral_loss"], loss["ortho_loss"], loss["cluster_loss"]]).detach()
    return xp.detach(), ap.detach(), losses, x64.grad, a64.grad, s64.grad


def _device(x, a, s, mask, gx, ga, gl, flags, dtype=torch.float32):
    xd, ad, sd = (t.to(DEV, dtype).requires_grad_(True) for t in (x, a, s))
    xp, ap, losses = F_.dense_pool(xd, ad, sd, loss_kind=F_.LOSS_DMON, graph_nodes=mask.sum(1).float().to(DEV), **flags)
    glv = torch.tensor([gl[0], gl[1], gl[2], 0.0], device=DEV)
    torch.autograd.backward([xp, ap, losses], [gx.to(DEV, dtype), ga.to(DEV, dtype), glv])
    return [t.detach().float().cpu() for t in (xp, ap, losses[:3], xd.grad, ad.grad, sd.grad)]


def _upstream(B, K, F, seed):
    return (*C.upstream(B, K, F, seed), (0.9, -1.1, 1.3))


def _check(got, exp, rtol, atol_x, atol_g, edge_weight_norm=False):
    names = ("x_pool", "adj_pool", "losses", "dX", "dA", "dS")
    for name, gv, ev in zip(names, got, exp):
        ev = ev.float()
        if name == "dA" and edge_weight_norm:
            # max-normalisation routes one gradient term to "the" arg-max; a symmetric adjacency ties (r,c) with
            # (c,r) and the reference's pick depends on rounding noise, so only the symmetric part of dA is defined
            gv, ev = 0.5 * (gv + gv.transpose(1, 2)), 0.5 * (ev + ev.transpose(1, 2))
        mx = float(ev.abs().max())
        if name == "losses":
            torch.testing.assert_close(gv, ev, rtol=rtol, atol=0.0, msg=lambda m, name=name: f"{name}: {m}")
        else:
            atol = (atol_g if name in ("dA", "dS") else atol_x) * mx
            torch.testing.assert_close(gv, ev, rtol=rtol if name not in ("dA", "dS") else 0.0, atol=atol,
                                       msg=lambda m, name=name: f"{name}: {m}")


@pytest.mark.parametrize("fused", [True, False])
@pytest.mark.parametrize("flags", FLAGSETS)
@pytest.mark.parametrize("shape", [(3, 256, 64, 128), (5, 200, 48, 100), (4, 100, 16, 33), (2, 96, 64, 36)])
def test_fp32_parity(shape, flags, fused, monkeypatch):
    if not fused:
        monkeypatch.setenv("TGPB200_BWD_FUSED", "0")
    B, N, K, F = shape
    x, a, s, mask = C.planted_partition(B, N, K, F, seed=sum(shape))
    gx, ga, gl = _upstream(B, K, F, sum(shape))
    exp = _oracle(x, a, s, mask, gx, ga, gl, flags)
    got = _device(x, a, s, mask, gx, ga, gl, flags)
    _check(got, exp, rtol=1e-5, atol_x=1e-5, atol_g=1e-4, edge_weight_norm=flags["edge_weight_norm"])


@pytest.mark.parametrize("shape", [(3, 256, 64, 128), (2, 256, 256, 64), (4, 100, 16, 32)])
def test_bf16_parity(shape):
    B, N, K, F = shape
    x, a, s, mask = C.planted_partition(B, N, K, F, seed=7 + sum(shape))
    x, a, s = (t.bfloat16().float() for t in (x, a, s))  # the oracle sees the rounded operands
    gx, ga, gl = _upstream(B, K, F, 7)
    gx, ga = gx.bfloat16().float(), ga.bfloat16().float()
    exp = _oracle(x, a, s, mask, gx, ga, gl, FLAGSETS[0])
    got = _device(x, a, s, mask, gx, ga, gl, FLAGSETS[0], dtype=torch.bfloat16)
    for name, gv, ev in zip(("x_pool", "adj_pool", "losses", "dX", "dA", "dS"), got, exp):
        ev = ev.float()
        torch.testing.assert_close(gv, ev, rtol=2e-2, atol=2e-2 * float(ev.abs().max()),
                                   msg=lambda m, name=name: f"{name}: {m}")


def test_patched_pooler_masked_ragged_batch():
    C.check_patched_pooler(DMoNPooling, lambda x, a, s, mask: D.dmon_pool(x, a, s, mask, 0.6, 1.4, 0.8), "cpu",
                           ("spectral_loss", "cluster_loss", "ortho_loss"),
                           select_output=lambda s: (T.SelectOutput if s.is_cuda else R.OracleSelectOutput)(s=s))


def test_hand_values_on_device():
    a = torch.zeros(1, 6, 6)
    for comp in ([0, 1, 2], [3, 4, 5]):
        for i in comp:
            for j in comp:
                if i != j:
                    a[0, i, j] = 1.0
    s = torch.zeros(1, 6, 2)
    s[0, :3, 0] = 1.0
    s[0, 3:, 1] = 1.0
    x = torch.randn(1, 6, 4)
    _, _, loss = T.dmon_pool(x.to(DEV), a.to(DEV), s.to(DEV))
    assert abs(loss["spectral_loss"].item() + 0.5) < 1e-6 and abs(loss["cluster_loss"].item()) < 1e-6
    one = torch.zeros(1, 6, 2)
    one[0, :, 0] = 1.0
    _, _, loss = T.dmon_pool(x.to(DEV), a.to(DEV), one.to(DEV))
    assert abs(loss["cluster_loss"].item() - (math.sqrt(2) - 1)) < 1e-6


def test_zero_degree_graph_gives_nan_on_device():
    x, a, s, mask = C.planted_partition(3, 64, 8, 16, seed=5, ragged=False)
    a[1] = 0.0
    _, _, losses = F_.dense_pool(x.to(DEV), a.to(DEV), s.to(DEV), loss_kind=F_.LOSS_DMON)
    assert torch.isnan(losses[0]).item() and torch.isfinite(losses[1:3]).all().item()


def test_deterministic():
    B, N, K, F = 8, 256, 64, 128
    x, a, s, mask = C.planted_partition(B, N, K, F, seed=3)
    gx, ga, gl = _upstream(B, K, F, 3)
    C.assert_deterministic(lambda: _device(x, a, s, mask, gx, ga, gl, FLAGSETS[1]), [])


def test_graph_replay_matches_eager():
    B, N, K, F = 6, 256, 64, 128
    x, a, s, mask = C.planted_partition(B, N, K, F, seed=9)
    gx, ga, _ = _upstream(B, K, F, 9)
    x, a, gx, ga = x.to(DEV).requires_grad_(True), a.to(DEV), gx.to(DEV), ga.to(DEV)
    s = s.to(DEV).requires_grad_(True)
    gn = mask.sum(1).float().to(DEV)
    gl = torch.tensor([1.0, 0.5, 2.0, 0.0], device=DEV)

    def step():
        x.grad = None
        s.grad = None
        xp, ap, losses = F_.dense_pool(x, a, s, loss_kind=F_.LOSS_DMON, graph_nodes=gn, **FLAGSETS[0])
        torch.autograd.backward([xp, ap, losses], [gx, ga, gl])
        return xp, ap, losses

    C.assert_replay_matches_eager(step, [x, s])


def test_argument_errors():
    s = torch.rand(2, 16, 4, device=DEV)
    x = torch.rand(2, 16, 8, device=DEV)
    with pytest.raises(ValueError, match="adj"):
        F_.dense_pool(x, None, s, loss_kind=F_.LOSS_DMON)
    with pytest.raises(RuntimeError, match="invalid argument"):  # the C ABI refuses it too
        torch.ops.tgp_b200.stas_fused(x, None, s, 0, 3, 1.0, 1.0)
    a = torch.rand(2, 16, 16, device=DEV)
    with pytest.raises(ValueError, match="graph_nodes"):
        F_.dense_pool(x, a, s, loss_kind=F_.LOSS_DMON, graph_nodes=torch.ones(3, device=DEV))
    with pytest.raises(RuntimeError, match="graph_nodes"):
        torch.ops.tgp_b200.stas_fused(x, a, s, 0, 3, 1.0, 1.0, torch.ones(3, device=DEV))
