"""B200: HOSC pooling (``hosc_losses`` / ``hosc_pool``) against the float64 oracle of ``tests/hosc_oracle.py``, per
gradient source, on shapes on and off the engine's TMA grid; bf16; hand values; determinism; graph replay; the patched
pooler; the term mask (no A A product when alpha = 0); the memory bound and argument errors."""
import pytest
import torch

import dense_loss_cases as C
import dropin_harness as H
import hosc_oracle as O
import tgp_b200 as T
from dense_loss_cases import DEV, FLAGSETS
from tgp_b200 import _lib as L
from tgp_b200 import functional as F_

pytestmark = pytest.mark.gpu
COEF = {"hosc": 1.7, "ortho": -0.8}
KEYS = {"hosc": "hosc_loss", "ortho": "ortho_loss"}


class HOSCPooling(H._DenseBase):  # the restated attributes of HOSCPooling
    mu, alpha, hosc_ortho = 0.2, 0.6, True


def _oracle(x, a, s, mask, alpha, hosc_ortho, flags, up):
    """float64 forward on the CPU and the (dX, dA, dS) of each gradient source alone."""
    leaves = tuple(t.double().requires_grad_(True) for t in (x, a, s))
    xp, ap, loss = O.hosc_pool(*leaves, mask, 0.3, alpha, hosc_ortho, **flags)
    losses = torch.stack([loss[KEYS["hosc"]], loss[KEYS["ortho"]]]).detach()
    return xp.detach(), ap.detach(), losses, C.per_source_grads(xp, ap, loss, up, leaves, COEF, KEYS)


def _device(x, a, s, mask, alpha, hosc_ortho, flags, up, dtype=torch.float32):
    leaves = tuple(t.to(DEV, dtype).requires_grad_(True) for t in (x, a, s))
    xp, ap, loss = T.hosc_pool(*leaves, mask.to(DEV), 0.3, alpha, hosc_ortho, **flags)
    losses = torch.stack([loss[KEYS["hosc"]], loss[KEYS["ortho"]]]).detach()
    grads = C.per_source_grads(xp, ap, loss, up, leaves, COEF, KEYS)
    return xp.detach(), ap.detach(), losses, {k: [t.cpu() for t in v] for k, v in grads.items()}


@pytest.mark.parametrize("hosc_ortho", [False, True])
@pytest.mark.parametrize("alpha", [0.0, 0.5, 1.0])
@pytest.mark.parametrize("flags", FLAGSETS)
@pytest.mark.parametrize("shape", [(3, 256, 64, 128), (5, 200, 48, 100), (4, 100, 16, 33), (2, 96, 64, 36)])
def test_fp32_parity(shape, flags, alpha, hosc_ortho):
    B, N, K, F = shape
    x, a, s, mask = C.planted_partition(B, N, K, F, seed=sum(shape))
    up = C.upstream(B, K, F, sum(shape))
    xp_e, ap_e, loss_e, g_e = _oracle(x, a, s, mask, alpha, hosc_ortho, flags, up)
    xp, ap, loss, g = _device(x, a, s, mask, alpha, hosc_ortho, flags, up)
    torch.testing.assert_close(loss.cpu().double(), loss_e, rtol=1e-5, atol=0.0)
    for name, gv, ev in (("x_pool", xp, xp_e), ("adj_pool", ap, ap_e)):
        torch.testing.assert_close(gv.cpu().double(), ev, rtol=1e-5, atol=1e-5 * float(ev.abs().max()), msg=name)
    C.check_per_source(g, g_e, 1e-4, flags["edge_weight_norm"])


@pytest.mark.parametrize("hosc_ortho", [False, True])
@pytest.mark.parametrize("shape", [(3, 256, 64, 128), (2, 512, 256, 64), (4, 100, 16, 32)])
def test_bf16_parity(shape, hosc_ortho):
    B, N, K, F = shape
    x, a, s, mask = C.planted_partition(B, N, K, F, seed=7 + sum(shape))
    x, a, s = (t.bfloat16().float() for t in (x, a, s))  # the oracle sees the rounded operands
    up = tuple(v.bfloat16().float() for v in C.upstream(B, K, F, 7))
    xp_e, ap_e, loss_e, g_e = _oracle(x, a, s, mask, 0.5, hosc_ortho, FLAGSETS[0], up)
    xp, ap, loss, g = _device(x, a, s, mask, 0.5, hosc_ortho, FLAGSETS[0], up, dtype=torch.bfloat16)
    torch.testing.assert_close(loss.cpu().double(), loss_e, rtol=2e-2, atol=0.0)
    for name, gv, ev in (("x_pool", xp, xp_e), ("adj_pool", ap, ap_e)):
        torch.testing.assert_close(gv.cpu().double(), ev, rtol=2e-2, atol=2e-2 * float(ev.abs().max()), msg=name)
    C.check_per_source(g, g_e, 2e-2, False)


def test_raw_terms_and_hand_values_on_device():
    """[L1, L2, O] of functional.hosc_losses: disjoint triangles with a one-hot S give A_M = A, L1 = L2 = -1, O = 0; a
    4-cycle split into two pairs gives L1 = -1/2 and, without a triangle, L2 = 0 (no NaN)."""
    a = torch.zeros(2, 6, 6)
    for comp in ([0, 1, 2], [3, 4, 5]):
        for i in comp:
            for j in comp:
                if i != j:
                    a[0, i, j] = 1.0
    for i in range(4):
        a[1, i, (i + 1) % 4] = a[1, (i + 1) % 4, i] = 1.0
    s = torch.zeros(2, 6, 2)
    s[0, :3, 0] = s[0, 3:, 1] = 1.0
    s[1, :2, 0] = s[1, 2:4, 1] = 1.0
    n = torch.tensor([6.0, 4.0])
    got = F_.hosc_losses(a[:1].to(DEV), s[:1].to(DEV), 0.5, True, graph_nodes=n[:1].to(DEV)).cpu()
    torch.testing.assert_close(got, torch.tensor([-1.0, -1.0, 0.0]), rtol=0, atol=1e-6)
    got = F_.hosc_losses(a[1:, :4, :4].contiguous().to(DEV), s[1:, :4].contiguous().to(DEV), 0.5, False).cpu()
    torch.testing.assert_close(got[:2], torch.tensor([-0.5, 0.0]), rtol=0, atol=1e-6)
    mask = torch.arange(6)[None, :] < n[:, None]
    exp = O.hosc_losses(a.double(), s.double(), mask)
    got = F_.hosc_losses(a.to(DEV), s.to(DEV), 0.5, True, graph_nodes=n.to(DEV)).cpu()
    torch.testing.assert_close(got.double(), exp, rtol=1e-5, atol=1e-7)


def _graph_inputs(B=6, N=256, K=64, F=128, seed=9):
    x, a, s, mask = C.planted_partition(B, N, K, F, seed=seed)
    up = C.upstream(B, K, F, seed)
    return (x.to(DEV).requires_grad_(True), a.to(DEV).requires_grad_(True), s.to(DEV).requires_grad_(True),
            mask.to(DEV), up[0].to(DEV), up[1].to(DEV))


def _step(x, a, s, mask, gx, ga):
    for t in (x, a, s):
        t.grad = None
    xp, ap, loss = T.hosc_pool(x, a, s, mask, 0.4, 0.5, True, **FLAGSETS[1])
    torch.autograd.backward([xp, ap, loss["hosc_loss"], loss["ortho_loss"]],
                            [gx, ga, torch.ones((), device=DEV), torch.ones((), device=DEV)])
    return xp, ap, loss["hosc_loss"], loss["ortho_loss"]


def test_deterministic():
    x, a, s, mask, gx, ga = _graph_inputs(B=8, seed=3)
    C.assert_deterministic(lambda: _step(x, a, s, mask, gx, ga), [x, a, s])


def test_graph_replay_matches_eager():
    x, a, s, mask, gx, ga = _graph_inputs()
    C.assert_replay_matches_eager(lambda: _step(x, a, s, mask, gx, ga), [x, a, s])


def test_patched_pooler_masked_ragged_batch():
    C.check_patched_pooler(HOSCPooling, lambda x, a, s, mask: O.hosc_pool(x, a, s, mask, 0.2, 0.6, True), "cpu",
                           KEYS.values())


def _launched(alpha, need_adj):
    x, a, s, mask = C.planted_partition(2, 128, 16, 8, seed=5)
    a, s = a.to(DEV).requires_grad_(need_adj), s.to(DEV).requires_grad_(True)
    torch.cuda.synchronize()
    L.time_kernel("*")
    try:
        losses = F_.hosc_losses(a, s, alpha, False)
        ((1 - alpha) * losses[0] + alpha * losses[1]).backward()
        names = [n for n, _ in L.kernel_trace()]
    finally:
        L.time_kernel(None)
    return names


@pytest.mark.parametrize("need_adj", [False, True])
def test_no_motif_work_when_alpha_is_zero(need_adj):
    names = _launched(0.0, need_adj)
    assert "k_hosc_stats" in names and "k_hosc_ds_elementwise" in names
    assert not any("k_hosc_motif" in n or "P=AA" in n or "AMS1" in n for n in names), names
    names = _launched(0.5, need_adj)
    assert "k_hosc_motif" in names and sum("P=AA" in n for n in names) == (2 if need_adj else 1), names


def test_extra_memory_of_forward_and_backward():
    """With only S requiring grad, the extra peak of a forward + backward stays below 2.5 B N^2 fp32 words: A_M (saved)
    is the one N^2 buffer that lives past the forward."""
    B, N, K = 16, 512, 64
    _, a, s, _ = C.planted_partition(B, N, K, 8, seed=1, ragged=False)
    a, s = a.to(DEV), s.to(DEV).requires_grad_(True)
    torch.cuda.synchronize()
    torch.cuda.reset_peak_memory_stats()
    base = torch.cuda.memory_allocated()
    losses = F_.hosc_losses(a, s, 0.5, True)
    losses.sum().backward()
    torch.cuda.synchronize()
    extra = torch.cuda.max_memory_allocated() - base
    assert extra < 2.5 * B * N * N * 4, (extra, B * N * N * 4)
    assert torch.isfinite(s.grad).all().item()


def test_argument_errors():
    s = torch.rand(2, 16, 4, device=DEV)
    a = torch.rand(2, 16, 16, device=DEV)
    with pytest.raises(RuntimeError, match="CUDA"):
        F_.hosc_losses(a.cpu(), s.cpu(), 0.5, False)
    with pytest.raises(NotImplementedError):  # no CPU kernel behind the op
        torch.ops.tgp_b200.hosc_losses(a.cpu(), s.cpu(), None, 3, 1e-8)
    with pytest.raises(ValueError, match="K >= 2"):
        F_.hosc_losses(a, s[..., :1].contiguous(), 0.5, False)
    with pytest.raises(ValueError, match="K >= 2"):
        torch.ops.tgp_b200.hosc_losses(a, s[..., :1].contiguous(), None, 3, 1e-8)
    with pytest.raises(ValueError, match="terms"):
        torch.ops.tgp_b200.hosc_losses(a, s, None, 0, 1e-8)
    with pytest.raises(RuntimeError, match="dtype"):
        F_.hosc_losses(a.bfloat16(), s, 0.5, False)
    with pytest.raises(RuntimeError, match=r"\[B, N, N\]"):
        F_.hosc_losses(a[:, :8], s, 0.5, False)
    with pytest.raises(RuntimeError, match="graph_nodes"):
        F_.hosc_losses(a, s, 0.5, True, graph_nodes=torch.ones(3, device=DEV))
