"""B200: Asymmetric Cheeger Cut pooling (``acc_losses`` / ``acc_pool``) against the float64 oracle of
``tests/acc_oracle.py``, per gradient source; the quantile value and row; bf16; determinism; graph replay; the patched
pooler; argument errors and the memory bound.  The oracle runs in float64 on the device (it is plain torch): at the
larger shapes its ``[B, N, N, K]`` intermediate does not fit a CPU run's time."""
import pytest
import torch

import acc_oracle as A
import dense_loss_cases as C
import dropin_harness as H
import tgp_b200 as T
from dense_loss_cases import DEV, FLAGSETS
from tgp_b200 import functional as F_

pytestmark = pytest.mark.gpu
COEF = {"tv": 1.7, "bal": -0.8}
KEYS = {"tv": "total_variation_loss", "bal": "balance_loss"}


class AsymCheegerCutPooling(H._DenseBase):  # the restated attributes of AsymCheegerCutPooling
    totvar_coeff, balance_coeff = 0.6, 1.4


def _oracle(x, a, s, flags, up, dev=DEV):
    """float64 forward and the (dX, dA, dS) of each gradient source alone."""
    x64, a64, s64 = (t.to(dev, torch.float64).requires_grad_(True) for t in (x, a, s))
    xp, ap, loss = A.acc_pool(x64, a64, s64, **flags)
    grads = C.per_source_grads(xp, ap, loss, up, (x64, a64, s64), COEF, KEYS)
    losses = torch.stack([loss[KEYS["tv"]], loss[KEYS["bal"]]]).detach()
    qv, qi = A.quantile(s64.detach())
    return xp.detach(), ap.detach(), losses, qv, qi, grads


def _saved_rows(saved, B, K):
    """The quantile rows [B, K] int32 of the forward's saved buffer (after nnz int64 [B], 256-byte aligned)."""
    off = -(-B * 8 // 256) * 256
    return saved[off:off + 4 * B * K].view(torch.int32).view(B, K)


def _device(x, a, s, flags, up, dtype=torch.float32):
    xd, ad, sd = (t.to(DEV, dtype).requires_grad_(True) for t in (x, a, s))
    xp, ap, loss = T.acc_pool(xd, ad, sd, **flags)
    grads = C.per_source_grads(xp, ap, loss, up, (xd, ad, sd), COEF, KEYS)
    losses = torch.stack([loss[KEYS["tv"]], loss[KEYS["bal"]]]).detach()
    _, quant, saved = torch.ops.tgp_b200.acc_losses(ad.detach().contiguous(), sd.detach().contiguous())
    return xp.detach(), ap.detach(), losses, quant, _saved_rows(saved, s.size(0), s.size(2)), grads


@pytest.mark.parametrize("flags", FLAGSETS)
@pytest.mark.parametrize("shape", [(3, 256, 64, 128), (5, 200, 48, 100), (4, 100, 16, 33), (2, 96, 64, 36)])
def test_fp32_parity(shape, flags):
    B, N, K, F = shape
    x, a, s, mask = C.planted_partition(B, N, K, F, seed=sum(shape))
    up = C.upstream(B, K, F, sum(shape))
    xp_e, ap_e, loss_e, qv_e, qi_e, g_e = _oracle(x, a, s, flags, up)
    xp, ap, loss, quant, rows, g = _device(x, a, s, flags, up)
    torch.testing.assert_close(loss.double(), loss_e, rtol=1e-5, atol=0.0)
    for name, gv, ev in (("x_pool", xp, xp_e), ("adj_pool", ap, ap_e)):
        torch.testing.assert_close(gv.double(), ev, rtol=1e-5, atol=1e-5 * float(ev.abs().max()), msg=name)
    assert torch.equal(quant, qv_e.float())  # bit for bit: the same element of S
    assert torch.equal(rows.long(), qi_e)
    C.check_per_source(g, g_e, 1e-4, flags["edge_weight_norm"])


def test_quantile_among_tied_padded_zeros():
    """Graphs with fewer valid nodes than N // K: the quantile falls among the padded zero rows (some stored as -0.0),
    and the stable sort's rank rule picks row n_b + (N // K - n_b) of them."""
    B, N, K, F = 3, 64, 4, 8
    x, a, s, mask = C.planted_partition(B, N, K, F, seed=4)
    n = torch.tensor([10, 5, 64])
    mask = torch.arange(N)[None, :] < n[:, None]
    s = s * mask[..., None]
    a = a * (mask[:, :, None] & mask[:, None, :])
    s[0, 12:20, 1] = -0.0  # the selected row of graph 0, column 1 is a -0.0
    up = C.upstream(B, K, F, 4)
    _, _, loss_e, qv_e, qi_e, g_e = _oracle(x, a, s, FLAGSETS[0], up, dev="cpu")  # the CPU sort: -0.0 ties +0.0
    _, _, loss, quant, rows, g = _device(x, a, s, FLAGSETS[0], up)
    assert qi_e[0].tolist() == [16] * K and qi_e[1].tolist() == [16] * K
    assert torch.equal(rows.cpu().long(), qi_e)
    assert torch.equal(quant.cpu().view(torch.int32), qv_e.float().view(torch.int32))
    assert quant[0, 1].view(torch.int32).item() == -2 ** 31
    torch.testing.assert_close(loss.cpu().double(), loss_e, rtol=1e-5, atol=0.0)
    C.check_per_source({k: [t.cpu() for t in v] for k, v in g.items()}, g_e, 1e-4, False)


def test_tie_column_rank_rule():
    s = torch.tensor([[[.5, .1], [.2, .2], [.2, .3], [.2, .9], [.1, .4]]])
    a = torch.tensor([[[0, 1, 0, 1, 0], [1, 0, 1, 0, 0], [0, 1, 0, 2, 1], [1, 0, 2, 0, 0], [0, 0, 1, 0, 1.]]])
    x = torch.randn(1, 5, 3)
    up = C.upstream(1, 2, 3, 0)
    _, _, loss_e, qv_e, qi_e, g_e = _oracle(x, a, s, FLAGSETS[2], up, dev="cpu")
    _, _, loss, quant, rows, g = _device(x, a, s, FLAGSETS[2], up)
    assert rows[0].tolist() == [2, 2] == qi_e[0].tolist()
    assert torch.equal(quant.cpu(), qv_e.float())
    torch.testing.assert_close(loss.cpu().double(), loss_e, rtol=1e-5, atol=1e-7)
    C.check_per_source({k: [t.cpu() for t in v] for k, v in g.items()}, g_e, 1e-4, False)


@pytest.mark.parametrize("shape", [(3, 256, 64, 128), (2, 512, 256, 64), (4, 100, 16, 32)])
def test_bf16_parity(shape):
    B, N, K, F = shape
    x, a, s, mask = C.planted_partition(B, N, K, F, seed=7 + sum(shape))
    x, a, s = (t.bfloat16().float() for t in (x, a, s))  # the oracle sees the rounded operands (and their ties)
    up = tuple(v.bfloat16().float() for v in C.upstream(B, K, F, 7))
    xp_e, ap_e, loss_e, qv_e, qi_e, g_e = _oracle(x, a, s, FLAGSETS[0], up)
    xp, ap, loss, quant, rows, g = _device(x, a, s, FLAGSETS[0], up, dtype=torch.bfloat16)
    torch.testing.assert_close(loss.double(), loss_e, rtol=2e-2, atol=0.0)
    for name, gv, ev in (("x_pool", xp, xp_e), ("adj_pool", ap, ap_e)):
        torch.testing.assert_close(gv.double(), ev, rtol=2e-2, atol=2e-2 * float(ev.abs().max()), msg=name)
    assert torch.equal(quant.double(), qv_e)  # the operands are bf16 values: the selected one is exact
    assert torch.equal(rows.long(), qi_e)
    C.check_per_source(g, g_e, 2e-2, False)


def _graph_inputs(B=6, N=256, K=64, F=128, seed=9):
    x, a, s, mask = C.planted_partition(B, N, K, F, seed=seed)
    up = C.upstream(B, K, F, seed)
    return (x.to(DEV).requires_grad_(True), a.to(DEV).requires_grad_(True), s.to(DEV).requires_grad_(True),
            up[0].to(DEV), up[1].to(DEV))


def _step(x, a, s, gx, ga):
    for t in (x, a, s):
        t.grad = None
    xp, ap, loss = T.acc_pool(x, a, s, 0.9, 1.3, **FLAGSETS[1])
    torch.autograd.backward([xp, ap, loss[KEYS["tv"]], loss[KEYS["bal"]]],
                            [gx, ga, torch.ones((), device=DEV), torch.ones((), device=DEV)])
    return xp, ap, loss[KEYS["tv"]], loss[KEYS["bal"]]


def test_deterministic():
    x, a, s, gx, ga = _graph_inputs(B=8, seed=3)
    C.assert_deterministic(lambda: _step(x, a, s, gx, ga), [x, a, s])


def test_graph_replay_matches_eager():
    x, a, s, gx, ga = _graph_inputs()
    C.assert_replay_matches_eager(lambda: _step(x, a, s, gx, ga), [x, a, s])


def test_patched_pooler_masked_ragged_batch():
    C.check_patched_pooler(AsymCheegerCutPooling, lambda x, a, s, mask: A.acc_pool(x, a, s, 0.6, 1.4), DEV,
                           KEYS.values())


def test_hand_values_and_edgeless_graph_on_device():
    a = torch.zeros(2, 6, 6)
    for comp in ([0, 1, 2], [3, 4, 5]):
        for i in comp:
            for j in comp:
                if i != j:
                    a[0, i, j] = 1.0
    a[0, 2, 3] = a[0, 3, 2] = 0.5
    s = torch.zeros(2, 6, 2)
    s[:, :3, 0] = 1.0
    s[:, 3:, 1] = 1.0
    losses = F_.acc_losses(a[:1].to(DEV), s[:1].to(DEV))
    assert abs(losses[0].item() - 1.0 / 14.0) < 1e-7 and abs(losses[1].item()) < 1e-7
    losses = F_.acc_losses(a.to(DEV), s.to(DEV))  # graph 1 has no edge
    assert torch.isnan(losses[0]).item() and abs(losses[1].item()) < 1e-7


def test_argument_errors():
    s = torch.rand(2, 16, 4, device=DEV)
    a = torch.rand(2, 16, 16, device=DEV)
    with pytest.raises(RuntimeError, match="CUDA"):
        F_.acc_losses(a.cpu(), s.cpu())
    with pytest.raises(NotImplementedError):  # no CPU kernel behind the op
        torch.ops.tgp_b200.acc_losses(a.cpu(), s.cpu())
    with pytest.raises(ValueError, match="K >= 2"):
        F_.acc_losses(a, s[..., :1].contiguous())
    with pytest.raises(ValueError, match="K >= 2"):
        torch.ops.tgp_b200.acc_losses(a, s[..., :1].contiguous())
    with pytest.raises(RuntimeError, match="dtype"):
        F_.acc_losses(a.bfloat16(), s)
    with pytest.raises(RuntimeError, match=r"\[B, N, N\]"):
        F_.acc_losses(a[:, :8], s)


def test_no_pairwise_tensor_in_memory():
    """The extra peak of a forward + backward at (64, 256, 64) stays below 2 x adj.nbytes (dA itself is one): the
    [B, N, N, K] difference tensor of the eager formulation would be 64 x adj.nbytes."""
    x, a, s, mask = C.planted_partition(64, 256, 64, 8, seed=1, ragged=False)
    a, s = a.to(DEV).requires_grad_(True), s.to(DEV).requires_grad_(True)
    torch.cuda.synchronize()
    torch.cuda.reset_peak_memory_stats()
    base = torch.cuda.memory_allocated()
    losses = F_.acc_losses(a, s)
    losses.sum().backward()
    torch.cuda.synchronize()
    extra = torch.cuda.max_memory_allocated() - base
    assert extra < 2 * a.nbytes, (extra, a.nbytes)
    assert a.grad is not None and torch.isfinite(s.grad).all().item()
