"""B200: every gradient source of the dense poolers on its own against the float64 oracle, per graph.

For each path of the dense backward (``grad_sources.PATHS``) and each source (``gx``, ``ga`` and every loss of the
family with a non-unit coefficient), the device gradients dS, dX, dA are compared with the oracle of that source alone:
(a) with explicit zero cotangents for the other outputs, (b) with the other outputs unused (their cotangents reach the
C ABI as null pointers, which selects other code), and (c) the per-source results must add up to one combined backward.
"""
import pytest
import torch

import grad_sources as G
from oracle import ref_path as R
from tgp_b200 import functional as F_

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


def run_device(case, sources, explicit_zeros, with_x=True, adj_grad=True):
    """Device {dS, dX, dA} of the sum of ``sources``.  ``explicit_zeros``: every output enters the backward (zero
    cotangents for the outputs no source uses); otherwise only the outputs the sources use do."""
    x, a, s, n, gx, ga = G.inputs(case)
    dt = torch.bfloat16 if case.bf16 else torch.float32
    xd = x.to(DEV, dt).requires_grad_(True) if with_x else None
    ad = a.to(DEV, dt).requires_grad_(adj_grad)
    sd = s.to(DEV, dt).requires_grad_(True)
    gn = n.float().to(DEV) if case.family == "dmon" else None
    xp, ap, losses = F_.dense_pool(xd, ad, sd, loss_kind=case.loss_kind, ent_div=case.ent_div, graph_nodes=gn,
                                   **case.kw)
    gl = torch.zeros(4, device=DEV)
    for src, idx in G.FAMILIES[case.family][1].items():
        if src in sources:
            gl[idx] = G.LOSS_COEF[src]
    pairs = []
    if with_x and (explicit_zeros or "gx" in sources):
        pairs.append((xp, gx.to(DEV, dt) if "gx" in sources else torch.zeros_like(xp)))
    if explicit_zeros or "ga" in sources:
        pairs.append((ap, ga.to(DEV, dt) if "ga" in sources else torch.zeros_like(ap)))
    if explicit_zeros or any(src in G.LOSS_COEF for src in sources):
        pairs.append((losses, gl))
    torch.autograd.backward([p[0] for p in pairs], [p[1] for p in pairs])
    torch.cuda.synchronize()
    if not adj_grad:
        assert ad.grad is None
    return {"dS": sd.grad, "dX": xd.grad if with_x else None, "dA": ad.grad if adj_grad else None}


def check_case(label, case, sources=None, with_x=True, adj_grad=True):
    sources = case.sources if sources is None else sources
    errors, total = [], {}
    for src in sources:
        ref = G.oracle(case, src)
        for explicit in (True, False):
            got = run_device(case, (src,), explicit, with_x, adj_grad)
            how = "zero cotangents" if explicit else "unused outputs"
            try:
                for k, t in got.items():
                    assert t is None or bool(torch.isfinite(t).all()), f"{k} not finite"
                if not explicit and src != "gx" and with_x:
                    assert not bool(got["dX"].any()), "dX is not exactly 0 without a cotangent of x_pool"
                G.check_grads(case, got, ref, f"{label} {src} ({how})")
            except AssertionError as e:
                errors.append(f"{src} ({how}): {e}")
            if explicit:
                for k, t in got.items():
                    if t is not None:
                        total[k] = total.get(k, 0) + t.double()
    # (c) linearity: the per-source gradients add up to the combined backward
    comb = run_device(case, sources, True, with_x, adj_grad)
    for k, t in comb.items():
        if t is None:
            continue
        try:
            G.assert_per_graph(total[k], t, case.tau, f"{label} sum of sources vs combined {k}")
        except AssertionError as e:
            errors.append(str(e))
    assert not errors, "\n".join(errors)


def _id(p):
    pid, _, c = p
    return f"{pid}-{c.family}-{'x'.join(map(str, c.shape))}-flags{c.flags}"


@pytest.mark.parametrize("pid,env,case", G.path_cases(), ids=[_id(p) for p in G.path_cases()])
def test_each_source_matches_oracle(pid, env, case, monkeypatch):
    for k, v in env.items():
        monkeypatch.setenv(k, v)
    check_case(pid, case)


@pytest.mark.parametrize("family", ["mincut", "diff", "dmon"])
def test_adjacency_only_pooling(family):
    """x = None: no X Gx^T pair in dS, no dX."""
    case = G.Case(family, (5, 200, 48, 100), 0)
    check_case("x=None", case, sources=case.sources[1:], with_x=False)


@pytest.mark.parametrize("family", ["mincut", "diff", "dmon"])
def test_adjacency_without_grad(family):
    """adj.requires_grad = False: dA is not computed (null output of the C ABI)."""
    case = G.Case(family, (5, 256, 64, 128), 1)
    check_case("no dA", case, adj_grad=False)


# --------------------------------------------------------------------------- #
# link-loss gradient when the assignment reproduces the adjacency (A ~ S S^T): the forward switches to the direct
# residual there; the gradient must follow
# --------------------------------------------------------------------------- #
@pytest.mark.parametrize("noise", [0.3, 3e-2, 1e-3, 0.0])
@pytest.mark.parametrize("bf16", [False, True])
def test_link_gradient_small_residual(noise, bf16):
    g = torch.Generator().manual_seed(int(noise * 1e4) + 5)
    B, N, K, F = 3, 192, 24, 32
    blocks = torch.randint(0, K, (B, N), generator=g)
    s = torch.nn.functional.one_hot(blocks, K).float()
    a = s @ s.transpose(1, 2)
    pert = torch.rand(B, N, N, generator=g) < 0.5
    a = a + noise * (pert | pert.transpose(1, 2)).float()
    x = torch.randn(B, N, F, generator=g)
    dt = torch.bfloat16 if bf16 else torch.float32
    x, a, s = (t.to(dt) for t in (x, a, s))
    coef = G.LOSS_COEF["link"]

    sd, ad = s.to(DEV).requires_grad_(True), a.to(DEV).requires_grad_(True)
    _, _, losses = F_.dense_pool(x.to(DEV), ad, sd, loss_kind=F_.LOSS_DIFFPOOL, ent_div=float(B * N), **G.FLAGSETS[0])
    losses.backward(torch.tensor([0.0, 0.0, coef, 0.0], device=DEV))
    got = {"dS": sd.grad.float().cpu(), "dA": ad.grad.float().cpu()}
    for k, t in got.items():
        assert bool(torch.isfinite(t).all()), k
    if noise == 0.0:  # the loss is exactly 0 and so is its gradient
        for k, t in got.items():
            assert not bool(t.any()), f"{k}: max |{k}| = {float(t.abs().max()):.3e} at a zero residual"
        return
    s64, a64 = s.double().requires_grad_(True), a.double().requires_grad_(True)
    ref = torch.autograd.grad(coef * R.link_pred_loss(s64, a64, normalize_loss=False), (s64, a64))
    tau = G.BF16_TAU if bf16 else G.FP32_TAU
    for (k, t), r in zip(got.items(), ref):
        G.assert_per_graph(t, r, tau, f"noise {noise} {k}")
