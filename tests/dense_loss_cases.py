"""Inputs and checks shared by the GPU tests of the dense poolers with losses of their own (DMoN, Asymmetric Cheeger
Cut, HOSC): the planted-partition batch, the upstream gradients, the connector flag sets, the gradient of each source
on its own, determinism and CUDA-graph replay of a step, and the patched pooler on a masked, ragged batch.

``per_source_grads`` / ``check_per_source`` take the gradient apart by source (``x_pool``'s and ``adj_pool``'s
cotangents, then each loss with a non-unit coefficient) and bound every (dX, dA, dS) of every source by
``tau * max|ref|`` over the batch.
"""
import torch

import dropin_harness as H
import tgp_b200 as T

DEV = "cuda:0"
FLAGSETS = [
    dict(remove_self_loops=True, degree_norm=True, adj_transpose=True, edge_weight_norm=False),
    dict(remove_self_loops=True, degree_norm=True, adj_transpose=False, edge_weight_norm=True),
    dict(remove_self_loops=False, degree_norm=False, adj_transpose=False, edge_weight_norm=False),
]


def planted_partition(B, N, K, F, seed, ragged=True):
    """(x, a, s, mask): planted-partition graphs (dense communities: many triangles) with communities of skewed sizes
    and an assignment that follows them.  The modularity and the size imbalance are far from zero, so no loss is a
    cancellation residue that float32 cannot resolve to rtol 1e-5.  Graph b has n_b valid nodes (padded rows / columns
    are zero)."""
    g = torch.Generator().manual_seed(seed)
    n = torch.tensor([N - (7 * b) % max(1, N // 3) if ragged else N for b in range(B)])
    mask = torch.arange(N)[None, :] < n[:, None]
    comm = (K * torch.rand(B, N, generator=g) ** 2).long().clamp(max=K - 1)
    same = comm[:, :, None] == comm[:, None, :]
    p = torch.where(same, torch.tensor(0.6), torch.tensor(0.3 / N))
    a = (torch.rand(B, N, N, generator=g) < p).float()
    a = torch.triu(a, 1)
    a = (a + a.transpose(1, 2)) * torch.rand(B, N, N, generator=g).add(0.5)
    a = (a + a.transpose(1, 2)) * 0.5 * (mask[:, :, None] & mask[:, None, :])
    logits = 4.0 * torch.nn.functional.one_hot(comm, K).float() + torch.randn(B, N, K, generator=g)
    s = torch.softmax(logits, -1) * mask[..., None]
    x = torch.randn(B, N, F, generator=g) * mask[..., None]
    return x, a, s, mask


def upstream(B, K, F, seed):
    """The cotangents (gx [B, K, F], ga [B, K, K]) of x_pool and adj_pool."""
    g = torch.Generator().manual_seed(seed + 100)
    return torch.randn(B, K, F, generator=g), torch.randn(B, K, K, generator=g)


def per_source_grads(xp, ap, loss, up, leaves, coef, keys):
    """{source: [dX, dA, dS]} of each source alone: "x" and "adj" (x_pool, adj_pool against the cotangents ``up``),
    then each loss ``loss[keys[src]]`` times ``coef[src]``; a leaf the source does not reach gets zeros."""
    grads = {}
    for src in ("x", "adj", *coef):
        if src in ("x", "adj"):
            out, cot = (xp, up[0]) if src == "x" else (ap, up[1])
            obj = (out * cot.to(out.device, out.dtype)).sum()
        else:
            obj = coef[src] * loss[keys[src]]
        g = torch.autograd.grad(obj, leaves, retain_graph=True, allow_unused=True)
        grads[src] = [torch.zeros_like(v) if gv is None else gv for gv, v in zip(g, leaves)]
    return grads


def check_per_source(got, exp, tau, edge_weight_norm):
    """max|got - ref| <= tau * max|ref| for every gradient of every source."""
    for src in exp:
        for name, gv, ev in zip(("dX", "dA", "dS"), got[src], exp[src]):
            gv, ev = gv.double(), ev.double()
            if name == "dA" and src == "adj" and edge_weight_norm:
                # max-normalisation routes one term to "the" arg-max, which a symmetric adjacency ties with its mirror
                gv, ev = 0.5 * (gv + gv.transpose(1, 2)), 0.5 * (ev + ev.transpose(1, 2))
            bound = tau * float(ev.abs().max())
            err = float((gv - ev).abs().max())
            assert err <= bound, f"{src} -> {name}: max error {err:.3e} > {bound:.3e}"


def assert_deterministic(step, tensors):
    """Three calls of ``step()`` give bit-identical outputs and ``.grad`` of each of ``tensors``."""
    runs = []
    for _ in range(3):
        out = step()
        runs.append([t.detach().clone() for t in out] + [t.grad.clone() for t in tensors])
    for r in runs[1:]:
        for u, v in zip(r, runs[0]):
            assert torch.equal(u, v)


def assert_replay_matches_eager(step, tensors):
    """``step()`` captured as one CUDA graph and replayed gives the eager call's outputs and ``.grad`` of each of
    ``tensors``, bit for bit.  ``step`` clears those gradients first, so that the capture allocates them."""
    eager = [t.detach().clone() for t in step()] + [t.grad.clone() for t in tensors]
    graphed = T.GraphedStep(step)
    out = graphed.replay()
    torch.cuda.synchronize()
    for got, exp in zip([*out, *(t.grad for t in tensors)], eager):
        assert torch.equal(got.detach(), exp)


def check_patched_pooler(pooler_cls, oracle_pool, oracle_device, keys, select_output=T.SelectOutput):
    """``pooler_cls`` patched with an MLP selector (softmax(linear(x)) * mask, its output wrapped by
    ``select_output(s=...)``) on a masked, ragged batch, against ``oracle_pool(x, a, s, mask)`` in float64 on
    ``oracle_device``: the loss keys, the losses, x_pool and the gradient of x."""
    g = torch.Generator().manual_seed(11)
    B, N, K, F = 5, 96, 16, 40
    x, a, _, mask = planted_partition(B, N, K, F, seed=11)
    wsel = torch.randn(F, K, generator=g)

    def select(x, mask):  # MLPSelect: softmax(linear(x)) * mask
        return select_output(s=torch.softmax(x @ wsel.to(x.device), -1) * mask[..., None])

    pooler = pooler_cls(selector=select, reducer=H.BaseReduce(), connector=H.DenseConnect(True, True, True, False))
    T.patch_pooler(pooler)
    xg = x.to(DEV).requires_grad_(True)
    out = pooler(x=xg, adj=a.to(DEV), mask=mask.to(DEV))
    xc = x.to(oracle_device, torch.float64).requires_grad_(True)
    mc = mask.to(oracle_device)
    s_c = torch.softmax(xc @ wsel.to(oracle_device, torch.float64), -1) * mc[..., None]
    xp_c, ap_c, loss_c = oracle_pool(xc, a.to(oracle_device, torch.float64), s_c, mc)
    assert set(out.loss) == set(keys) == set(loss_c)
    for k in loss_c:
        # an MLP assignment leaves the modularity near zero: DMoN's spectral loss is a small residue, hence the atol
        torch.testing.assert_close(out.loss[k].detach().to(oracle_device).double(), loss_c[k].detach(), rtol=1e-5,
                                   atol=1e-6, msg=k)
    sc = lambda t: float(t.abs().max())  # noqa: E731
    torch.testing.assert_close(out.x.detach().to(oracle_device).double(), xp_c.detach(), rtol=1e-5,
                               atol=1e-5 * sc(xp_c))
    (out.x.sum() + out.edge_index.sum() + sum(out.loss.values())).backward()
    (xp_c.sum() + ap_c.sum() + sum(loss_c.values())).backward()
    torch.testing.assert_close(xg.grad.to(oracle_device).double(), xc.grad, rtol=1e-4, atol=1e-5 * sc(xc.grad))
