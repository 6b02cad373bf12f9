"""GPU parity tests added in round 2: bf16 forward + backward of the dense poolers, the link loss when A ~ S S^T,
component-wise fp32 bounds, determinism of the normalised sparse path (forward + backward), BASELINE-shaped sparse
inputs (power-law hub, 128-graph batch), the no-host-read (padded) connect and CUDA-graph replay of whole steps.

Bounds used here (also tabulated in DESIGN.md section 2):
* integer outputs (edge_index, order, batch vectors, counts): bit-exact;
* fp32 sums: |got - ref| <= 1e-5 * (sum of |terms| of that output element) -- the component-wise form of
  "rtol 1e-5" for a sum that may cancel (two correct fp32 implementations differ by exactly this kind of amount);
  scalars (losses) and cancellation-free outputs: plain rtol 1e-5;
* bf16: rtol 2e-2 against the fp32 oracle on bf16-rounded inputs, absolute floor 2e-2 * max|ref| of the tensor.
"""
import os
import sys

import pytest
import torch

import tgp_b200 as T
from tgp_b200 import functional as F_
from oracle import ref_path as R

pytestmark = pytest.mark.gpu
DEV = "cuda"
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def close_bf16(got, ref, name):
    scale = float(ref.abs().max()) if ref.numel() else 1.0
    torch.testing.assert_close(got.float().cpu(), ref.float(), rtol=2e-2, atol=2e-2 * max(scale, 1e-30),
                               msg=lambda m: f"{name}: {m}")


def close_cw(got, ref, cond, name, rtol=1e-5):
    """component-wise bound: |got - ref| <= rtol * cond (cond = sum of the absolute values of the terms)."""
    err = (got.double().cpu() - ref.double()).abs()
    bound = rtol * cond.double() + 1e-30
    bad = err > bound
    assert not bool(bad.any()), f"{name}: {int(bad.sum())} elements beyond {rtol} * cond, worst ratio " \
                                f"{float((err / bound).max()):.3f}"


def _dense_inputs(g, B, N, K, F, p=0.1):
    a = (torch.rand(B, N, N, generator=g) < p).float()
    a = torch.triu(a, 1)
    a = a + a.transpose(1, 2)
    return a, torch.randn(B, N, K, generator=g), torch.randn(B, N, F, generator=g)


# --------------------------------------------------------------------------- #
# (i) bf16 forward + backward, incl. the K = 256 shapes of C3 level 1
# --------------------------------------------------------------------------- #
@pytest.mark.parametrize("B,N,K,F", [(4, 512, 256, 256), (4, 256, 64, 256), (3, 128, 32, 64), (2, 64, 16, 256),
                                     # K = 256: the fused forward does not fit, the per-product launches run
                                     (2, 256, 256, 256), (3, 512, 256, 512)])
@pytest.mark.parametrize("kind", ["mincut", "diff"])
def test_dense_pool_bf16_forward_backward(B, N, K, F, kind):
    g = torch.Generator().manual_seed(B * N + K + len(kind))
    a, s_raw, x = _dense_inputs(g, B, N, K, F, p=0.05)
    s = torch.softmax(s_raw, -1).bfloat16()
    xb, ab = x.bfloat16(), a.bfloat16()
    gx = torch.randn(B, K, F, generator=g).bfloat16()
    ga = torch.randn(B, K, K, generator=g).bfloat16()

    def run(mod, dev, dt):
        ss = s.to(dev, dt).requires_grad_(True)
        xx = xb.to(dev, dt).requires_grad_(True)
        aa = ab.to(dev, dt).requires_grad_(True)
        fn = mod.mincut_pool if kind == "mincut" else mod.diff_pool
        xp, ap, loss = fn(xx, aa, ss)
        tot = (xp.float() * gx.to(dev).float()).sum() + (ap.float() * ga.to(dev).float()).sum()
        tot = tot + sum(v.float() for v in loss.values())
        tot.backward()
        return [t.detach().float().cpu() for t in (xp, ap, *loss.values(), ss.grad, xx.grad, aa.grad)]

    exp = run(R, "cpu", torch.float32)
    got = run(T, DEV, torch.bfloat16)
    for n_, e_, g_ in zip(["x_pool", "adj_pool", "loss0", "loss1", "grad_s", "grad_x", "grad_adj"], exp, got):
        close_bf16(g_, e_, f"{kind} bf16 {(B, N, K, F)} {n_}")


# --------------------------------------------------------------------------- #
# (ii) link loss when the assignment reproduces the adjacency (A ~ S S^T)
# --------------------------------------------------------------------------- #
@pytest.mark.parametrize("noise", [0.0, 1e-3, 3e-2, 0.3])
@pytest.mark.parametrize("dt", [torch.float32, torch.bfloat16])
def test_link_loss_small_residual(noise, dt):
    g = torch.Generator().manual_seed(int(noise * 1e4) + 5)
    B, N, K, F = 3, 192, 24, 32
    blocks = torch.randint(0, K, (B, N), generator=g)
    s = torch.nn.functional.one_hot(blocks, K).float()          # hard, block-structured assignment
    a = s @ s.transpose(1, 2)                                    # A = S S^T exactly (block diagonal of ones)
    pert = torch.rand(B, N, N, generator=g) < 0.5
    a = (a + noise * (pert | pert.transpose(1, 2)).float()).to(dt)
    s, x = s.to(dt), torch.randn(B, N, F, generator=g).to(dt)
    ref = torch.linalg.norm(a.double() - s.double() @ s.double().transpose(1, 2))     # losses.py:674-676
    _, _, loss = T.diff_pool(x.to(DEV), a.to(DEV), s.to(DEV), normalize_loss=False)
    got = float(loss["link_loss"])
    na = float(torch.linalg.norm(a.double()))
    rtol = 1e-5 if dt == torch.float32 else 2e-2
    if float(ref) == 0.0:
        assert got <= 1e-6 * na, (got, na)
    else:
        assert abs(got - float(ref)) <= rtol * float(ref), (got, float(ref), na)


# --------------------------------------------------------------------------- #
# (iii) fp32 with component-wise bounds, against the fp32 AND the float64 oracle
# --------------------------------------------------------------------------- #
@pytest.mark.parametrize("B,N,K,F", [(3, 256, 64, 128), (4, 100, 16, 33)])
def test_dense_fp32_componentwise_bounds(B, N, K, F):
    g = torch.Generator().manual_seed(91 + N)
    a, s_raw, x = _dense_inputs(g, B, N, K, F)
    a = a * (torch.rand(B, N, N, generator=g) + 0.5)
    a = 0.5 * (a + a.transpose(1, 2))
    s = torch.softmax(s_raw, -1)
    gx = torch.randn(B, K, F, generator=g)
    kw = dict(remove_self_loops=False, degree_norm=False)

    def run(mod, dev, dtp):
        ss = s.to(dev, dtp).requires_grad_(True)
        xx = x.to(dev, dtp).requires_grad_(True)
        xp, ap, loss = mod.mincut_pool(xx, a.to(dev, dtp), ss, **kw)
        ((xp * gx.to(dev, dtp)).sum()).backward()
        return xp.detach().cpu(), ap.detach().cpu(), {k: v.detach().cpu() for k, v in loss.items()}, xx.grad.cpu()

    got = run(T, DEV, torch.float32)
    cond_xp = s.abs().transpose(1, 2).double() @ x.abs().double()
    cond_ap = s.abs().transpose(1, 2).double() @ a.abs().double() @ s.abs().double()
    cond_dx = s.abs().double() @ gx.abs().double()
    for dtp in (torch.float64, torch.float32):
        exp = run(R, "cpu", dtp)
        close_cw(got[0], exp[0], cond_xp, f"x_pool vs {dtp}")
        close_cw(got[1], exp[1], cond_ap, f"S^T A S vs {dtp}")
        close_cw(got[3], exp[3], cond_dx, f"dX vs {dtp}")
        for k in exp[2]:
            torch.testing.assert_close(got[2][k].double(), exp[2][k].double(), rtol=1e-5, atol=0.0, msg=k)


# --------------------------------------------------------------------------- #
# fused dense backward (one launch, W = A S in tensor memory) against the one-product-per-launch chain
@pytest.mark.parametrize("B,N,K,F", [(3, 256, 64, 128), (2, 384, 64, 128), (5, 200, 48, 100), (4, 128, 16, 64), (2, 96, 64, 36)])
@pytest.mark.parametrize("kind", ["mincut", "diff", "plain"])
def test_fused_dense_backward_matches_product_chain(B, N, K, F, kind, monkeypatch):
    g = torch.Generator().manual_seed(7 * N + K)
    a, s_raw, x = _dense_inputs(g, B, N, K, F)
    a = a * (torch.rand(B, N, N, generator=g) + 0.5)  # weighted, not symmetric
    s = torch.softmax(s_raw, -1)
    gx, ga = torch.randn(B, K, F, generator=g).to(DEV), torch.randn(B, K, K, generator=g).to(DEV)

    def run(fused):
        monkeypatch.setenv("TGPB200_BWD_FUSED", "1" if fused else "0")
        ss = s.to(DEV).requires_grad_(True)
        xx = x.to(DEV).requires_grad_(True)
        if kind == "mincut":
            xp, ap, loss = T.mincut_pool(xx, a.to(DEV), ss)
        elif kind == "diff":
            xp, ap, loss = T.diff_pool(xx, a.to(DEV), ss)
        else:
            xp, ap, loss = T.mincut_pool(xx, a.to(DEV), ss, remove_self_loops=False, degree_norm=False)
            loss = {}
        total = (xp * gx).sum() + (ap * ga).sum()
        for v in loss.values():
            total = total + v
        total.backward()
        torch.cuda.synchronize()
        return ss.grad.clone(), xx.grad.clone()

    ds0, dx0 = run(False)
    ds1, dx1 = run(True)
    # same 3xTF32 products, different accumulation grouping: a few fp32 ulps of the largest partial sums
    for got, ref, name in ((ds1, ds0, "dS"), (dx1, dx0, "dX")):
        scale = float(ref.abs().max())
        torch.testing.assert_close(got, ref, rtol=2e-6, atol=2e-6 * scale, msg=lambda m: f"{name}: {m}")


def test_sparse_weights_gradients_rtol_1e5():
    """kept-node + cluster paths: pooled features bit-identical to the sequential CPU sums, edge weights and all
    gradients at rtol 1e-5 (component-wise floor for the degree-normalised sums)."""
    g = torch.Generator().manual_seed(3)
    n, e, K = 3000, 40_000, 700
    ei = torch.randint(0, n, (2, e), generator=g)
    ei = ei[:, torch.argsort(ei[0] * n + ei[1], stable=True)]
    ew = torch.rand(e, generator=g) + 0.5
    x = torch.randn(n, 32, generator=g)
    cluster = torch.randint(0, K, (n,), generator=g)
    for op in ("sum", "mean", "max", "min", "mul"):
        wc = (ew if op != "mul" else 0.9 + 0.2 * torch.rand(e, generator=g)).clone().double().requires_grad_(True)
        so_c = R.OracleSelectOutput(cluster_index=cluster, num_supernodes=K)
        eo, wo = R.sparse_connect_so(ei, so_c, edge_weight=wc, reduce_op=op)
        coef = torch.randn(wo.numel(), generator=g).double()
        (wo * coef).sum().backward()
        wg = wc.detach().float().to(DEV).requires_grad_(True)
        so_g = T.SelectOutput(cluster_index=cluster.to(DEV), num_supernodes=K)
        eg, wgo = T.B200SparseConnect(op)(ei.to(DEV), so_g, edge_weight=wg)
        assert torch.equal(eg.cpu(), eo)
        (wgo * coef.float().to(DEV)).sum().backward()
        torch.testing.assert_close(wgo.detach().cpu().double(), wo.detach(), rtol=2e-5, atol=1e-6, msg=op)
        torch.testing.assert_close(wg.grad.cpu().double(), wc.grad, rtol=2e-5, atol=1e-6, msg=f"{op} grad")


# --------------------------------------------------------------------------- #
# (iv) determinism incl. both normalisations and the backward; unsorted rows take the sort-grouped sums
# --------------------------------------------------------------------------- #
@pytest.mark.parametrize("sorted_rows", [True, False])
@pytest.mark.parametrize("path", ["kept", "cluster"])
def test_determinism_with_normalisations_and_backward(sorted_rows, path):
    g = torch.Generator().manual_seed(17)
    n, e, K, G = 20_000, 300_000, 5_000, 8
    ei = torch.randint(0, n, (2, e), generator=g)
    if sorted_rows:
        ei = ei[:, torch.argsort(ei[0] * n + ei[1], stable=True)]
    ew = torch.rand(e, generator=g) + 0.5
    batch = torch.sort(torch.randint(0, G, (n,), generator=g))[0]
    if path == "kept":
        so_c = R.topk_select(torch.randn(n, generator=g), None, 0.5, batch)
        so_args = dict(s=so_c.s.to(DEV))
    else:
        cluster = torch.randint(0, K, (n,), generator=g)
        so_c = R.OracleSelectOutput(cluster_index=cluster, num_supernodes=K)
        so_args = dict(cluster_index=cluster.to(DEV), num_supernodes=K)
    bp_c = R.reduce_batch(so_c, batch)
    outs = []
    for _ in range(3):
        so = T.SelectOutput(**so_args)
        w = ew.to(DEV).requires_grad_(True)
        bp = T.Reduce.reduce_batch(so, batch.to(DEV))
        eo, wo = T.B200SparseConnect(degree_norm=True, edge_weight_norm=True)(ei.to(DEV), so, edge_weight=w,
                                                                              batch_pooled=bp)
        (wo * torch.arange(1, wo.numel() + 1, device=DEV).float().sqrt()).sum().backward()
        outs.append((eo, wo.detach(), w.grad))
    for a, b in zip(outs[0], outs[1]):
        assert torch.equal(a, b)
    for a, b in zip(outs[0], outs[2]):
        assert torch.equal(a, b)
    # and the values are the oracle's
    wc = ew.clone().requires_grad_(True)
    e_ref, w_ref = R.sparse_connect_so(ei, so_c, edge_weight=wc, batch_pooled=bp_c, degree_norm=True,
                                       edge_weight_norm=True)
    (w_ref * torch.arange(1, w_ref.numel() + 1).float().sqrt()).sum().backward()
    assert torch.equal(outs[0][0].cpu(), e_ref)
    torch.testing.assert_close(outs[0][1].cpu(), w_ref.detach(), rtol=1e-5, atol=1e-7)
    scale = float(wc.grad.abs().max())
    torch.testing.assert_close(outs[0][2].cpu(), wc.grad, rtol=1e-4, atol=1e-5 * scale)


# --------------------------------------------------------------------------- #
# (v) BASELINE-shaped sparse inputs: a power-law hub (one coarse edge with > 1e5 duplicates), the 128-graph C1 batch
# --------------------------------------------------------------------------- #
def test_cluster_connect_powerlaw_hub():
    g = torch.Generator().manual_seed(23)
    n, spokes, K = 200_000, 150_000, 1000
    hub = torch.zeros(spokes, dtype=torch.long)
    leaves = torch.arange(1, spokes + 1)
    rnd = torch.randint(0, n, (2, 300_000), generator=g)
    ei = torch.cat([torch.stack([hub, leaves]), torch.stack([leaves, hub]), rnd], 1)
    ei = ei[:, torch.argsort(ei[0] * n + ei[1], stable=True)]
    cluster = torch.randint(2, K, (n,), generator=g)
    cluster[0] = 0
    cluster[1:spokes + 1] = 1                              # coarse edges (0,1) and (1,0): 150 000 duplicates each
    ew = torch.rand(ei.size(1), generator=g) + 0.5
    so_c = R.OracleSelectOutput(cluster_index=cluster, num_supernodes=K)
    so_g = T.SelectOutput(cluster_index=cluster.to(DEV), num_supernodes=K)
    for op in ("sum", "max", "mean"):
        eo, wo = R.sparse_connect_so(ei, so_c, edge_weight=ew, reduce_op=op)
        eg, wg = T.B200SparseConnect(op)(ei.to(DEV), so_g, edge_weight=ew.to(DEV))
        assert torch.equal(eg.cpu(), eo)
        torch.testing.assert_close(wg.cpu(), wo, rtol=1e-5, atol=1e-7, msg=op)
    # degree normalisation over a 150 000-edge row: unit weights make every partial sum exact in fp32
    eo, wo = R.sparse_connect_so(ei, so_c, edge_weight=torch.ones_like(ew), degree_norm=True)
    eg, wg = T.B200SparseConnect(degree_norm=True)(ei.to(DEV), so_g, edge_weight=torch.ones_like(ew).to(DEV))
    assert torch.equal(eg.cpu(), eo)
    torch.testing.assert_close(wg.cpu(), wo, rtol=1e-5, atol=1e-9)
    # unweighted: duplicates dropped
    eo, wo = R.sparse_connect_so(ei, so_c)
    eg, wg = T.B200SparseConnect()(ei.to(DEV), so_g)
    assert wg is None and wo is None and torch.equal(eg.cpu(), eo)


def _c1_batch():
    sys.path.insert(0, ROOT)
    import bench

    return bench.er_batch(bench.SPARSE["c1"], 0)


def test_c1_batch_topk_pool_parity_padded_and_graph_replay():
    ei, batch, N = _c1_batch()
    g = torch.Generator().manual_seed(0)
    x = torch.randn(N, 64, generator=g)
    p = torch.randn(1, 64, generator=g)
    ew = torch.rand(ei.size(1), generator=g) + 0.5
    so_c = R.topk_select(x, p, 0.5, batch)
    so_g = T.topk_select(x.to(DEV), p.to(DEV), 0.5, batch.to(DEV), num_graphs=128)
    assert torch.equal(so_g.node_index.cpu(), so_c.node_index)
    assert torch.equal(so_g.cluster_index.cpu(), so_c.cluster_index)
    for dn, ewn in ((False, False), (True, True)):
        xc, wc = x.clone().requires_grad_(True), ew.clone().requires_grad_(True)
        xp_c, ei_c, ew_c, bp_c = R.topk_pool(xc, ei, wc, so_c, batch=batch, degree_norm=dn, edge_weight_norm=ewn)
        (xp_c.sum() + (ew_c * torch.arange(1, ew_c.numel() + 1)).sum()).backward()
        so = T.SelectOutput(s=so_c.s.detach().to(DEV))
        xg, wg = x.to(DEV).requires_grad_(True), ew.to(DEV).requires_grad_(True)
        xp, eo, wo, bp = T.sparse_pool(xg, ei.to(DEV), so, edge_weight=wg, batch=batch.to(DEV), degree_norm=dn,
                                       edge_weight_norm=ewn)
        (xp.sum() + (wo * torch.arange(1, wo.numel() + 1, device=DEV)).sum()).backward()
        assert torch.equal(eo.cpu(), ei_c) and torch.equal(bp.cpu(), bp_c)
        assert torch.equal(xp.detach().cpu(), xp_c.detach())
        torch.testing.assert_close(wo.detach().cpu(), ew_c.detach(), rtol=1e-5, atol=1e-7)
        torch.testing.assert_close(xg.grad.cpu(), xc.grad, rtol=1e-5, atol=1e-7)
        sc = float(wc.grad.abs().max())
        torch.testing.assert_close(wg.grad.cpu(), wc.grad, rtol=1e-4, atol=1e-5 * sc)
        # the no-host-read form: same values in the first `count` columns
        xg2, wg2 = x.to(DEV).requires_grad_(True), ew.to(DEV).requires_grad_(True)
        so2 = T.SelectOutput(s=so_c.s.detach().to(DEV))
        E = ei.size(1)
        coef = torch.zeros(E, device=DEV)
        coef[: wo.numel()] = torch.arange(1, wo.numel() + 1, device=DEV).float()
        ei_d, batch_d = ei.to(DEV), batch.to(DEV)

        def step():
            xg2.grad = None
            wg2.grad = None
            so2._b200_csr = None
            xp2, e2, w2, bp2, cnt = T.sparse_pool_padded(xg2, ei_d, so2, edge_weight=wg2, batch=batch_d,
                                                         degree_norm=dn, edge_weight_norm=ewn, num_graphs=128)
            torch.autograd.backward([xp2, w2], [torch.ones_like(xp2), coef])
            return xp2, e2, w2, bp2, cnt

        xp2, e2, w2, bp2, cnt = step()
        n_out = int(cnt)
        assert n_out == eo.size(1) and torch.equal(e2[:, :n_out], eo) and torch.equal(bp2, bp)
        assert torch.equal(w2[:n_out].detach(), wo.detach()) and torch.equal(xp2.detach(), xp.detach())
        assert torch.equal(wg2.grad, wg.grad) and torch.equal(xg2.grad, xg.grad)
        # ... and replayed as one CUDA graph (the eager outputs must be released first: they keep the autograd
        # graph, and with it AccumulateGrad nodes bound to the default stream, alive across the capture)
        del xp2, e2, w2, bp2, cnt
        graphed = T.GraphedStep(step)
        wg2.grad.zero_()
        xp3, e3, w3, bp3, cnt3 = graphed.replay()
        torch.cuda.synchronize()
        assert int(cnt3) == n_out and torch.equal(e3[:, :n_out], eo) and torch.equal(w3[:n_out].detach(), wo.detach())
        assert torch.equal(wg2.grad, wg.grad) and torch.equal(xg2.grad, xg.grad) and torch.equal(xp3.detach(), xp.detach())
        assert graphed.kernels_per_replay > 0


@pytest.mark.parametrize("op", ["sum", "mean"])
def test_cluster_pool_padded_and_graph_replay(op):
    """Cluster branch (row-bucketed coalesce incl. hub rows) in the no-host-read form: same coarse edges, weights and
    gradients as the exact-size call in the first `count` columns, eagerly and replayed as one CUDA graph."""
    g = torch.Generator().manual_seed(31)
    n, spokes, K, F = 20_000, 3_000, 700, 32
    hub = torch.zeros(spokes, dtype=torch.long)
    leaves = torch.arange(1, spokes + 1)
    rnd = torch.randint(0, n, (2, 80_000), generator=g)
    ei = torch.cat([torch.stack([hub, leaves]), torch.stack([leaves, hub]), rnd], 1)
    ei = ei[:, torch.argsort(ei[0] * n + ei[1], stable=True)].to(DEV)
    cluster = torch.randint(2, K, (n,), generator=g)
    cluster[0] = 0
    cluster[1:spokes + 1] = 1
    E = ei.size(1)
    x0, w0 = torch.randn(n, F, generator=g).to(DEV), (torch.rand(E, generator=g) + 0.5).to(DEV)
    so = T.SelectOutput(cluster_index=cluster.to(DEV), num_nodes=n, num_supernodes=K)
    xg, wg = x0.clone().requires_grad_(True), w0.clone().requires_grad_(True)
    xp, eo, wo, _ = T.sparse_pool(xg, ei, so, edge_weight=wg, reduce_op="mean", connect_op=op)
    n_out = eo.size(1)
    coef = torch.zeros(E, device=DEV)
    coef[:n_out] = torch.arange(1, n_out + 1, device=DEV).float().sqrt()
    torch.autograd.backward([xp, wo], [torch.ones_like(xp), coef[:n_out]])
    xg2, wg2 = x0.clone().requires_grad_(True), w0.clone().requires_grad_(True)

    def step():
        xg2.grad = None
        wg2.grad = None
        xp2, e2, w2, _, cnt = T.sparse_pool_padded(xg2, ei, so, edge_weight=wg2, reduce_op="mean", connect_op=op)
        torch.autograd.backward([xp2, w2], [torch.ones_like(xp2), coef])
        return xp2, e2, w2, cnt

    xp2, e2, w2, cnt = step()
    assert int(cnt) == n_out and torch.equal(e2[:, :n_out], eo)
    assert torch.equal(w2[:n_out].detach(), wo.detach()) and torch.equal(xp2.detach(), xp.detach())
    assert torch.equal(wg2.grad, wg.grad) and torch.equal(xg2.grad, xg.grad)
    del xp2, e2, w2, cnt
    graphed = T.GraphedStep(step)
    wg2.grad.zero_()
    xp3, e3, w3, cnt3 = graphed.replay()
    torch.cuda.synchronize()
    assert int(cnt3) == n_out and torch.equal(e3[:, :n_out], eo) and torch.equal(w3[:n_out].detach(), wo.detach())
    assert torch.equal(wg2.grad, wg.grad) and torch.equal(xg2.grad, xg.grad) and torch.equal(xp3.detach(), xp.detach())


def test_dense_step_graph_replay_matches_eager():
    g = torch.Generator().manual_seed(2)
    B, N, K, F = 6, 256, 64, 128
    a, s_raw, x = _dense_inputs(g, B, N, K, F)
    a, x = a.to(DEV), x.to(DEV).requires_grad_(True)
    s = torch.softmax(s_raw, -1).to(DEV).requires_grad_(True)
    gx, ga = torch.randn(B, K, F, generator=g).to(DEV), torch.randn(B, K, K, generator=g).to(DEV)
    gl = torch.tensor([1.0, 1.0, 0.0, 0.0], device=DEV)

    def step():
        x.grad = None
        s.grad = None
        xp, ap, losses = F_.dense_pool(x, a, s, remove_self_loops=True, degree_norm=True, adj_transpose=True,
                                       loss_kind=F_.LOSS_MINCUT)
        torch.autograd.backward([xp, ap, losses], [gx, ga, gl])
        return xp, ap, losses

    eager = [t.detach().clone() for t in step()] + [x.grad.clone(), s.grad.clone()]
    graphed = T.GraphedStep(step)
    x0 = x.detach().clone()
    with torch.no_grad():
        x.copy_(torch.randn_like(x0))  # new data in the static input buffer ...
    graphed.replay()
    assert not torch.equal(graphed.outputs[0].detach(), eager[0])
    with torch.no_grad():
        x.copy_(x0)  # ... and the original data again: the replay must reproduce the eager step bit for bit
    out = graphed.replay()
    torch.cuda.synchronize()
    for got, exp in zip([*out, x.grad, s.grad], eager):
        assert torch.equal(got.detach(), exp)
    assert graphed.kernels_per_replay >= 5


def test_segment_reduce_unsorted_node_index_raises():
    x = torch.randn(10, 4, device=DEV, requires_grad=True)
    node = torch.tensor([3, 1, 2], device=DEV)
    with pytest.raises(ValueError):
        F_.segment_reduce(x, node, torch.tensor([0, 1, 1], device=DEV), None, 2).sum().backward()


# --------------------------------------------------------------------------- #
# pooler-level drop-in: patch_pooler on stand-ins of the reference poolers, called with the reference's kwargs
# --------------------------------------------------------------------------- #
def test_patched_topk_pooler_matches_oracle():
    import dropin_harness as H

    ei, batch, N = _c1_batch()
    g = torch.Generator().manual_seed(1)
    x = torch.randn(N, 64, generator=g)
    p = torch.randn(1, 64, generator=g)
    ew = torch.rand(ei.size(1), generator=g) + 0.5
    pooler = H.TopkPooling(selector=lambda x, batch: T.topk_select(x, p.to(DEV), 0.5, batch, num_graphs=128),
                           reducer=H.BaseReduce(), connector=H.SparseConnect("sum", True, True, True))
    T.patch_pooler(pooler)
    xp, eo, wo, bp, so = pooler(x=x.to(DEV), adj=ei.to(DEV), edge_weight=ew.to(DEV), batch=batch.to(DEV))
    so_c = R.topk_select(x, p, 0.5, batch)
    xp_c, ei_c, ew_c, bp_c = R.topk_pool(x, ei, ew, so_c, batch=batch, degree_norm=True, edge_weight_norm=True)
    assert torch.equal(eo.cpu(), ei_c) and torch.equal(bp.cpu(), bp_c)
    torch.testing.assert_close(xp.cpu(), xp_c, rtol=1e-5, atol=1e-6)
    torch.testing.assert_close(wo.cpu(), ew_c, rtol=1e-5, atol=1e-7)


@pytest.mark.parametrize("kind", ["mincut", "diff"])
def test_patched_dense_pooler_fused_forward_matches_oracle(kind):
    import dropin_harness as H

    g = torch.Generator().manual_seed(4)
    B, N, K, F = 5, 96, 16, 40
    a, s_raw, x = _dense_inputs(g, B, N, K, F)
    mask = torch.ones(B, N, dtype=torch.bool)
    mask[1, 80:] = False
    mask[3, 50:] = False
    a = a * (mask[:, :, None] & mask[:, None, :])
    wsel = torch.randn(F, K, generator=g)

    def select(x, mask):  # MLPSelect (tgp/select/mlp_select.py:120-150): softmax(linear(x)) * mask
        s = torch.softmax(x @ wsel.to(x.device), -1) * mask[..., None]
        return (T.SelectOutput if x.is_cuda else R.OracleSelectOutput)(s=s)

    cls = H.MinCutPooling if kind == "mincut" else H.DiffPool
    pooler = cls(selector=select, reducer=H.BaseReduce(), connector=H.DenseConnect(True, True, True, False, False))
    T.patch_pooler(pooler)
    xg = x.to(DEV).requires_grad_(True)
    out = pooler(x=xg, adj=a.to(DEV), mask=mask.to(DEV))
    xc = x.clone().requires_grad_(True)
    s_c = torch.softmax(xc @ wsel, -1) * mask[..., None]
    if kind == "mincut":
        xp_c, ap_c, loss_c = R.mincut_pool(xc, a, s_c, cut_loss_coeff=0.7, ortho_loss_coeff=1.3)
    else:
        xp_c, ap_c, loss_c = R.diff_pool(xc, a, s_c, num_nodes=int(mask.sum()), link_loss_coeff=0.5,
                                         ent_loss_coeff=2.0, normalize_loss=False)
    sc = lambda t: float(t.abs().max())
    torch.testing.assert_close(out.x.detach().cpu(), xp_c.detach(), rtol=1e-5, atol=1e-5 * sc(xp_c))
    torch.testing.assert_close(out.edge_index.detach().cpu(), ap_c.detach(), rtol=1e-5, atol=1e-5 * sc(ap_c))
    assert set(out.loss) == set(loss_c)
    for k in loss_c:
        torch.testing.assert_close(out.loss[k].detach().cpu(), loss_c[k].detach(), rtol=1e-5, atol=1e-7, msg=k)
    (out.x.sum() + out.edge_index.sum() + sum(out.loss.values())).backward()
    (xp_c.sum() + ap_c.sum() + sum(loss_c.values())).backward()
    torch.testing.assert_close(xg.grad.cpu(), xc.grad, rtol=1e-4, atol=1e-5 * sc(xc.grad))


def test_postprocess_adj_pool_dense_standalone():
    from tgp_b200.connect import postprocess_adj_pool_dense

    g = torch.Generator().manual_seed(9)
    ap = torch.rand(4, 24, 24, generator=g) + 0.1
    for rsl, dn, tr, ewn in [(True, True, True, False), (False, True, False, True), (True, False, True, True)]:
        exp = R.postprocess_adj_pool_dense(ap.clone(), remove_self_loops=rsl, degree_norm=dn, adj_transpose=tr,
                                           edge_weight_norm=ewn)
        got = postprocess_adj_pool_dense(ap.to(DEV), remove_self_loops=rsl, degree_norm=dn, adj_transpose=tr,
                                         edge_weight_norm=ewn)
        torch.testing.assert_close(got.cpu(), exp, rtol=1e-5, atol=1e-6)


def test_lift_dense_off_grid_shapes_and_multigraph():
    g = torch.Generator().manual_seed(10)
    B, N, K, F = 3, 50, 10, 7  # K, F not multiples of 4: the tensor-core engine declines, the FP32-pipe tiles take over
    s = torch.softmax(torch.randn(B, N, K, generator=g), -1)
    xp = torch.randn(B, K, F, generator=g)
    sg, xg = s.to(DEV).requires_grad_(True), xp.to(DEV).requires_grad_(True)
    out = T.B200Lift()(xg, T.SelectOutput(s=sg))
    out.sum().backward()
    torch.testing.assert_close(out.detach().cpu(), s @ xp, rtol=1e-5, atol=1e-5)
    torch.testing.assert_close(sg.grad.cpu(), torch.ones(B, N, F) @ xp.transpose(1, 2), rtol=1e-5, atol=1e-5)
    torch.testing.assert_close(xg.grad.cpu(), s.transpose(1, 2) @ torch.ones(B, N, F), rtol=1e-5, atol=1e-5)
    # dense [N, K] assignment over a multi-graph batch
    sizes = [5, 9, 3]
    batch = torch.cat([torch.full((n,), i) for i, n in enumerate(sizes)])
    s2 = torch.softmax(torch.randn(sum(sizes), K, generator=g), -1)
    xp2 = torch.randn(len(sizes) * K, F, generator=g)
    got = T.B200Lift()(xp2.to(DEV), T.SelectOutput(s=s2.to(DEV), batch=batch.to(DEV)), batch=batch.to(DEV))
    exp = torch.cat([s2[batch == i] @ xp2[i * K:(i + 1) * K] for i in range(len(sizes))])
    torch.testing.assert_close(got.cpu(), exp, rtol=1e-5, atol=1e-5)
    with pytest.raises(ValueError):
        T.B200Lift(reduce_op="max")


# --------------------------------------------------------------------------- #
# row-bucketed coalesce (row-sorted inputs): tiles, hub rows, long runs, isolated nodes, empty clusters
# --------------------------------------------------------------------------- #
@pytest.mark.parametrize("n,e,K", [(5000, 200_000, 3), (5000, 200_000, 40), (60_000, 900_000, 25_000),
                                   (300_000, 700_000, 290_000), (2_000, 30, 1_500), (70_000, 2_000_000, 70_000)])
@pytest.mark.parametrize("weighted", [True, False])
def test_bucketed_coalesce_matches_oracle(n, e, K, weighted):
    g = torch.Generator().manual_seed(n + e + K)
    ei = torch.randint(0, n, (2, e), generator=g)
    ei[:, : e // 50] = ei[:, e // 50: 2 * (e // 50)]                     # exact duplicate edges
    ei = ei[:, torch.argsort(ei[0] * n + ei[1], stable=True)]
    cluster = torch.randint(0, max(K - K // 10, 1), (n,), generator=g)    # the last 10 % of the clusters are empty
    ew = (torch.rand(e, generator=g) + 0.5) if weighted else None
    so_c = R.OracleSelectOutput(cluster_index=cluster, num_supernodes=K)
    so_g = T.SelectOutput(cluster_index=cluster.to(DEV), num_supernodes=K)
    for op in (("sum", "mean", "max", "mul") if weighted else ("sum",)):
        w64 = None if ew is None else (ew.double() if op != "mul" else (0.98 + 0.04 * (ew.double() - 0.5)))
        eo, wo = R.sparse_connect_so(ei, so_c, edge_weight=w64, reduce_op=op)
        wg_in = None if w64 is None else w64.float().to(DEV).requires_grad_(True)
        eg, wg = T.B200SparseConnect(op)(ei.to(DEV), so_g, edge_weight=wg_in)
        assert torch.equal(eg.cpu(), eo), op
        if weighted:
            # long runs are sequential fp32 sums (like the reference's own CPU path): 2e-5 against the exact value
            # (a 20 000-term fp32 product accumulates ~1e-3 of rounding: the mul bound scales with the run length)
            torch.testing.assert_close(wg.detach().cpu().double(), wo, rtol=2e-5 if op != "mul" else 5e-3, atol=1e-6,
                                       msg=op)
            if op in ("sum", "mean"):
                wc = w64.clone().requires_grad_(True)
                _, wo2 = R.sparse_connect_so(ei, so_c, edge_weight=wc, reduce_op=op)
                coef = torch.randn(wo2.numel(), generator=g).double()
                (wo2 * coef).sum().backward()
                (wg * coef.float().to(DEV)).sum().backward()
                torch.testing.assert_close(wg_in.grad.cpu().double(), wc.grad, rtol=1e-5, atol=1e-7, msg=f"{op} grad")
        else:
            assert wg is None and wo is None


def test_bucketed_coalesce_mul_gradient_with_zero_weights():
    g = torch.Generator().manual_seed(31)
    n, e, K = 400, 6000, 30
    ei = torch.randint(0, n, (2, e), generator=g)
    ei = ei[:, torch.argsort(ei[0] * n + ei[1], stable=True)]
    cluster = torch.randint(0, K, (n,), generator=g)
    ew = 0.9 + 0.2 * torch.rand(e, generator=g)
    ew[torch.randint(0, e, (40,), generator=g)] = 0.0       # runs with one zero, with several zeros
    wc = ew.clone().double().requires_grad_(True)
    eo, wo = R.sparse_connect_so(ei, R.OracleSelectOutput(cluster_index=cluster, num_supernodes=K), edge_weight=wc,
                                 reduce_op="mul", remove_self_loops=False)
    coef = torch.randn(wo.numel(), generator=g).double()
    (wo * coef).sum().backward()
    wg = ew.to(DEV).requires_grad_(True)
    eg, wgo = T.B200SparseConnect("mul", remove_self_loops=False)(
        ei.to(DEV), T.SelectOutput(cluster_index=cluster.to(DEV), num_supernodes=K), edge_weight=wg)
    assert torch.equal(eg.cpu(), eo)
    (wgo * coef.float().to(DEV)).sum().backward()
    torch.testing.assert_close(wg.grad.cpu().double(), wc.grad, rtol=1e-4, atol=1e-9)


# --------------------------------------------------------------------------- #
# unbatched dense mode: sparse adjacency, SpMM + batched product, sparse loss twins (reference-generated golden)
# --------------------------------------------------------------------------- #
def test_unbatched_sparse_path_matches_reference_golden():
    from tgp_b200 import unbatched as U

    cases = torch.load(os.path.join(ROOT, "tests", "golden", "ref_unbatched.pt"), weights_only=False)
    for name, c in cases.items():
        ei, ew, b = c["edge_index"].to(DEV), c["edge_weight"], c["batch"]
        bg = None if b is None else b.to(DEV)
        sr = c["s_raw"].to(DEV).requires_grad_(True)
        wg = None if ew is None else ew.to(DEV).requires_grad_(True)
        s = torch.softmax(sr, -1)
        cut = U.sparse_mincut_loss(ei, s, wg, bg)
        ortho = U.unbatched_orthogonality_loss(s, bg)
        link = U.sparse_link_pred_loss(s, ei, wg, bg, normalize_loss=False)
        link_n = U.sparse_link_pred_loss(s, ei, wg, bg, normalize_loss=True)
        for got, key in ((cut, "cut"), (ortho, "ortho"), (link, "link"), (link_n, "link_norm")):
            torch.testing.assert_close(got.detach().cpu(), c[key], rtol=1e-5, atol=1e-7, msg=f"{name}:{key}")
        (cut + 0.5 * ortho + 0.25 * link).backward()
        sc = float(c["grad_s_raw"].abs().max())
        torch.testing.assert_close(sr.grad.cpu(), c["grad_s_raw"], rtol=1e-4, atol=1e-5 * sc, msg=name)
        if wg is not None:
            sc = float(c["grad_w"].abs().max())
            torch.testing.assert_close(wg.grad.cpu(), c["grad_w"], rtol=1e-4, atol=1e-5 * sc, msg=name)
        K = s.size(1)
        nb = 1 if b is None else int(b.max()) + 1
        bp = torch.arange(nb, device=DEV).repeat_interleave(K)
        so = T.SelectOutput(s=torch.softmax(c["s_raw"], -1).to(DEV), batch=bg)
        for so_flag in (False, True):
            for dn in (False, True):
                a_ref, w_ref = c[f"adj_so{int(so_flag)}_dn{int(dn)}"]
                conn = T.B200DenseConnect(True, dn, False, False, so_flag)
                a, w = conn(ei, so, edge_weight=None if ew is None else ew.to(DEV), batch=bg, batch_pooled=bp)
                if so_flag:
                    assert torch.equal(a.cpu(), a_ref), name
                    torch.testing.assert_close(w.cpu(), w_ref, rtol=1e-5, atol=1e-6)
                else:
                    torch.testing.assert_close(a.cpu(), a_ref, rtol=1e-5, atol=1e-6, msg=f"{name} dn{dn}")


def test_unbatched_mincut_pool_equals_batched_on_large_ragged_batch():
    """tests/poolers/test_dense_poolers_batched_vs_unbatched.py:36-174 at a size where the padded adjacency would be
    64x the edge list: the sparse path must agree with the batched tensor-core path (rtol 1e-5)."""
    from tgp_b200 import unbatched as U

    g = torch.Generator().manual_seed(13)
    sizes = [int(v) for v in torch.randint(40, 400, (24,), generator=g)]
    K, F = 12, 20
    batch = torch.cat([torch.full((n,), i) for i, n in enumerate(sizes)])
    N = batch.numel()
    eis, off = [], 0
    for n in sizes:
        r = torch.randint(0, n, (2, 4 * n), generator=g)
        r = r[:, r[0] != r[1]]
        eis.append(torch.cat([r, r.flip(0)], 1) + off)
        off += n
    ei = torch.cat(eis, 1)
    ei = torch.unique(ei, dim=1)  # distinct, row-sorted edges
    ew = torch.rand(ei.size(1), generator=g) + 0.5
    s = torch.softmax(torch.randn(N, K, generator=g), -1).to(DEV)
    x = torch.randn(N, F, generator=g).to(DEV)
    xp_u, ap_u, loss_u = U.mincut_pool_unbatched(x, ei.to(DEV), ew.to(DEV), s, batch.to(DEV), num_graphs=len(sizes))
    B = len(sizes)
    s3, _ = F_.to_dense_batch(s, batch.to(DEV), B)
    x3, _ = F_.to_dense_batch(x, batch.to(DEV), B, s3.size(1))
    adj = F_.to_dense_adj(ei.to(DEV), batch.to(DEV), ew.to(DEV), num_graphs=B, max_num_nodes=s3.size(1))
    xp_b, ap_b, loss_b = T.mincut_pool(x3, adj, s3, adj_transpose=False)
    sc = lambda t: float(t.abs().max())
    torch.testing.assert_close(xp_u, xp_b, rtol=1e-5, atol=1e-5 * sc(xp_b))
    torch.testing.assert_close(ap_u, ap_b, rtol=1e-5, atol=1e-5 * sc(ap_b))
    for k in loss_b:
        torch.testing.assert_close(loss_u[k], loss_b[k], rtol=2e-5, atol=1e-7, msg=k)
