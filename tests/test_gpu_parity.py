"""GPU parity tests: CUDA path (through the C ABI) vs the CPU oracle and the golden fixtures.

Bars (BASELINE.json north_star): bit-exact for cluster index, coarse edge_index, edge ordering and
TopK-driven relabelling; rtol 1e-5 (fp32) / 2e-2 (bf16) for pooled features, edge weights, losses
and gradients.
"""
import math

import pytest
import torch

import tgp_b200 as T
from tgp_b200 import functional as F_
from oracle import ref_path as R

pytestmark = pytest.mark.gpu
DEV = "cuda"
FP32 = dict(rtol=1e-5, atol=1e-6)
BF16 = dict(rtol=2e-2, atol=2e-2)


def close32(got, ref, name="", rtol=1e-5):
    """fp32 bar of the north star (rtol 1e-5), with the absolute floor tied to the tensor's own scale: entries that
    are small only through cancellation carry the rounding of their O(scale) partial sums (tensor-core fp32
    accumulation included), exactly as two fp32 matmul implementations differ from each other."""
    scale = float(ref.abs().max()) if ref.numel() else 1.0
    torch.testing.assert_close(got, ref, rtol=rtol, atol=rtol * max(scale, 1e-30), msg=lambda m: f"{name}: {m}")


def _flags(name):
    return {p[:-1]: bool(int(p[-1])) for p in name.split("_") if p[:-1] in ("dn", "ewn", "rsl", "t")}


def _cu(t):
    return None if t is None else t.to(DEV)


def test_native_library_is_loaded():
    from tgp_b200 import _lib as L

    L.load()
    maps = open("/proc/self/maps").read()
    assert "libtgp_b200.so" in maps


# --------------------------------------------------------------------------- #
# primitives through build_csr (scan + stable radix sort)
# --------------------------------------------------------------------------- #
@pytest.mark.parametrize("nnz,K", [(0, 3), (1, 1), (31, 5), (4096, 7), (4097, 300), (100_003, 65_537), (1_000_000, 17),
                                   (2_000_000, 1_100_000),
                                   # boundaries of the small-input paths: one-tile radix passes (2048 keys), the
                                   # single-block scan (32768 counters) against the one-pass look-back scan
                                   (2047, 3), (2048, 2048), (2049, 5), (50_000, 32_766), (50_000, 32_767),
                                   (50_000, 32_768), (50_000, 40_000),
                                   # the same radix boundaries above the single-block build (K > 8192)
                                   (2047, 9000), (2048, 9000), (2049, 9000),
                                   # single-block build (nnz <= 8192 and K <= 8192): chunk / warp boundaries, one
                                   # cluster holding everything, both limits and one past each
                                   (32, 1), (33, 2), (1024, 1024), (1025, 2), (5000, 8192), (8192, 1), (8192, 8192),
                                   (8193, 8192), (8192, 8193)])
def test_build_csr_matches_stable_argsort(nnz, K):
    g = torch.Generator().manual_seed(nnz + K)
    c = torch.randint(0, K, (nnz,), generator=g)
    order, ptr = F_.build_csr(c.to(DEV), K)
    exp_order = torch.sort(c, stable=True)[1].to(torch.int32)
    exp_ptr = torch.zeros(K + 1, dtype=torch.int32)
    exp_ptr[1:] = torch.bincount(c, minlength=K).cumsum(0)
    assert torch.equal(ptr.cpu(), exp_ptr)
    assert torch.equal(order.cpu()[:nnz], exp_order)


@pytest.mark.parametrize("nnz,K", [(700, 40), (8192, 8192), (20_000, 300)])
def test_build_csr_clamps_out_of_range_ids(nnz, K):
    """Ids outside [0, K) are never dereferenced: both builds (single block / radix) file them under K - 1."""
    g = torch.Generator().manual_seed(nnz)
    c = torch.randint(-3, K + 3, (nnz,), generator=g)
    order, ptr = F_.build_csr(c.to(DEV), K)
    cc = torch.where((c < 0) | (c >= K), torch.full_like(c, K - 1), c)
    exp_ptr = torch.zeros(K + 1, dtype=torch.int32)
    exp_ptr[1:] = torch.bincount(cc, minlength=K).cumsum(0)
    assert torch.equal(ptr.cpu(), exp_ptr)
    assert torch.equal(order.cpu()[:nnz], torch.sort(cc, stable=True)[1].to(torch.int32))


# --------------------------------------------------------------------------- #
# sparse reduce
# --------------------------------------------------------------------------- #
@pytest.mark.parametrize("op", ["sum", "mean", "max", "min"])
@pytest.mark.parametrize("F", [1, 3, 64, 128, 200])
def test_segment_reduce_fp32(op, F):
    g = torch.Generator().manual_seed(F)
    N, K = 500, 130
    sel = torch.randperm(N, generator=g)[:400]
    cluster = torch.randint(0, K - 5, (400,), generator=g)  # last 5 clusters empty
    w = torch.rand(400, generator=g) + 0.5
    x = torch.randn(N, F, generator=g)
    if op in ("max", "min"):  # create exact ties
        x[sel[1]] = x[sel[0]]
        cluster[1] = cluster[0]
        w[1] = w[0]
    so_c = R.OracleSelectOutput(node_index=sel, num_nodes=N, cluster_index=cluster, num_supernodes=K, weight=w)
    xc = x.clone().requires_grad_(True)
    wc = so_c.s.values().clone().requires_grad_(True)
    so_c2 = R.OracleSelectOutput(s=torch.sparse_coo_tensor(so_c.s.indices(), wc, so_c.s.shape, is_coalesced=True))
    exp, _ = (R.base_reduce(xc, so_c2) if op == "sum" else R.aggr_reduce(xc, so_c2, op))
    gout = torch.randn(K, F, generator=g)
    (exp * gout).sum().backward()

    xg = x.to(DEV).requires_grad_(True)
    wg = so_c.s.values().to(DEV).requires_grad_(True)
    so_g = T.SelectOutput(s=torch.sparse_coo_tensor(so_c.s.indices().to(DEV), wg, so_c.s.shape, is_coalesced=True))
    got, _ = T.B200Reduce(op)(xg, so_g)
    (got * gout.to(DEV)).sum().backward()
    if op == "sum":
        assert torch.equal(got.detach().cpu(), exp.detach()), "fp32 sums are sequential and must be bit-identical"
    torch.testing.assert_close(got.detach().cpu(), exp.detach(), **FP32)
    torch.testing.assert_close(xg.grad.cpu(), xc.grad, **FP32)
    torch.testing.assert_close(wg.grad.cpu(), wc.grad, rtol=1e-4, atol=1e-5)
    assert torch.all(got[K - 5:] == 0)


@pytest.mark.parametrize("op", ["sum", "mean"])
@pytest.mark.parametrize("F", [4, 128, 200])
@pytest.mark.parametrize("layout", ["hard_all", "hard_subset", "soft_multi"])
def test_segment_reduce_backward_without_weight_grad(op, F, layout):
    """sum / mean backward when only x needs a gradient (the multi-node-per-warp fast path): every node selected
    once, a subset selected (zero rows for the rest), and nodes assigned to several clusters."""
    g = torch.Generator().manual_seed(17 * F + len(layout))
    N, K = 1003, 257
    if layout == "hard_all":
        node = torch.arange(N)
    elif layout == "hard_subset":
        node = torch.sort(torch.randperm(N, generator=g)[:611]).values
    else:
        node = torch.sort(torch.randint(0, N, (2500,), generator=g)).values
    cluster = torch.randint(0, K - 3, (node.numel(),), generator=g)
    if layout == "soft_multi":  # coalesced COO: unique (node, cluster) pairs
        key = torch.unique(node * K + cluster)
        node, cluster = key // K, key % K
    w = torch.rand(node.numel(), generator=g) + 0.5
    x = torch.randn(N, F, generator=g)
    gout = torch.randn(K, F, generator=g)
    so_c = R.OracleSelectOutput(node_index=node, num_nodes=N, cluster_index=cluster, num_supernodes=K, weight=w)
    xc = x.clone().requires_grad_(True)
    exp, _ = (R.base_reduce(xc, so_c) if op == "sum" else R.aggr_reduce(xc, so_c, op))
    (exp * gout).sum().backward()
    so_g = T.SelectOutput(node_index=node.to(DEV), num_nodes=N, cluster_index=cluster.to(DEV), num_supernodes=K,
                          weight=w.to(DEV))
    xg = x.to(DEV).requires_grad_(True)
    got, _ = T.B200Reduce(op)(xg, so_g)
    (got * gout.to(DEV)).sum().backward()
    torch.testing.assert_close(got.detach().cpu(), exp.detach(), **FP32)
    torch.testing.assert_close(xg.grad.cpu(), xc.grad, **FP32)


def test_segment_reduce_bf16():
    g = torch.Generator().manual_seed(3)
    N, K, F = 300, 90, 128
    cluster = torch.randint(0, K, (N,), generator=g)
    x = torch.randn(N, F, generator=g).bfloat16()
    w = (torch.rand(N, generator=g) + 0.5).bfloat16()
    so_c = R.OracleSelectOutput(cluster_index=cluster, num_supernodes=K, weight=w.float())
    exp, _ = R.base_reduce(x.float(), so_c)
    so_g = T.SelectOutput(cluster_index=cluster.to(DEV), num_supernodes=K, weight=w.to(DEV))
    xg = x.to(DEV).requires_grad_(True)
    got, _ = T.B200Reduce()(xg, so_g)
    assert got.dtype == torch.bfloat16
    torch.testing.assert_close(got.float().cpu(), exp, **BF16)
    got.float().sum().backward()
    assert xg.grad.dtype == torch.bfloat16 and torch.isfinite(xg.grad.float()).all()


def test_reduce_batch_and_readout():
    g = torch.Generator().manual_seed(5)
    N, K = 64, 20
    batch = torch.sort(torch.randint(0, 4, (N,), generator=g))[0]
    sel = torch.randperm(N, generator=g)[:30]
    cluster = torch.randint(0, K, (30,), generator=g)
    so_c = R.OracleSelectOutput(node_index=sel, num_nodes=N, cluster_index=cluster, num_supernodes=K)
    so_g = T.SelectOutput(node_index=sel.to(DEV), num_nodes=N, cluster_index=cluster.to(DEV), num_supernodes=K)
    assert torch.equal(T.Reduce.reduce_batch(so_g, batch.to(DEV)).cpu(), R.reduce_batch(so_c, batch))
    x = torch.randn(N, 6, generator=g)
    for op in ("sum", "mean", "max", "min"):
        exp, eb = R.readout(x, op, batch)
        got, gb = T.B200Reduce(op)(x.to(DEV), None, batch=batch.to(DEV))
        torch.testing.assert_close(got.cpu(), exp, **FP32)
        assert torch.equal(gb.cpu(), eb)
    x3 = torch.tensor([[[1.0, 2.0], [3.0, 4.0], [5.0, 6.0]], [[-1.0, 0.0], [0.0, 1.0], [2.0, -2.0]]])
    got, _ = T.B200Reduce("max")(x3.to(DEV), None)
    assert torch.equal(got.cpu(), torch.tensor([[5.0, 6.0], [2.0, 1.0]]))  # tests/reduce/test_global_reduce.py:9-37


# --------------------------------------------------------------------------- #
# golden fixtures generated by the reference's own files
# --------------------------------------------------------------------------- #
def test_golden_topk_cases(golden):
    names = sorted(k for k in golden if k.startswith("topk_"))
    assert len(names) == 16
    for name in names:
        c, f = golden[name], _flags(name)
        x = c["x"].to(DEV).requires_grad_(True)
        sw = c["weight"].to(DEV).requires_grad_(True)
        w = None if c["edge_weight"] is None else c["edge_weight"].to(DEV).requires_grad_(True)
        idx = torch.stack([c["node_index"], c["cluster_index"]]).to(DEV)
        so = T.SelectOutput(s=torch.sparse_coo_tensor(idx, sw, (c["num_nodes"], c["num_supernodes"]), is_coalesced=True))
        xp, ei, ew, bp = T.sparse_pool(x, c["edge_index"].to(DEV), so, edge_weight=w, batch=c["batch"].to(DEV),
                                       remove_self_loops=f["rsl"], degree_norm=f["dn"], edge_weight_norm=f["ewn"])
        assert torch.equal(ei.cpu(), c["edge_index_out"]), name
        assert ei.is_contiguous() and ei.dtype == torch.long
        assert torch.equal(bp.cpu(), c["batch_pool"]), name
        torch.testing.assert_close(xp.detach().cpu(), c["x_pool"], **FP32)
        if c["edge_weight_out"] is None:
            assert ew is None, name
        else:
            torch.testing.assert_close(ew.detach().cpu(), c["edge_weight_out"], **FP32)
        loss = xp.square().sum()
        if ew is not None and ew.requires_grad:
            loss = loss + (ew * torch.arange(1, ew.numel() + 1, device=DEV)).sum()
        loss.backward()
        # grad wrt x in the fixture includes the path through the TopK score; compare the reduce part
        # by replaying the oracle with detached select weights
        xo = c["x"].clone().requires_grad_(True)
        swo = c["weight"].clone().requires_grad_(True)
        so_o = R.OracleSelectOutput(s=torch.sparse_coo_tensor(idx.cpu(), swo, (c["num_nodes"], c["num_supernodes"]),
                                                              is_coalesced=True))
        wo = None if c["edge_weight"] is None else c["edge_weight"].clone().requires_grad_(True)
        xpo, eio, ewo, _ = R.topk_pool(xo, c["edge_index"], wo, so_o, batch=c["batch"], remove_self_loops=f["rsl"],
                                       degree_norm=f["dn"], edge_weight_norm=f["ewn"])
        lo = xpo.square().sum()
        if ewo is not None and ewo.requires_grad:
            lo = lo + (ewo * torch.arange(1, ewo.numel() + 1)).sum()
        lo.backward()
        torch.testing.assert_close(x.grad.cpu(), xo.grad, **FP32)
        torch.testing.assert_close(sw.grad.cpu(), swo.grad, rtol=1e-4, atol=1e-5)
        if w is not None:
            torch.testing.assert_close(w.grad.cpu(), c["grad_w"], rtol=1e-4, atol=1e-5, msg=name)


def test_golden_cluster_cases(golden):
    names = sorted(k for k in golden if k.startswith("cluster_"))
    assert len(names) == 40
    for name in names:
        c, f = golden[name], _flags(name)
        op = name.split("_")[1]
        x = c["x"].to(DEV).requires_grad_(True)
        w = None if c["edge_weight"] is None else c["edge_weight"].to(DEV).requires_grad_(True)
        so = T.SelectOutput(cluster_index=c["cluster"].to(DEV), num_nodes=x.size(0), num_supernodes=c["num_supernodes"])
        xp, bp = T.B200Reduce()(x, so, batch=c["batch"].to(DEV))
        conn = T.B200SparseConnect(op, f["rsl"], f["ewn"], f["dn"])
        ei, ew = conn(c["edge_index"].to(DEV), so, edge_weight=w, batch_pooled=c["batch_pooled"].to(DEV))
        assert torch.equal(ei.cpu(), c["edge_index_out"]), name
        assert torch.equal(bp.cpu(), c["batch_pool"]), name
        torch.testing.assert_close(xp.detach().cpu(), c["x_pool"], **FP32)
        if c["edge_weight_out"] is None:
            assert ew is None, name
        else:
            torch.testing.assert_close(ew.detach().cpu(), c["edge_weight_out"], **FP32, msg=name)
        loss = xp.square().sum()
        if ew is not None and ew.requires_grad:
            loss = loss + (ew * torch.arange(1, ew.numel() + 1, device=DEV)).sum()
        loss.backward()
        torch.testing.assert_close(x.grad.cpu(), c["grad_x"], **FP32)
        if w is not None and op != "mul":
            torch.testing.assert_close(w.grad.cpu(), c["grad_w"], rtol=1e-4, atol=1e-5, msg=name)


def test_golden_dense_cases(golden):
    names = sorted(k for k in golden if k.startswith("dense_"))
    assert len(names) == 16
    for name in names:
        c, f = golden[name], _flags(name)
        sr = c["s_raw"].to(DEV).requires_grad_(True)
        x = c["x"].to(DEV).requires_grad_(True)
        a = c["adj"].to(DEV).requires_grad_(True)
        mask = c["mask"].to(DEV)
        s = torch.softmax(sr, -1) * mask[..., None]
        kw = dict(remove_self_loops=f["rsl"], degree_norm=f["dn"], adj_transpose=f["t"], edge_weight_norm=f["ewn"])
        xp, post, lm = T.mincut_pool(x, a, s, **kw)
        _, post2, ld = T.diff_pool(x, a, s, num_nodes=int(mask.sum()), normalize_loss=False, **kw)
        _, _, ldn = T.diff_pool(x, a, s, num_nodes=int(mask.sum()), normalize_loss=True, **kw)
        raw = T.B200DenseConnect().dense_connect(a, s)
        for got, key in ((xp, "x_pool"), (raw, "adj_pool_raw"), (post, "adj_pool"), (post2, "adj_pool"),
                         (lm["cut_loss"], "cut"), (lm["ortho_loss"], "ortho"), (ld["link_loss"], "link"),
                         (ldn["link_loss"], "link_norm"), (ld["entropy_loss"], "ent")):
            close32(got.detach().cpu(), c[key], f"{name}:{key}")
        wts = (torch.arange(1, post.numel() + 1, dtype=torch.float, device=DEV).view_as(post) / post.numel())
        total = (xp.square().sum() + (post * wts).sum() + lm["cut_loss"] + lm["ortho_loss"] + 0.5 * ld["link_loss"]
                 + 0.25 * ld["entropy_loss"])
        total.backward()
        # the fixture total used x_pool/post from one forward; ours reuses xp/post from mincut_pool only
        close32(sr.grad.cpu(), c["grad_s_raw"], f"{name} dS", rtol=1e-4)
        close32(x.grad.cpu(), c["grad_x"], f"{name} dX")
        ga, ea = a.grad.cpu(), c["grad_adj"]
        if f["ewn"]:
            # max-normalisation routes one gradient term to "the" arg-max; a symmetric adjacency ties (r,c) with
            # (c,r) and the reference's own pick depends on fp32 rounding noise, so only the symmetric part of dA
            # is well defined for these cases.
            ga, ea = 0.5 * (ga + ga.transpose(1, 2)), 0.5 * (ea + ea.transpose(1, 2))
        close32(ga, ea, f"{name} dA", rtol=1e-4)


# --------------------------------------------------------------------------- #
# sparse connect at larger random sizes (bit-exact indices vs oracle)
# --------------------------------------------------------------------------- #
def _random_graph(g, n, e, weighted=True):
    ei = torch.randint(0, n, (2, e), generator=g)
    order = torch.argsort(ei[0] * n + ei[1], stable=True)
    ei = ei[:, order]
    ew = (torch.rand(e, generator=g) + 0.5) if weighted else None
    return ei, ew


@pytest.mark.parametrize("weighted", [True, False])
@pytest.mark.parametrize("dn,ewn", [(False, False), (True, True)])
def test_kept_node_connect_large(weighted, dn, ewn):
    g = torch.Generator().manual_seed(11)
    n, e = 50_000, 400_000
    ei, ew = _random_graph(g, n, e, weighted)
    score = torch.randn(n, generator=g)
    batch = torch.sort(torch.randint(0, 16, (n,), generator=g))[0]
    so_c = R.topk_select(score, None, 0.5, batch, act=torch.tanh)
    bp_c = R.reduce_batch(so_c, batch)
    eo, wo = R.sparse_connect_so(ei, so_c, edge_weight=ew, batch_pooled=bp_c, degree_norm=dn, edge_weight_norm=ewn)
    so_g = T.SelectOutput(s=so_c.s.to(DEV))
    bp_g = T.Reduce.reduce_batch(so_g, batch.to(DEV))
    assert torch.equal(bp_g.cpu(), bp_c)
    eg, wg = T.B200SparseConnect(degree_norm=dn, edge_weight_norm=ewn)(ei.to(DEV), so_g, edge_weight=_cu(ew),
                                                                        batch_pooled=bp_g)
    assert torch.equal(eg.cpu(), eo)
    if wo is None:
        assert wg is None
    else:
        torch.testing.assert_close(wg.cpu(), wo, **FP32)


@pytest.mark.parametrize("weighted", [True, False])
@pytest.mark.parametrize("K", [300, 40_000, 90_000])  # 32-bit and 64-bit key paths
def test_cluster_connect_large(weighted, K):
    g = torch.Generator().manual_seed(K)
    n, e = 100_000, 600_000
    ei, ew = _random_graph(g, n, e, weighted)
    cluster = torch.randint(0, K, (n,), generator=g)
    so_c = R.OracleSelectOutput(cluster_index=cluster, num_supernodes=K)
    eo, wo = R.sparse_connect_so(ei, so_c, edge_weight=ew, degree_norm=True)
    so_g = T.SelectOutput(cluster_index=cluster.to(DEV), num_supernodes=K)
    eg, wg = T.B200SparseConnect(degree_norm=True)(ei.to(DEV), so_g, edge_weight=_cu(ew))
    assert torch.equal(eg.cpu(), eo)
    torch.testing.assert_close(wg.cpu(), wo, **FP32)
    key = eg[0] * K + eg[1]
    assert bool((key[1:] > key[:-1]).all())  # lexicographic, duplicate-free


def test_connect_edge_cases():
    so = T.SelectOutput(cluster_index=torch.tensor([0, 1, 0, 2], device=DEV), num_supernodes=4)
    empty = torch.empty((2, 0), dtype=torch.long, device=DEV)
    ei, ew = T.B200SparseConnect()(empty, so)
    assert ei.shape == (2, 0) and ew is None
    ei, ew = T.B200SparseConnect()(empty, so, edge_weight=torch.empty(0, device=DEV))
    assert ei.shape == (2, 0) and ew.shape == (0,)
    # all edges intra-cluster -> all removed as self loops
    e2 = torch.tensor([[0, 2], [2, 0]], device=DEV)
    ei, ew = T.B200SparseConnect()(e2, so, edge_weight=torch.ones(2, device=DEV))
    assert ei.shape == (2, 0)
    # tiny weights dropped (tests/utils/test_ops.py:254-269)
    e3 = torch.tensor([[0, 1], [1, 0]], device=DEV)
    ei, ew = T.B200SparseConnect(remove_self_loops=False)(e3, so, edge_weight=torch.tensor([0.0, 1.0], device=DEV))
    assert ei.shape == (2, 1) and torch.equal(ew.cpu(), torch.tensor([1.0]))
    # [E,1] weights flatten, [E,2] raise (tests/poolers/test_graclus.py:50-74)
    ei, ew = T.B200SparseConnect()(e3, so, edge_weight=torch.ones(2, 1, device=DEV))
    assert ew.dim() == 1
    with pytest.raises(RuntimeError):
        T.B200SparseConnect()(e3, so, edge_weight=torch.ones(2, 2, device=DEV))
    with pytest.raises(ValueError):
        T.B200SparseConnect()(e3.to(torch.int32), so)
    # torch COO in -> coalesced torch COO out, weights None (base_conn.py:103-110)
    coo = torch.sparse_coo_tensor(torch.tensor([[0, 1, 3], [1, 3, 0]], device=DEV),
                                  torch.tensor([1.0, 2.0, 3.0], device=DEV), (4, 4)).coalesce()
    out, w = T.B200SparseConnect()(coo, so)
    exp, _ = R.sparse_connect_so(coo.cpu(), R.OracleSelectOutput(cluster_index=torch.tensor([0, 1, 0, 2]), num_supernodes=4))
    assert w is None and out.is_sparse
    assert torch.equal(out.indices().cpu(), exp.indices()) and torch.allclose(out.values().cpu(), exp.values())


def test_determinism_run_twice():
    g = torch.Generator().manual_seed(7)
    n, e, K = 20_000, 300_000, 5_000
    ei, ew = _random_graph(g, n, e)
    cluster = torch.randint(0, K, (n,), generator=g)
    x = torch.randn(n, 64, generator=g).to(DEV)
    outs = []
    for _ in range(2):
        so = T.SelectOutput(cluster_index=cluster.to(DEV), num_supernodes=K)
        xp, _ = T.B200Reduce("mean")(x, so)
        eo, wo = T.B200SparseConnect()(ei.to(DEV), so, edge_weight=ew.to(DEV))
        outs.append((xp, eo, wo))
    for a, b in zip(outs[0], outs[1]):
        assert torch.equal(a, b)


# --------------------------------------------------------------------------- #
# dense path at non-trivial shapes
# --------------------------------------------------------------------------- #
def _dense_inputs(g, B, N, K, F, p=0.1):
    a = (torch.rand(B, N, N, generator=g) < p).float()
    a = torch.triu(a, 1)
    a = a + a.transpose(1, 2)
    s_raw = torch.randn(B, N, K, generator=g)
    x = torch.randn(B, N, F, generator=g)
    return a, s_raw, x


@pytest.mark.parametrize("B,N,K,F", [(4, 100, 16, 33), (3, 256, 64, 128), (2, 64, 16, 256)])
@pytest.mark.parametrize("kind", ["mincut", "diff"])
def test_dense_pool_fp32_vs_oracle(B, N, K, F, kind):
    g = torch.Generator().manual_seed(B * N + K)
    a, s_raw, x = _dense_inputs(g, B, N, K, F)
    gx = torch.randn(B, K, F, generator=g)
    ga = torch.randn(B, K, K, generator=g)

    def run(mod, dev, dt):
        sr = s_raw.detach().clone().to(dev, dt).requires_grad_(True)
        xx = x.detach().clone().to(dev, dt).requires_grad_(True)
        aa = a.detach().clone().to(dev, dt).requires_grad_(True)
        s = torch.softmax(sr, -1)
        fn = mod.mincut_pool if kind == "mincut" else mod.diff_pool
        xp, ap, loss = fn(xx, aa, s)
        tot = (xp * gx.to(dev, dt)).sum() + (ap * ga.to(dev, dt)).sum() + sum(loss.values())
        tot.backward()
        return [t.detach().cpu().float() for t in (xp, ap, *loss.values(), sr.grad, xx.grad, aa.grad)]

    # The oracle is evaluated in float64: the reference's own fp32 CPU value of the batch-global Frobenius
    # norm (link loss) carries ~1e-5 of summation error at these sizes, i.e. as much as the tolerance.
    exp = run(R, "cpu", torch.float64)
    got = run(T, DEV, torch.float32)
    names = ["x_pool", "adj_pool", "loss0", "loss1", "grad_s", "grad_x", "grad_adj"]
    for n_, e_, g_ in zip(names, exp, got):
        close32(g_, e_, f"{kind} {n_}", rtol=1e-5 if not n_.startswith("grad") else 1e-4)


@pytest.mark.parametrize("elems,self_loops", [(64, 1), (128, 0), (32768, 1), (600, 0)])
@pytest.mark.parametrize("K", [6, 12, 32, 128])
def test_dense_per_graph_kernels_all_strip_plans(monkeypatch, elems, self_loops, K):
    """The per-graph epilogue / backward kernels run as clusters of row strips; every plan (cluster size 1..8,
    scalar / 128-bit paths) must give the same answer as the float64 oracle for every flag set, with and without
    weighted self loops in the input adjacency."""
    monkeypatch.setenv("TGPB200_STRIP_ELEMS", str(elems))
    B, N, F = 3, 160, 32
    g = torch.Generator().manual_seed(1000 + K)
    a, s_raw, x = _dense_inputs(g, B, N, K, F)
    loops = torch.diag_embed(torch.rand(B, N, generator=g))
    if self_loops:
        a = a + loops
    gx = torch.randn(B, K, F, generator=g)
    ga = torch.randn(B, K, K, generator=g)
    ga = ga + ga.transpose(1, 2)
    for kind in ("mincut", "diff"):
        for rsl, dn, tr, ewn in [(True, True, True, False), (True, True, False, False), (False, True, True, True),
                                 (True, False, True, True), (False, False, False, False), (True, True, False, True)]:
            kw = dict(remove_self_loops=rsl, degree_norm=dn, adj_transpose=tr, edge_weight_norm=ewn)

            def run(mod, dev, dt):
                sr = s_raw.detach().clone().to(dev, dt).requires_grad_(True)
                xx = x.detach().clone().to(dev, dt).requires_grad_(True)
                aa = a.detach().clone().to(dev, dt).requires_grad_(True)
                s = torch.softmax(sr, -1)
                fn = mod.mincut_pool if kind == "mincut" else mod.diff_pool
                xp, ap, loss = fn(xx, aa, s, **kw)
                tot = (xp * gx.to(dev, dt)).sum() + (ap * ga.to(dev, dt)).sum() + sum(loss.values())
                tot.backward()
                ag = aa.grad
                if ewn:  # only the symmetric part of dA is well defined under max-normalisation (see above)
                    ag = 0.5 * (ag + ag.transpose(1, 2))
                return [t.detach().cpu().float() for t in (xp, ap, *loss.values(), sr.grad, xx.grad, ag)]

            exp = run(R, "cpu", torch.float64)
            got = run(T, DEV, torch.float32)
            names = ["x_pool", "adj_pool", "loss0", "loss1", "grad_s", "grad_x", "grad_adj"]
            for n_, e_, g_ in zip(names, exp, got):
                close32(g_, e_, f"{kind} {kw} {n_}", rtol=1e-5 if not n_.startswith("grad") else 1e-4)


def test_fused_forward_exact_and_inexact_adjacency_blocks():
    """3xTF32 residuals are zero for adjacency entries that are exact in tf32 (0/1) and non-zero for weighted ones.
    Mix both inside one graph and across the graphs a CTA visits, so that every pipeline slot of the fused forward
    sees exact and inexact 16-row blocks in turn (guards any data-dependent shortcut in the split warps)."""
    B, N, K, F = 150, 256, 64, 128  # 150 graphs > 148 SMs: two CTAs process a second graph
    g = torch.Generator().manual_seed(77)
    a01, s_raw, x = _dense_inputs(g, B, N, K, F)
    wts = torch.rand(B, N, N, generator=g) + 0.5
    wts = 0.5 * (wts + wts.transpose(1, 2))
    a = a01.clone()
    a[1::3] = (a01 * wts)[1::3]                       # fully weighted graphs
    a[2::3, :128] = (a01 * wts)[2::3, :128]           # first half of the rows weighted, second half 0/1
    a[0, 200:216] = a01[0, 200:216] * wts[0, 200:216]  # one weighted k-block in an otherwise exact graph
    s = torch.softmax(s_raw, -1)
    exp = R.mincut_pool(x.double(), a.double(), s.double(), remove_self_loops=False, degree_norm=False)
    got = T.mincut_pool(x.to(DEV), a.to(DEV), s.to(DEV), remove_self_loops=False, degree_norm=False)
    close32(got[0].cpu(), exp[0].float(), "x_pool")
    close32(got[1].cpu(), exp[1].float(), "adj_pool (raw S^T A S)")
    for k in exp[2]:
        close32(got[2][k].cpu(), exp[2][k].float(), k)


@pytest.mark.parametrize("B,N,K,F", [(5, 200, 48, 100), (3, 72, 20, 36), (2, 256, 256, 64), (150, 64, 8, 16)])
@pytest.mark.parametrize("fused_ts", ["1", "0"])
def test_dense_pool_fp32_ragged_shapes(monkeypatch, fused_ts, B, N, K, F):
    """Shapes off the tile grid (partial last k-block, K not a multiple of 16 / 32, more graphs than SMs, a K too
    wide for any fused forward) through the TMEM-operand fused forward and through its shared-memory sibling."""
    monkeypatch.setenv("TGPB200_FUSED_TS", fused_ts)
    g = torch.Generator().manual_seed(B + 7 * N + K)
    a, s_raw, x = _dense_inputs(g, B, N, K, F)
    a = a * (torch.rand(B, N, N, generator=g) + 0.5)
    a = 0.5 * (a + a.transpose(1, 2))
    gx = torch.randn(B, K, F, generator=g)
    ga = torch.randn(B, K, K, generator=g)

    def run(mod, dev, dt):
        sr = s_raw.detach().clone().to(dev, dt).requires_grad_(True)
        xx = x.detach().clone().to(dev, dt).requires_grad_(True)
        aa = a.detach().clone().to(dev, dt).requires_grad_(True)
        xp, ap, loss = mod.mincut_pool(xx, aa, torch.softmax(sr, -1))
        ((xp * gx.to(dev, dt)).sum() + (ap * ga.to(dev, dt)).sum() + sum(loss.values())).backward()
        return [t.detach().cpu().float() for t in (xp, ap, *loss.values(), sr.grad, xx.grad, aa.grad)]

    exp = run(R, "cpu", torch.float64)
    got = run(T, DEV, torch.float32)
    for n_, e_, g_ in zip(["x_pool", "adj_pool", "cut", "ortho", "grad_s", "grad_x", "grad_adj"], exp, got):
        close32(g_, e_, n_, rtol=1e-5 if not n_.startswith("grad") else 1e-4)


def test_dense_pool_bf16_vs_oracle():
    g = torch.Generator().manual_seed(21)
    B, N, K, F = 3, 128, 32, 64
    a, s_raw, x = _dense_inputs(g, B, N, K, F)
    s = torch.softmax(s_raw, -1).bfloat16()
    xb, ab = x.bfloat16(), a.bfloat16()
    exp = R.diff_pool(xb.float(), ab.float(), s.float())
    got = T.diff_pool(xb.to(DEV), ab.to(DEV), s.to(DEV))
    assert got[0].dtype == torch.bfloat16 and got[1].dtype == torch.bfloat16
    torch.testing.assert_close(got[0].float().cpu(), exp[0], **BF16)
    torch.testing.assert_close(got[1].float().cpu(), exp[1], **BF16)
    for k in exp[2]:
        torch.testing.assert_close(got[2][k].float().cpu(), exp[2][k], **BF16)


def test_dense_connect_hand_matrix():
    # tests/connect/test_dense_conn.py:210-232
    s = torch.tensor([[1.0, 0.0], [0.0, 1.0], [1.0, 0.0]], device=DEV)
    adj = torch.tensor([[0.0, 1.0, 2.0], [1.0, 0.0, 3.0], [2.0, 3.0, 0.0]], device=DEV)
    out = T.B200DenseConnect().dense_connect(adj=adj, s=s)
    assert out.shape == (1, 2, 2)
    assert torch.equal(out[0].cpu(), torch.tensor([[4.0, 4.0], [4.0, 0.0]]))


# --------------------------------------------------------------------------- #
# TopK selection (bit-exact)
# --------------------------------------------------------------------------- #
@pytest.mark.parametrize("N,G,ratio", [(6, 1, 0.5), (1000, 7, 0.5), (5000, 128, 0.3), (200_000, 1, 0.5), (50_000, 64, 3)])
def test_topk_select_bit_exact(N, G, ratio):
    g = torch.Generator().manual_seed(N + G)
    batch = torch.sort(torch.randint(0, G, (N,), generator=g))[0]
    batch[0], batch[-1] = 0, G - 1
    score = torch.tanh(torch.randn(N, generator=g))
    score[torch.randint(0, N, (N // 10,), generator=g)] = 0.25  # many exact ties
    score[:3] = torch.tensor([0.0, -0.0, 0.0])[: min(3, N)]
    so_c = R.topk_select(score, None, ratio, batch, act=lambda v: v)
    ni, ci = T.topk(score.to(DEV), ratio, batch.to(DEV))
    assert torch.equal(ni.cpu(), so_c.node_index)
    assert torch.equal(ci.cpu(), so_c.cluster_index)
    so_g = T.topk_select(score.to(DEV), None, ratio, batch.to(DEV), act="linear")
    assert torch.equal(so_g.weight.cpu(), so_c.weight) and so_g.num_supernodes == so_c.num_supernodes


def test_topk_reference_pins():
    # tests/poolers/test_topk.py:22-34 (scores 1..5, ratio .5 -> {2,3,4}) and :60-63 (k = ceil(0.5 * 6) = 3)
    so = T.topk_select(torch.arange(1.0, 6.0, device=DEV).unsqueeze(-1), None, 0.5, None, act="linear")
    assert torch.equal(so.node_index.sort(descending=True)[0].cpu(), torch.tensor([4, 3, 2]))
    x = torch.randn(6, 4, device=DEV)
    p = torch.randn(1, 4, device=DEV, requires_grad=True)
    so = T.topk_select(x, p, 0.5)
    assert so.num_supernodes == 3
    so.weight.sum().backward()
    assert p.grad is not None and torch.isfinite(p.grad).all()


# --------------------------------------------------------------------------- #
# sparse output of dense poolers, dense pre-processing
# --------------------------------------------------------------------------- #
def test_block_diag_and_finalize_sparse_output():
    g = torch.Generator().manual_seed(4)
    B, N, K, F = 5, 20, 6, 7
    s = torch.softmax(torch.randn(B, N, K, generator=g), -1)
    s[:, :, 4] = 0.0          # an empty supernode in every graph
    s[2, :, 1] = 0.0
    adj_pool = torch.randn(B, K, K, generator=g)
    adj_pool[0, 1, 2] = 1e-9  # below eps
    x_pool = torch.randn(B, K, F, generator=g)
    mask = R.out_mask_from_dense_s(s)
    for m in (None, mask):
        ap = adj_pool.clone().requires_grad_(True)
        exp = R.finalize_sparse_output(x_pool, ap, None, None, m)
        (exp[2] * torch.arange(1, exp[2].numel() + 1)).sum().backward()
        ag = adj_pool.clone().to(DEV).requires_grad_(True)
        got = F_.finalize_sparse_output(x_pool.to(DEV), ag, None, None, None if m is None else m.to(DEV))
        (got[2] * torch.arange(1, got[2].numel() + 1, device=DEV)).sum().backward()
        assert torch.equal(got[1].cpu(), exp[1])
        assert torch.equal(got[2].detach().cpu(), exp[2].detach())
        assert torch.equal(got[0].cpu(), exp[0]) and torch.equal(got[3].cpu(), exp[3])
        assert torch.equal(ag.grad.cpu(), ap.grad)
    ei, ew = F_.dense_to_block_diag(torch.zeros(2, 3, 3, device=DEV))
    assert ei.shape == (2, 0) and ew.shape == (0,)


def test_dense_preprocessing_matches_pyg_semantics():
    from oracle import pyg_shim as pyg

    g = torch.Generator().manual_seed(8)
    sizes = [5, 9, 1, 7]
    batch = torch.cat([torch.full((n,), i) for i, n in enumerate(sizes)])
    N = batch.numel()
    x = torch.randn(N, 6, generator=g)
    eis, off = [], 0
    for n in sizes:
        eis.append(torch.randint(0, n, (2, 3 * n), generator=g) + off)
        off += n
    ei = torch.cat(eis, 1)
    ew = torch.rand(ei.size(1), generator=g)
    xd, m = pyg.to_dense_batch(x, batch)
    xg, mg = F_.to_dense_batch(x.to(DEV), batch.to(DEV))
    assert torch.equal(xg.cpu(), xd) and torch.equal(mg.cpu(), m)
    for w in (None, ew):
        ad = pyg.to_dense_adj(ei, batch, w)
        ag = F_.to_dense_adj(ei.to(DEV), batch.to(DEV), _cu(w))
        torch.testing.assert_close(ag.cpu(), ad, rtol=1e-6, atol=1e-6)
        agt = F_.to_dense_adj(ei.to(DEV), batch.to(DEV), _cu(w), transpose=True)
        torch.testing.assert_close(agt.cpu(), ad.transpose(1, 2), rtol=1e-6, atol=1e-6)


@pytest.mark.parametrize("sparse_output", [False, True])
def test_unbatched_dense_mode_matches_oracle_and_batched(sparse_output):
    # tests/poolers/test_dense_poolers_batched_vs_unbatched.py:36-174: batched == unbatched (rtol 1e-5)
    g = torch.Generator().manual_seed(12)
    sizes = [12, 20, 7]
    K, F = 4, 5
    batch = torch.cat([torch.full((n,), i) for i, n in enumerate(sizes)])
    N = batch.numel()
    eis, off = [], 0
    for n in sizes:
        up = torch.triu(torch.rand(n, n, generator=g) < 0.4, 1)
        r, c = up.nonzero(as_tuple=True)
        eis.append(torch.cat([torch.stack([r, c]), torch.stack([c, r])], 1) + off)
        off += n
    ei = torch.cat(eis, 1)
    ew = torch.rand(ei.size(1), generator=g) + 0.5
    s = torch.softmax(torch.randn(N, K, generator=g), -1)
    x = torch.randn(N, F, generator=g)
    bp = torch.arange(len(sizes)).repeat_interleave(K)
    exp_a, exp_w = R.dense_connect_forward_unbatched(ei, ew, batch, s, bp, sparse_output=sparse_output)
    so = T.SelectOutput(s=s.to(DEV), batch=batch.to(DEV))
    conn = T.B200DenseConnect(adj_transpose=False, sparse_output=sparse_output)
    got_a, got_w = conn(ei.to(DEV), so, edge_weight=ew.to(DEV), batch=batch.to(DEV), batch_pooled=bp.to(DEV))
    if sparse_output:
        assert torch.equal(got_a.cpu(), exp_a)
        close32(got_w.cpu(), exp_w, "unbatched sparse weights")
    else:
        assert got_w is None
        close32(got_a.cpu(), exp_a, "unbatched dense adj")
    exp_x, exp_b = R.base_reduce(x, R.OracleSelectOutput(s=s), batch=batch)
    got_x, got_b = T.B200Reduce()(x.to(DEV), so, batch=batch.to(DEV))
    close32(got_x.cpu(), exp_x, "unbatched reduce")
    assert torch.equal(got_b.cpu(), exp_b)
    got_xb, _ = T.B200Reduce()(x.to(DEV), so, batch=batch.to(DEV), return_batched=True)
    assert got_xb.shape == (len(sizes), K, F)


# --------------------------------------------------------------------------- #
# lift (tgp/lift/base_lift.py:113-123 sparse, dense batched matmul)
# --------------------------------------------------------------------------- #
def test_lift_sparse_and_dense():
    g = torch.Generator().manual_seed(6)
    N, K, F = 300, 80, 32
    cluster = torch.randint(0, K, (N,), generator=g)
    w = torch.rand(N, generator=g) + 0.5
    xp = torch.randn(K, F, generator=g)
    xpc, wc = xp.clone().requires_grad_(True), w.clone().requires_grad_(True)
    exp = xpc[cluster] * wc.view(-1, 1)          # scatter(x_pool[col] * values, row) with row = arange(N)
    gout = torch.randn(N, F, generator=g)
    (exp * gout).sum().backward()
    xpg, wg = xp.to(DEV).requires_grad_(True), w.to(DEV).requires_grad_(True)
    so = T.SelectOutput(s=torch.sparse_coo_tensor(torch.stack([torch.arange(N), cluster]).to(DEV), wg, (N, K),
                                                   is_coalesced=True, check_invariants=False))
    got = T.B200Lift()(xpg, so)
    (got * gout.to(DEV)).sum().backward()
    torch.testing.assert_close(got.detach().cpu(), exp.detach(), **FP32)
    torch.testing.assert_close(xpg.grad.cpu(), xpc.grad, rtol=1e-5, atol=1e-5)
    torch.testing.assert_close(wg.grad.cpu(), wc.grad, rtol=1e-4, atol=1e-5)
    # TopK-style: only kept nodes receive features, the rest are zero rows
    keep = torch.sort(torch.randperm(N, generator=g)[:K])[0]
    so2 = T.SelectOutput(node_index=keep.to(DEV), num_nodes=N, cluster_index=torch.arange(K, device=DEV), num_supernodes=K)
    lifted = T.B200Lift()(xp.to(DEV), so2).cpu()
    assert torch.equal(lifted[keep], xp) and float(lifted.abs().sum()) == float(xp.abs().sum())
    # dense batched: S x_pool
    B, Nn, Kk, Ff = 3, 128, 32, 64
    s = torch.softmax(torch.randn(B, Nn, Kk, generator=g), -1)
    xpd = torch.randn(B, Kk, Ff, generator=g)
    sc, xc = s.clone().double().requires_grad_(True), xpd.clone().double().requires_grad_(True)
    ed = sc @ xc
    gd = torch.randn(B, Nn, Ff, generator=g)
    (ed * gd.double()).sum().backward()
    sg, xg = s.to(DEV).requires_grad_(True), xpd.to(DEV).requires_grad_(True)
    gotd = T.B200Lift()(xg, T.SelectOutput(s=sg))
    (gotd * gd.to(DEV)).sum().backward()
    close32(gotd.detach().cpu(), ed.detach().float(), "lift dense")
    close32(sg.grad.cpu(), sc.grad.float(), "lift dS", rtol=1e-4)
    close32(xg.grad.cpu(), xc.grad.float(), "lift dXp", rtol=1e-4)
