"""B200: HOSC pooling on a sparse adjacency (``unbatched.hosc_losses_unbatched`` / ``hosc_pool_unbatched``) against the
float64 ``hosc_oracle`` on the densified graphs, per gradient source, in fp32 and bf16; the batched device path on
``to_dense_adj`` of the same graphs; the motif weights against scipy on a power-law graph with hubs and on a directed
graph; hand values; zero-weight runs keep their gradient; determinism; the term mask; the workspace contract of the
new entry points; and one graph of 200 000 nodes whose dense adjacency would need 160 GB."""
import os
import sys

import numpy as np
import pytest
import scipy.sparse as sp
import torch

import dense_loss_cases as C
import hosc_oracle as O
import hosc_sparse_oracle as SO
import tgp_b200 as T
from dense_loss_cases import DEV, FLAGSETS
from tgp_b200 import _lib as L
from tgp_b200 import functional as F_
from tgp_b200 import ops as OPS
from tgp_b200 import unbatched as U

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

pytestmark = pytest.mark.gpu
COEF = {"hosc": 1.7, "ortho": -0.8}
KEYS = {"hosc": "hosc_loss", "ortho": "ortho_loss"}
MU = 0.3

CASES = {
    "ragged": lambda bf16=False: SO.random_case([40, 23, 61, 7], 6.0, 8, seed=1, bf16_weights=bf16),
    "directed": lambda bf16=False: SO.random_case([50, 31], 5.0, 6, seed=2, directed=True, bf16_weights=bf16),
    "isolated_trianglefree_edgeless": lambda bf16=False: _special_case(),
}


def _special_case():
    """graph 0: a triangle with a zero-weight chord pair plus an isolated node; graph 1: a 4-cycle; graph 2: no edge."""
    ei = torch.tensor([[0, 1, 1, 2, 2, 0, 0, 3, 4, 5, 5, 6, 6, 7, 7, 4],
                       [1, 0, 2, 1, 0, 2, 0, 0, 5, 4, 6, 5, 7, 6, 4, 7]])
    w = torch.tensor([1.0, 1.0, 0.5, 0.5, 2.0, 2.0, 0.75, 0.0, 1.0, 1.0, 1.5, 1.5, 1.0, 1.0, 0.75, 0.75],
                     dtype=torch.float64)
    batch = torch.tensor([0, 0, 0, 0, 1, 1, 1, 1, 2, 2, 2])
    s = torch.softmax(torch.randn(11, 3, generator=torch.Generator().manual_seed(3), dtype=torch.float64), -1)
    return ei, w, s, batch, 3


def _terms(alpha, hosc_ortho):
    return (1 if alpha != 1.0 else 0) | (2 if alpha != 0.0 else 0) | (4 if hosc_ortho else 0)


def _per_graph_check(got, exp, groups, tau, what):
    """max|got - ref| <= tau * max|ref| inside every graph (groups: graph of every row / edge)."""
    got, exp = got.double().cpu(), exp.double().cpu()
    for b in torch.unique(groups).tolist():
        sel = groups == b
        bound = tau * float(exp[sel].abs().max()) if sel.any() else 0.0
        err = float((got[sel] - exp[sel]).abs().max()) if sel.any() else 0.0
        assert err <= bound + 1e-30, f"{what}, graph {b}: max error {err:.3e} > {bound:.3e}"


@pytest.mark.parametrize("hosc_ortho", [False, True])
@pytest.mark.parametrize("alpha", [0.0, 0.5, 1.0])
@pytest.mark.parametrize("case", list(CASES))
def test_losses_fp32_against_sparse_restatement(case, alpha, hosc_ortho):
    ei, w, s, batch, B = CASES[case]()
    g = (0.7, -1.3, 0.9)
    exp_l, exp_ds, exp_dw = SO.forward_backward(ei.numpy(), w.numpy(), s.numpy(), batch.numpy(), B, g,
                                                _terms(alpha, hosc_ortho))
    wd, sd = w.float().to(DEV).requires_grad_(True), s.float().to(DEV).requires_grad_(True)
    losses = U.hosc_losses_unbatched(ei.to(DEV), wd, sd, batch.to(DEV), alpha, hosc_ortho)
    (losses * torch.tensor(g, device=DEV)).sum().backward()
    torch.testing.assert_close(losses.cpu().double(), torch.tensor(exp_l), rtol=1e-5, atol=0.0)
    _per_graph_check(sd.grad, torch.tensor(exp_ds), batch, 1e-4, "dS")
    _per_graph_check(wd.grad, torch.tensor(exp_dw), batch[ei[0]], 1e-4, "d edge_weight")


def test_hand_values():
    tri = torch.tensor([(i, j) for comp in ([0, 1, 2], [3, 4, 5]) for i in comp for j in comp if i != j]).T
    s = torch.zeros(6, 2)
    s[:3, 0] = s[3:, 1] = 1.0
    got = U.hosc_losses_unbatched(tri.to(DEV), None, s.to(DEV), None, 0.5, True).cpu()
    torch.testing.assert_close(got, torch.tensor([-1.0, -1.0, 0.0]), rtol=0, atol=1e-6)
    cyc = torch.tensor([(i, (i + 1) % 4) for i in range(4)] + [((i + 1) % 4, i) for i in range(4)]).T
    s = torch.zeros(4, 2)
    s[:2, 0] = s[2:, 1] = 1.0
    got = U.hosc_losses_unbatched(cyc.to(DEV), None, s.to(DEV), None, 0.5, False).cpu()
    assert torch.isfinite(got).all()
    torch.testing.assert_close(got[:2], torch.tensor([-0.5, 0.0]), rtol=0, atol=1e-6)


def test_zero_weight_runs_keep_their_gradient():
    """Runs whose weights sum to 0 (a zero edge; a pair of duplicates +w, -w) stay on the pattern: their gradient is
    the restatement's, not 0."""
    ei = torch.tensor([[0, 1, 1, 2, 2, 0, 0, 0, 2, 3, 3],
                       [1, 0, 2, 1, 0, 2, 3, 3, 3, 2, 0]])
    w = torch.tensor([1.0, 1.0, 0.5, 0.5, 2.0, 2.0, 0.75, -0.75, 0.0, 1.25, 1.0], dtype=torch.float64)
    s = torch.softmax(torch.randn(4, 3, generator=torch.Generator().manual_seed(5), dtype=torch.float64), -1)
    batch = torch.zeros(4, dtype=torch.long)
    _, _, exp_dw = SO.forward_backward(ei.numpy(), w.numpy(), s.numpy(), batch.numpy(), 1, (1.0, 1.0, 0.0), 3)
    wd = w.float().to(DEV).requires_grad_(True)
    U.hosc_losses_unbatched(ei.to(DEV), wd, s.float().to(DEV), None, 0.5, False).sum().backward()
    assert float(np.abs(exp_dw[6:9]).min()) > 1e-3  # the zero runs do carry a gradient
    torch.testing.assert_close(wd.grad.cpu().double(), torch.tensor(exp_dw), rtol=1e-4,
                               atol=1e-4 * float(np.abs(exp_dw).max()))


def _oracle_pool(ei, w, s, x, batch, B, alpha, hosc_ortho, flags, up):
    """float64 hosc_oracle.hosc_pool on the densified graph (adj_transpose off) and the (dX, dw, dS) per source."""
    wl, sl, xl = (t.double().requires_grad_(True) for t in (w, s, x))
    adj, S, mask = SO.densify(ei, wl, sl, batch, B)
    X = SO.densify(ei, wl.detach(), xl, batch, B)[1]
    fl = dict(flags, adj_transpose=False)
    xp, ap, loss = O.hosc_pool(X, adj, S, mask, MU, alpha, hosc_ortho, **fl)
    grads = C.per_source_grads(xp, ap, loss, up, (xl, wl, sl), COEF, KEYS)
    return xp.detach(), ap.detach(), torch.stack([loss[k] for k in KEYS.values()]).detach(), grads, (adj, S, X, mask)


def _check_pool(xp, ap, losses, grads, ref, tau, loss_rtol, scale_dense=1e-5):
    xp_e, ap_e, loss_e, g_e = ref[:4]
    torch.testing.assert_close(losses.cpu().double(), loss_e, rtol=loss_rtol, atol=0.0)
    for name, gv, ev in (("x_pool", xp, xp_e), ("adj_pool", ap, ap_e)):
        torch.testing.assert_close(gv.cpu().double(), ev, rtol=scale_dense, atol=scale_dense * float(ev.abs().max()),
                                   msg=name)
    for src in g_e:
        for name, gv, ev in zip(("dX", "dw", "dS"), grads[src], g_e[src]):
            bound = tau * float(ev.abs().max())
            err = float((gv.cpu().double() - ev).abs().max())
            assert err <= bound + 1e-30, f"{src} -> {name}: max error {err:.3e} > {bound:.3e}"


def _device_pool(ei, w, s, x, batch, alpha, hosc_ortho, flags, up, dtype):
    wd = w.float().to(DEV).requires_grad_(True)
    sd, xd = (t.to(DEV, dtype).requires_grad_(True) for t in (s, x))
    fl = {k: v for k, v in flags.items() if k != "adj_transpose"}
    xp, ap, loss = U.hosc_pool_unbatched(xd, ei.to(DEV), wd, sd, batch.to(DEV), None, MU, alpha, hosc_ortho, **fl)
    grads = C.per_source_grads(xp, ap, loss, up, (xd, wd, sd), COEF, KEYS)
    losses = torch.stack([loss[k] for k in KEYS.values()]).detach()
    return xp.detach(), ap.detach(), losses, {k: [t.cpu() for t in v] for k, v in grads.items()}


@pytest.mark.parametrize("hosc_ortho", [False, True])
@pytest.mark.parametrize("alpha", [0.0, 0.5, 1.0])
@pytest.mark.parametrize("flags", FLAGSETS)
@pytest.mark.parametrize("case", ["ragged", "directed"])
def test_pool_fp32_parity_and_batched_agreement(case, flags, alpha, hosc_ortho):
    ei, w, s, batch, B = CASES[case]()
    F = 24
    x = torch.randn(s.size(0), F, generator=torch.Generator().manual_seed(7), dtype=torch.float64)
    K = s.size(1)
    up = C.upstream(B, K, F, 3)
    ref = _oracle_pool(ei, w, s, x, batch, B, alpha, hosc_ortho, flags, up)
    got = _device_pool(ei, w, s, x, batch, alpha, hosc_ortho, flags, up, torch.float32)
    _check_pool(*got, ref, 1e-4, 1e-5)
    # the batched device path on to_dense_adj of the same graphs meets the same oracle bounds (dense leaves: dA)
    adj, S, X, mask = (t.detach().float() if t.is_floating_point() else t for t in ref[4])
    leaves = tuple(t.to(DEV).requires_grad_(True) for t in (X, adj, S))
    fl = dict(flags, adj_transpose=False)
    xp, ap, loss = T.hosc_pool(*leaves, mask.to(DEV), MU, alpha, hosc_ortho, **fl)
    torch.testing.assert_close(torch.stack([loss[k] for k in KEYS.values()]).detach().cpu().double(), ref[2],
                               rtol=1e-5, atol=0.0)
    torch.testing.assert_close(ap.detach().cpu().double(), ref[1], rtol=1e-5, atol=1e-5 * float(ref[1].abs().max()))


@pytest.mark.parametrize("hosc_ortho", [False, True])
@pytest.mark.parametrize("case", ["ragged", "directed"])
def test_pool_bf16_parity(case, hosc_ortho):
    ei, w, s, batch, B = CASES[case](bf16=True)
    F = 32
    x = torch.randn(s.size(0), F, generator=torch.Generator().manual_seed(8), dtype=torch.float64)
    s, x = s.bfloat16().double(), x.bfloat16().double()  # the oracle sees the rounded operands
    up = tuple(v.bfloat16().float() for v in C.upstream(B, s.size(1), F, 4))
    ref = _oracle_pool(ei, w, s, x, batch, B, 0.5, hosc_ortho, FLAGSETS[0], up)
    got = _device_pool(ei, w, s, x, batch, 0.5, hosc_ortho, FLAGSETS[0], up, torch.bfloat16)
    _check_pool(*got, ref, 2e-2, 2e-2, 2e-2)


def _coalesced(ei, n, w=None):
    """(row, col, w, row_ptr, col_ptr, col_order) of one graph on the device, as hosc_losses_unbatched builds them."""
    w = torch.ones(ei.size(1), device=DEV) if w is None else w
    slot = torch.arange(n, device=DEV)
    eic, wc, _, _, _, _ = OPS.remap_coalesce(ei[0].contiguous(), ei[1].contiguous(), w, slot, None, None, n, n, L.SUM,
                                             0, -1.0, False, False)
    _, row_ptr = F_.build_csr(eic[0], n)
    col_order, col_ptr = F_.build_csr(eic[1], n)
    return eic[0], eic[1], wc, row_ptr, col_ptr, col_order


def _motif_check(ei, n, w=None):
    row, col, wc, rp, cp, co = _coalesced(ei, n, w)
    s3 = torch.softmax(torch.randn(1, n, 4, device=DEV), -1)
    nnz = row.numel()
    _, _, saved = OPS._T.hosc_losses_sparse(row, col, wc, rp, cp, co, s3, None, 2, 1e-8)
    P = saved[: 4 * nnz].view(torch.float32).double().cpu().numpy()
    r, c, wv = (np.array(t.cpu().numpy()) for t in (row, col, wc.double()))  # writable copies for scipy indexing
    A = sp.csr_matrix((wv, (r, c)), shape=(n, n))
    Aabs = sp.csr_matrix((np.abs(wv), (r, c)), shape=(n, n))
    pat = sp.csr_matrix((np.ones_like(wv), (r, c)), shape=(n, n))
    exp = np.asarray((A @ A)[r, c]).reshape(-1)
    mag = np.asarray((Aabs @ Aabs)[r, c]).reshape(-1)
    terms = np.asarray((pat @ pat)[r, c]).reshape(-1)
    err = np.abs(P - exp)
    bound = (terms + 1) * 2.0 ** -24 * mag
    assert np.all(err <= bound), (float((err - bound).max()), int((err > bound).sum()))
    return nnz, int(terms.sum())


def test_motif_weights_power_law_with_hubs():
    import bench

    n = 200_000
    ei = bench.powerlaw_graph(n, 1_200_000, DEV, seed=3)
    w = torch.rand(ei.size(1), device=DEV) + 0.5
    nnz, work = _motif_check(ei, n, w)
    assert nnz >= 1_000_000 and work > 0


def test_motif_weights_directed():
    g = torch.Generator(device=DEV).manual_seed(4)
    n = 3000
    ei = torch.randint(0, n, (2, 60_000), device=DEV, generator=g)
    _motif_check(ei, n, torch.randn(ei.size(1), device=DEV, generator=g))


def _step(ei, w, s, x, batch):
    for t in (w, s, x):
        t.grad = None
    xp, ap, loss = U.hosc_pool_unbatched(x, ei, w, s, batch, None, MU, 0.5, True)
    (xp.sum() + ap.square().sum() + loss["hosc_loss"] + loss["ortho_loss"]).backward()
    return xp, ap, loss["hosc_loss"], loss["ortho_loss"]


def test_deterministic():
    import bench

    n = 20_000
    ei = bench.powerlaw_graph(n, 400_000, DEV, seed=5)
    w = (torch.rand(ei.size(1), device=DEV) + 0.5).requires_grad_(True)
    s = torch.softmax(torch.randn(n, 16, device=DEV), -1).requires_grad_(True)
    x = torch.randn(n, 8, device=DEV).requires_grad_(True)
    batch = torch.zeros(n, dtype=torch.long, device=DEV)
    C.assert_deterministic(lambda: _step(ei, w, s, x, batch), [w, s, x])


@pytest.mark.parametrize("need_w", [False, True])
def test_no_motif_work_when_alpha_is_zero(need_w):
    ei, w, s, batch, _ = CASES["ragged"]()

    def names(alpha):
        wd = w.float().to(DEV).requires_grad_(need_w)
        sd = s.float().to(DEV).requires_grad_(True)
        torch.cuda.synchronize()
        L.time_kernel("*")
        try:
            U.hosc_losses_unbatched(ei.to(DEV), wd, sd, batch.to(DEV), alpha, False).sum().backward()
            return [n for n, _ in L.kernel_trace()]
        finally:
            L.time_kernel(None)

    got = names(0.0)
    assert "k_hosc_stats" in got and "k_hosc_ds_elementwise" in got
    assert not any("isect" in n for n in got), got
    got = names(0.5)
    assert sum("k_hosc_isect_warp" in n for n in got) == (2 if need_w else 1), got


def _abi_inputs(n=300, e=3000, K=16, dtype=torch.float32):
    g = torch.Generator(device=DEV).manual_seed(6)
    ei = torch.randint(0, n, (2, e), device=DEV, generator=g)
    row, col, wc, rp, cp, co = _coalesced(ei, n, torch.rand(e, device=DEV, generator=g))
    s3 = torch.softmax(torch.randn(1, n, K, device=DEV, generator=g), -1).to(dtype)
    return row, col, wc, rp, cp, co, s3


def _fwd(inp, terms, saved_b, ws_b):
    row, col, wc, rp, cp, co, s3 = inp
    B, N, K = s3.shape
    lib = L.load()
    dt = L.dtype_code(s3.dtype)
    saved = torch.full((saved_b,), 7, dtype=torch.uint8, device=DEV)
    ws = torch.full((ws_b,), 7, dtype=torch.uint8, device=DEV)
    losses = torch.zeros(3, device=DEV)
    as1 = torch.zeros(B, N, (K + 8) // 8 * 8, device=DEV)
    gn = torch.full((B,), float(N), device=DEV)
    before = lib.tgpb200_debug_launch_count()
    rc = lib.tgpb200_hosc_sparse_loss_fwd(L.ptr(row), L.ptr(col), L.ptr(wc), L.ptr(rp), L.ptr(cp), L.ptr(co),
                                          L.ptr(s3), L.ptr(gn), B, N, K, row.numel(), dt, terms, 1e-8, L.ptr(losses),
                                          L.ptr(as1), L.ptr(saved), saved_b, L.ptr(ws), ws_b, L.stream())
    return rc, lib.tgpb200_debug_launch_count() - before, losses, as1, saved, gn


def _bwd(inp, terms, saved, saved_b, gn, ws_b, gas, need_w):
    row, col, wc, rp, cp, co, s3 = inp
    B, N, K = s3.shape
    lib = L.load()
    dt = L.dtype_code(s3.dtype)
    ws = torch.full((ws_b,), 7, dtype=torch.uint8, device=DEV)
    gl = torch.tensor([0.7, -1.1, 0.4], device=DEV)
    gs = torch.zeros_like(s3)
    gw = torch.zeros(row.numel(), device=DEV)
    before = lib.tgpb200_debug_launch_count()
    rc = lib.tgpb200_hosc_sparse_loss_bwd(L.ptr(row), L.ptr(col), L.ptr(wc), L.ptr(rp), L.ptr(cp), L.ptr(co),
                                          L.ptr(s3), L.ptr(gn), L.ptr(saved), saved_b, L.ptr(gl), L.ptr(gas), B, N, K,
                                          row.numel(), dt, terms, L.ptr(gs), L.ptr(gw) if need_w else None, L.ptr(ws),
                                          ws_b, L.stream())
    return rc, lib.tgpb200_debug_launch_count() - before, gs, gw


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
@pytest.mark.parametrize("terms", [1, 3, 6, 7])
def test_workspace_contract(terms, dtype):
    """Each entry point runs with the queried bytes and gives the same outputs with twice as many; 256 bytes less in
    any one buffer returns TGPB200_ERR_WORKSPACE (-2) before any launch."""
    inp = _abi_inputs(dtype=dtype)
    row, s3 = inp[0], inp[6]
    B, N, K = s3.shape
    nnz = row.numel()
    lib = L.load()
    dt = L.dtype_code(dtype)
    sb = lib.tgpb200_hosc_sparse_loss_saved_bytes(B, N, K, nnz, terms)
    fb = lib.tgpb200_hosc_sparse_loss_fwd_workspace_bytes(B, N, K, nnz, terms, dt)
    rc, launches, losses, as1, saved, gn = _fwd(inp, terms, sb, fb)
    assert rc == 0 and launches > 0
    rc2, _, losses2, as12, _, _ = _fwd(inp, terms, 2 * sb, 2 * fb)
    assert rc2 == 0 and torch.equal(losses, losses2) and torch.equal(as1, as12)
    for short in ((sb - 256, fb), (sb, fb - 256)):
        rc3, launches3, *_ = _fwd(inp, terms, *short)
        assert rc3 == -2 and launches3 == 0, (short, rc3, launches3)
    torch.cuda.synchronize()
    gas = torch.randn_like(as1)
    for has_gas, need_w in ((False, False), (True, True), (False, True)):
        bb = lib.tgpb200_hosc_sparse_loss_bwd_workspace_bytes(B, N, K, nnz, terms, dt, int(has_gas), int(need_w))
        g = gas if has_gas else None
        rc, launches, gs, gw = _bwd(inp, terms, saved, sb, gn, bb, g, need_w)
        assert rc == 0 and launches > 0
        rc2, _, gs2, gw2 = _bwd(inp, terms, saved, sb, gn, 2 * bb, g, need_w)
        assert rc2 == 0 and torch.equal(gs, gs2) and torch.equal(gw, gw2)
        for sbs, bbs in ((sb - 256, bb), (sb, bb - 256)):
            rc3, launches3, _, _ = _bwd(inp, terms, saved, sbs, gn, bbs, g, need_w)
            assert rc3 == -2 and launches3 == 0, (sbs, bbs, rc3, launches3)


def test_memory_of_a_200k_node_graph():
    """N = 200 000, E ~ 4 M, K = 64: forward + backward in a few GB (the dense adjacency alone would be 160 GB); the
    extra peak stays within the bytes the entry points report plus the padded S copies and the outputs, and the losses
    match the sparse float64 restatement."""
    n, e, K = 200_000, 4_000_000, 64
    g = torch.Generator(device=DEV).manual_seed(9)
    src = torch.randint(0, n, (e // 2,), device=DEV, generator=g)
    dst = torch.randint(0, n, (e // 2,), device=DEV, generator=g)
    ei = torch.stack([torch.cat([src, dst]), torch.cat([dst, src])])
    w = (torch.rand(e // 2, device=DEV, generator=g) + 0.5).repeat(2).requires_grad_(True)
    s = torch.softmax(torch.randn(n, K, device=DEV, generator=g), -1).requires_grad_(True)
    torch.cuda.synchronize()
    torch.cuda.reset_peak_memory_stats()
    base = torch.cuda.memory_allocated()
    losses = U.hosc_losses_unbatched(ei, w, s, None, 0.5, True, num_graphs=1, max_num_nodes=n)
    losses.sum().backward()
    torch.cuda.synchronize()
    extra = torch.cuda.max_memory_allocated() - base
    lib = L.load()
    nnz = e  # upper bound of the coalesced edge count
    K1 = (K + 8) // 8 * 8
    reported = (lib.tgpb200_hosc_sparse_loss_saved_bytes(1, n, K, nnz, 7)
                + lib.tgpb200_hosc_sparse_loss_fwd_workspace_bytes(1, n, K, nnz, 7, L.F32)
                + lib.tgpb200_hosc_sparse_loss_bwd_workspace_bytes(1, n, K, nnz, 7, L.F32, 0, 1)
                + lib.tgpb200_remap_coalesce_workspace_bytes(e, n)
                + lib.tgpb200_build_csr_workspace_bytes(e, n))
    edges = nnz * (2 * 8 + 4 + 4 + 4) + e * (4 + 4 + 8)  # coalesced list, weights, CSRs, slots, gradients
    padded = 3 * n * K * 4 + 2 * n * K1 * 4  # s3, its gradient, dS; as1 and its cotangent
    assert extra <= reported + edges + padded, (extra, reported, edges, padded)
    assert extra < 8e9
    exp, _, _ = SO.forward_backward(ei.cpu().numpy(), w.detach().cpu().numpy(), s.detach().cpu().numpy(),
                                    np.zeros(n, dtype=np.int64), 1, terms=7, grads=False)
    torch.testing.assert_close(losses.detach().cpu().double(), torch.tensor(exp), rtol=1e-5, atol=0.0)
    assert torch.isfinite(w.grad).all() and torch.isfinite(s.grad).all()


def test_argument_errors():
    ei, w, s, batch, _ = CASES["ragged"]()
    ei, w, s, batch = ei.to(DEV), w.float().to(DEV), s.float().to(DEV), batch.to(DEV)
    with pytest.raises(ValueError, match="K >= 2"):
        U.hosc_losses_unbatched(ei, w, s[:, :1].contiguous(), batch)
    with pytest.raises(RuntimeError, match="CUDA"):
        U.hosc_losses_unbatched(ei.cpu(), w.cpu(), s.cpu(), batch.cpu())
    with pytest.raises(RuntimeError, match="dtype"):
        U.hosc_losses_unbatched(ei, w, s.half(), batch)
