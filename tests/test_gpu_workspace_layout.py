"""GPU: every workspace and saved-buffer size query measures exactly what its entry point carves.

Each entry point is called through ctypes with the queried bytes (it must succeed), with twice as many (the outputs
must not change), and, one buffer at a time, with the queried bytes minus 256: that call must return
TGPB200_ERR_WORKSPACE before it enqueues any kernel.  Empty inputs return before they touch the workspace, so they
only take the first two checks."""
import pytest
import torch

from tgp_b200 import _lib as L

pytestmark = pytest.mark.gpu

DEV = "cuda:0"
OK, ERR_WORKSPACE = 0, -2


class _Probed(Exception):
    def __init__(self, rc, launched):
        super().__init__(rc, launched)
        self.rc, self.launched = rc, launched


class _Run:
    """Buffers for one run of a case: `scale` times the queried bytes, or 256 bytes short for the buffer `probe`
    (a key "<entry point>:<argument>"), in which case the call of that entry point ends the run."""

    def __init__(self, scale=1, probe=None):
        self.scale, self.probe, self.sizes = scale, probe, {}

    def buf(self, nbytes, key):
        self.sizes[key] = nbytes
        n = nbytes - 256 if key == self.probe else nbytes * self.scale
        return torch.empty(n, dtype=torch.uint8, device=DEV) if n > 0 else None

    def again(self, t, key):
        """`t` handed to another entry point (a saved buffer, the workspace of a later phase)."""
        nbytes = 0 if t is None else t.numel() // self.scale
        if key == self.probe:
            return self.buf(nbytes, key)
        self.sizes[key] = nbytes
        return t

    def call(self, name, *args):
        before = L.kernel_launches()
        rc = _raw(name, *args)
        if self.probe is not None and self.probe.split(":")[0] == name:
            raise _Probed(rc, L.kernel_launches() - before)
        assert rc == OK, f"{name} returned {rc}"


def _raw(name, *args):
    return getattr(L.load(), name)(*[a.data_ptr() if torch.is_tensor(a) else a for a in args])


def _nb(t):
    return 0 if t is None else t.numel()


def _p(t):
    return None if t is None or t.numel() == 0 else t


def _full(n, value, dtype):
    return torch.full((max(n, 1),), value, dtype=dtype, device=DEV)


def _gen(seed=0):
    return torch.Generator().manual_seed(seed)


# ---------------------------------------------------------------------------------------------------------------
# cases: (run, *shape) -> list of output tensors
# ---------------------------------------------------------------------------------------------------------------
def _csr(r, cluster, K):
    nnz = cluster.numel()
    order, ptr = _full(nnz, -7, torch.int32), _full(K + 1, -7, torch.int32)
    ws = r.buf(L.load().tgpb200_build_csr_workspace_bytes(nnz, K), "tgpb200_build_csr:ws")
    r.call("tgpb200_build_csr", _p(cluster), nnz, K, order, ptr, ws, _nb(ws), L.stream())
    return order, ptr


def case_build_csr(r, nnz, K):
    cluster = torch.randint(0, K, (nnz,), generator=_gen()).to(DEV)
    return list(_csr(r, cluster, K))


def case_segment_reduce_bwd(r, N, K, F, op):
    g = _gen()
    x = torch.randn(N, F, generator=g).to(DEV)
    node = torch.arange(N, device=DEV)
    cluster = torch.randint(0, K, (N,), generator=g).to(DEV)
    order, ptr = _csr(r, cluster, K)
    pool = torch.zeros(K, F, device=DEV)
    assert _raw("tgpb200_segment_reduce_fwd", _p(x), _p(node), None, _p(order), ptr, N, N, K, F, op, L.F32, L.F32, pool,
                L.stream()) == OK
    gpool = torch.randn(K, F, generator=g).to(DEV)
    gx = torch.full((max(N, 1), max(F, 1)), -7.0, device=DEV)
    ws = r.buf(L.load().tgpb200_segment_reduce_bwd_workspace_bytes(N, N, K, F, op), "tgpb200_segment_reduce_bwd:ws")
    r.call("tgpb200_segment_reduce_bwd", _p(x), _p(node), _p(cluster), None, _p(order), ptr, pool, gpool, N, N, K, F,
           op, L.F32, L.F32, gx, None, ws, _nb(ws), L.stream())
    return [gx]


def _edges(E, N, sort_rows=False, seed=0):
    g = _gen(seed)
    row = torch.randint(0, max(N, 1), (E,), generator=g)
    col = torch.randint(0, max(N, 1), (E,), generator=g)
    if sort_rows:
        row = torch.sort(row)[0]
    w = torch.rand(E, generator=g) + 0.5
    return row.to(DEV), col.to(DEV), w.to(DEV)


def case_filter_relabel(r, E, N, kept):
    row, col, w = _edges(E, N)
    node = torch.sort(torch.randperm(N, generator=_gen(1))[:kept])[0].to(DEV)
    out_row, out_col = _full(E, -7, torch.int64), _full(E, -7, torch.int64)
    out_w, src, count = _full(E, -7.0, torch.float32), _full(E, -7, torch.int32), _full(1, -7, torch.int64)
    ws = r.buf(L.load().tgpb200_filter_relabel_onepass_workspace_bytes(E, N), "tgpb200_filter_relabel_onepass:ws")
    r.call("tgpb200_filter_relabel_onepass", _p(row), _p(col), _p(w), E, _p(node), kept, N, L.REMOVE_SELF_LOOPS, 1e-8,
           out_row, out_col, out_w, src, count, ws, _nb(ws), L.stream())
    return [out_row, out_col, out_w, src, count]


def _remap(r, E, N, K, op):
    row, col, w = _edges(E, N)
    cluster = torch.randint(0, K, (N,), generator=_gen(2)).to(DEV)
    count = _full(1, -7, torch.int64)
    ws = r.buf(L.load().tgpb200_remap_coalesce_workspace_bytes(E, K), "tgpb200_remap_coalesce_count:ws")
    r.call("tgpb200_remap_coalesce_count", _p(row), _p(col), _p(w), E, cluster, N, K, op, L.REMOVE_SELF_LOOPS, 1e-8,
           count, ws, _nb(ws), L.stream())
    out_row, out_col, out_w = _full(E, -7, torch.int64), _full(E, -7, torch.int64), _full(E, -7.0, torch.float32)
    slot, run_len = _full(E, -7, torch.int32), _full(E, -7, torch.int32)
    ws = r.again(ws, "tgpb200_remap_coalesce_emit:ws")
    r.call("tgpb200_remap_coalesce_emit", E, K, 1, L.REMOVE_SELF_LOOPS, 1e-8, out_row, out_col, out_w, slot, run_len,
           ws, _nb(ws), L.stream())
    return w, count, [count, out_row, out_col, out_w, slot, run_len]


def case_remap_coalesce(r, E, N, K):
    return _remap(r, E, N, K, L.SUM)[2]


def case_coalesce_bwd(r, E, N, K, op):
    w, count, outs = _remap(r, E, N, K, op)
    n_out = int(count.item())
    gout = torch.randn(max(n_out, 1), generator=_gen(3)).to(DEV)
    gin = _full(E, -7.0, torch.float32)
    ws = r.buf(L.load().tgpb200_coalesce_bwd_workspace_bytes(E, n_out, op), "tgpb200_coalesce_bwd:ws")
    r.call("tgpb200_coalesce_bwd", w, outs[3], gout, outs[4], outs[5], None, E, n_out, op, gin, ws, _nb(ws),
           L.stream())
    return [gin]


def case_bucket_coalesce(r, E, N, K):
    row, col, w = _edges(E, N, sort_rows=True)
    cluster = torch.randint(0, K, (N,), generator=_gen(2)).to(DEV)
    order, ptr = _csr(r, cluster, K)
    plan, count = _full(4, -7, torch.int64), _full(1, -7, torch.int64)
    ws = r.buf(L.load().tgpb200_bucket_coalesce_workspace_bytes(E, N, K), "tgpb200_bucket_coalesce_plan:ws")
    r.call("tgpb200_bucket_coalesce_plan", _p(row), E, cluster, order, ptr, N, K, plan, ws, _nb(ws), L.stream())
    ws = r.again(ws, "tgpb200_bucket_coalesce_count:ws")
    r.call("tgpb200_bucket_coalesce_count", _p(row), _p(col), _p(w), E, cluster, order, ptr, N, K, L.SUM,
           L.REMOVE_SELF_LOOPS, 1e-8, -1, -1, 1, count, ws, _nb(ws), L.stream())
    out_row, out_col, out_w = _full(E, -7, torch.int64), _full(E, -7, torch.int64), _full(E, -7.0, torch.float32)
    slot, run_len, aux = _full(E, -7, torch.int32), _full(E, -7, torch.int32), _full(E, -7.0, torch.float32)
    ws = r.again(ws, "tgpb200_bucket_coalesce_emit:ws")
    r.call("tgpb200_bucket_coalesce_emit", E, N, K, 1, -1, out_row, out_col, out_w, slot, run_len, aux, ws, _nb(ws),
           L.stream())
    return [plan, count, out_row, out_col, out_w, slot, run_len]


def case_edge_norm(r, E, K, rows_sorted):
    row, col, w = _edges(E, K, sort_rows=bool(rows_sorted))
    lib, st = L.load(), L.stream()
    nb = lib.tgpb200_edge_norm_workspace_bytes(E, K)
    deg, w_out = _full(K, -7.0, torch.float32), _full(E, -7.0, torch.float32)
    ws = r.buf(nb, "tgpb200_degree_norm_fwd:ws")
    r.call("tgpb200_degree_norm_fwd", _p(row), _p(col), _p(w), E, None, K, 1e-8, rows_sorted, deg, w_out, ws, _nb(ws),
           st)
    deg2 = _full(K, -7.0, torch.float32)
    ws = r.buf(nb, "tgpb200_degree_accumulate:ws")
    r.call("tgpb200_degree_accumulate", _p(row), _p(w), E, None, K, rows_sorted, deg2, ws, _nb(ws), st)
    gout = torch.randn(max(E, 1), generator=_gen(4)).to(DEV)
    gd, gw = _full(K, -7.0, torch.float32), _full(E, -7.0, torch.float32)
    ws = r.buf(nb, "tgpb200_degree_norm_bwd:ws")
    r.call("tgpb200_degree_norm_bwd", _p(row), _p(col), _p(w), deg, gout, E, None, K, 1e-8, rows_sorted, gd, gw, ws,
           _nb(ws), st)
    gd2 = _full(K, -7.0, torch.float32)
    ws = r.buf(nb, "tgpb200_degree_bwd_accumulate:ws")
    r.call("tgpb200_degree_bwd_accumulate", _p(row), _p(col), _p(w), deg, gout, E, None, K, 1e-8, rows_sorted, gd2, ws,
           _nb(ws), st)
    # weight norm over G graphs of the K pooled nodes
    G = 8
    batch = torch.sort(torch.randint(0, G, (K,), generator=_gen(5)))[0].to(DEV)
    mx, arg, wn = _full(G, -7.0, torch.float32), _full(G, -7, torch.int32), _full(E, -7.0, torch.float32)
    assert _raw("tgpb200_weight_norm_fwd", _p(row), _p(w), batch, E, None, G, mx, arg, wn, st) == OK
    acc, gwn = _full(G, -7.0, torch.float32), _full(E, -7.0, torch.float32)
    ws = r.buf(lib.tgpb200_edge_norm_workspace_bytes(E, max(K, G)), "tgpb200_weight_norm_bwd:ws")
    r.call("tgpb200_weight_norm_bwd", _p(row), _p(w), batch, mx, arg, gout, E, None, K, G, rows_sorted, acc, gwn, ws,
           _nb(ws), st)
    return [deg, w_out, deg2, gd, gw, gd2, acc, gwn]


def case_topk_select(r, N, G):
    g = _gen()
    score = torch.randn(N, generator=g).to(DEV)
    batch = torch.sort(torch.randint(0, G, (N,), generator=g))[0].to(DEV)
    node, cluster, count = _full(N, -7, torch.int64), _full(N, -7, torch.int64), _full(1, -7, torch.int64)
    ws = r.buf(L.load().tgpb200_topk_select_workspace_bytes(N, G), "tgpb200_topk_select:ws")
    r.call("tgpb200_topk_select", _p(score), _p(batch), N, G, 0.5, node, cluster, count, ws, _nb(ws), L.stream())
    return [node, cluster, count]


def case_block_diag(r, B, K):
    g = _gen()
    adj = (torch.rand(B, K, K, generator=g) < 0.3).float().to(DEV)
    mask = (torch.rand(B, K, generator=g) < 0.7).to(torch.uint8).to(DEV)
    n = B * K * K
    valid, count = _full(1, -7, torch.int64), _full(1, -7, torch.int64)
    ws = r.buf(L.load().tgpb200_block_diag_workspace_bytes(B, K), "tgpb200_block_diag_count:ws")
    r.call("tgpb200_block_diag_count", _p(adj), _p(mask), B, K, L.F32, 1e-8, valid, count, ws, _nb(ws), L.stream())
    out_row, out_col = _full(n, -7, torch.int64), _full(n, -7, torch.int64)
    out_w, src = _full(n, -7.0, torch.float32), _full(n, -7, torch.int32)
    ws = r.again(ws, "tgpb200_block_diag_emit:ws")
    r.call("tgpb200_block_diag_emit", _p(adj), _p(mask), B, K, L.F32, 1e-8, out_row, out_col, out_w, src, ws, _nb(ws),
           L.stream())
    return [valid, count, out_row, out_col, out_w, src]


def case_graph_ptr(r, N, B):
    batch = torch.sort(torch.randint(0, B, (N,), generator=_gen()))[0].to(DEV)
    ptr = _full(B + 1, -7, torch.int32)
    ws = r.buf(L.load().tgpb200_graph_ptr_workspace_bytes(B), "tgpb200_graph_ptr:ws")
    r.call("tgpb200_graph_ptr", _p(batch), N, B, ptr, ws, _nb(ws), L.stream())
    return [ptr]


def _dense_inputs(B, N, K, F, dtype):
    g = _gen()
    a = (torch.rand(B, N, N, generator=g) < 0.1).float()
    a = a + a.transpose(1, 2)
    s = torch.softmax(torch.randn(B, N, K, generator=g), -1)
    x = torch.randn(B, N, F, generator=g)
    return [t.to(DEV, dtype) for t in (a, s, x)]


def case_dense_pool(r, B, N, K, F, dtype, grad_adj):
    lib, st, dt = L.load(), L.stream(), L.dtype_code(dtype)
    a, s, x = _dense_inputs(B, N, K, F, dtype)
    xp, ap = torch.zeros(B, K, F, device=DEV, dtype=dtype), torch.zeros(B, K, K, device=DEV, dtype=dtype)
    losses = torch.zeros(4, device=DEV)
    saved = r.buf(lib.tgpb200_dense_pool_saved_bytes(B, N, K), "tgpb200_dense_pool_fwd_v2:saved")
    r.call("tgpb200_dense_pool_fwd_v2", a, s, x, B, N, K, F, dt, 0, 1, 1e-8, 1.0, 1.0, xp, ap, losses, saved,
           _nb(saved), st, None)
    g = _gen(6)
    gxp, gap = torch.randn(B, K, F, generator=g).to(DEV, dtype), torch.randn(B, K, K, generator=g).to(DEV, dtype)
    gl = torch.randn(4, generator=g).to(DEV)
    gs, gx = torch.full_like(s, -7.0), torch.full_like(x, -7.0)
    ga = torch.full_like(a, -7.0) if grad_adj else None
    saved = r.again(saved, "tgpb200_dense_pool_bwd_v2:saved")
    ws = r.buf(lib.tgpb200_dense_pool_bwd_workspace_bytes(B, N, K, int(grad_adj)), "tgpb200_dense_pool_bwd_v2:ws")
    r.call("tgpb200_dense_pool_bwd_v2", a, s, x, gxp, gap, gl, B, N, K, F, dt, 0, 1, 1e-8, 1.0, 1.0, gs, gx, ga, saved,
           _nb(saved), ws, _nb(ws), st, None)
    return [xp, ap, losses, gs, gx] + ([ga] if grad_adj else [])


def case_acc(r, B, N, K, dtype):
    lib, st, dt = L.load(), L.stream(), L.dtype_code(dtype)
    a, s, _ = _dense_inputs(B, N, K, 1, dtype)
    losses, quant = torch.full((2,), -7.0, device=DEV), torch.full((B, K), -7.0, device=DEV, dtype=dtype)
    saved = r.buf(lib.tgpb200_acc_loss_saved_bytes(B, K), "tgpb200_acc_loss_fwd:saved")
    ws = r.buf(lib.tgpb200_acc_loss_fwd_workspace_bytes(B, N, K), "tgpb200_acc_loss_fwd:ws")
    r.call("tgpb200_acc_loss_fwd", a, s, B, N, K, dt, losses, quant, saved, _nb(saved), ws, _nb(ws), st)
    gl = torch.randn(2, generator=_gen(7)).to(DEV)
    gs, ga = torch.full_like(s, -7.0), torch.full_like(a, -7.0)
    saved = r.again(saved, "tgpb200_acc_loss_bwd:saved")
    r.call("tgpb200_acc_loss_bwd", a, s, saved, _nb(saved), gl, B, N, K, dt, gs, ga, st)
    return [losses, quant, gs, ga]


def case_hosc(r, B, N, K, dtype, terms, grad_adj):
    lib, st, dt = L.load(), L.stream(), L.dtype_code(dtype)
    a, s, _ = _dense_inputs(B, N, K, 1, dtype)
    losses = torch.full((3,), -7.0, device=DEV)
    saved = r.buf(lib.tgpb200_hosc_loss_saved_bytes(B, N, K, terms, dt), "tgpb200_hosc_loss_fwd:saved")
    ws = r.buf(lib.tgpb200_hosc_loss_fwd_workspace_bytes(B, N, K, terms, dt), "tgpb200_hosc_loss_fwd:ws")
    r.call("tgpb200_hosc_loss_fwd", a, s, None, B, N, K, dt, terms, 1e-8, losses, saved, _nb(saved), ws, _nb(ws), st)
    gl = torch.randn(3, generator=_gen(8)).to(DEV)
    gs = torch.full_like(s, -7.0)
    ga = torch.full_like(a, -7.0) if grad_adj else None
    saved = r.again(saved, "tgpb200_hosc_loss_bwd:saved")
    ws = r.buf(lib.tgpb200_hosc_loss_bwd_workspace_bytes(B, N, K, dt, int(grad_adj)), "tgpb200_hosc_loss_bwd:ws")
    r.call("tgpb200_hosc_loss_bwd", a, s, None, saved, _nb(saved), gl, B, N, K, dt, terms, gs, ga, ws, _nb(ws), st)
    return [losses, gs] + ([ga] if grad_adj else [])


F32, BF16 = torch.float32, torch.bfloat16
# (case, shape, empty): empty inputs return before they carve anything
CASES = [
    (case_build_csr, (0, 5), False),
    (case_build_csr, (1000, 30), False),
    (case_build_csr, (300_000, 5000), False),
    (case_segment_reduce_bwd, (0, 4, 0, L.SUM), True),
    (case_segment_reduce_bwd, (500, 50, 64, L.SUM), False),
    (case_segment_reduce_bwd, (100_000, 3000, 32, L.MAX), False),
    (case_filter_relabel, (0, 10, 5), False),
    (case_filter_relabel, (4000, 600, 300), False),
    (case_filter_relabel, (2_000_000, 200_000, 100_000), False),
    (case_remap_coalesce, (0, 10, 5), True),
    (case_remap_coalesce, (3000, 600, 200), False),
    (case_remap_coalesce, (2_000_000, 200_000, 100_000), False),
    (case_coalesce_bwd, (3000, 600, 200, L.SUM), False),
    (case_coalesce_bwd, (3000, 600, 200, L.MAX), False),
    (case_bucket_coalesce, (0, 10, 5), False),
    (case_bucket_coalesce, (4000, 600, 200), False),
    (case_bucket_coalesce, (2_000_000, 200_000, 1000), False),
    (case_edge_norm, (0, 5, 1), True),
    (case_edge_norm, (4000, 200, 1), False),
    (case_edge_norm, (4000, 200, 0), False),
    (case_edge_norm, (2_000_000, 100_000, 1), False),
    (case_topk_select, (0, 1), True),
    (case_topk_select, (600, 8), False),
    (case_topk_select, (1_000_000, 128), False),
    (case_block_diag, (0, 4), True),
    (case_block_diag, (4, 32), False),
    (case_block_diag, (64, 64), False),
    (case_graph_ptr, (0, 3), False),
    (case_graph_ptr, (600, 8), False),
    (case_graph_ptr, (1_000_000, 50_000), False),
    (case_dense_pool, (2, 64, 16, 32, F32, True), False),
    (case_dense_pool, (4, 128, 32, 64, BF16, False), False),
    (case_acc, (2, 64, 8, F32), False),
    (case_acc, (3, 200, 16, BF16), False),
    (case_hosc, (2, 64, 8, F32, 3, True), False),
    (case_hosc, (2, 96, 16, BF16, 7, False), False),
]


@pytest.mark.parametrize("case,shape,empty", CASES,
                         ids=[f"{c.__name__[5:]}-{'-'.join(str(x).replace('torch.', '') for x in s)}"
                              for c, s, _ in CASES])
def test_queried_bytes_are_exactly_what_the_call_carves(case, shape, empty):
    exact = _Run()
    out = case(exact, *shape)
    roomy = case(_Run(scale=2), *shape)
    torch.cuda.synchronize()
    for a, b in zip(out, roomy):
        assert torch.equal(a, b)
    if empty:
        return
    for key, nbytes in exact.sizes.items():
        if nbytes < 256:  # nothing to carve (coalesce_bwd of SUM / MEAN)
            continue
        with pytest.raises(_Probed) as probed:
            case(_Run(probe=key), *shape)
        assert probed.value.rc == ERR_WORKSPACE, key
        assert probed.value.launched == 0, key
    torch.cuda.synchronize()
