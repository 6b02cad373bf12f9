"""CPU: the float64 sparse restatement of HOSC pooling (``hosc_sparse_oracle``) equals ``hosc_oracle`` plus torch
autograd on the densified inputs -- losses, dS and the gradient of every input edge weight -- on ragged batches with
self loops, duplicate, zero- and negative-weight edges, directed edges, an isolated node, a triangle-free and an
edgeless graph, for alpha in {0, 0.5, 1} and both orthogonality terms; the sparse ops are registered and refuse CPU
tensors."""
import numpy as np
import pytest
import torch

import hosc_oracle as O
import hosc_sparse_oracle as SO


def _cases():
    yield "ragged", SO.random_case([7, 5, 9], 4.0, 4, seed=1)
    yield "directed", SO.random_case([12, 6], 3.0, 3, seed=2, directed=True)
    # graph 0: a triangle plus an isolated node; graph 1: a 4-cycle (no triangle); graph 2: no edge at all
    ei = torch.tensor([[0, 1, 1, 2, 2, 0, 4, 5, 5, 6, 6, 7, 7, 4],
                       [1, 0, 2, 1, 0, 2, 5, 4, 6, 5, 7, 6, 4, 7]])
    w = torch.tensor([1.0, 1.0, 0.5, 0.5, 2.0, 2.0, 1.0, 1.0, 1.5, 1.5, 1.0, 1.0, 0.7, 0.7], dtype=torch.float64)
    batch = torch.tensor([0, 0, 0, 0, 1, 1, 1, 1, 2, 2, 2])
    s = torch.softmax(torch.randn(11, 3, generator=torch.Generator().manual_seed(3), dtype=torch.float64), -1)
    yield "isolated_trianglefree_edgeless", (ei, w, s, batch, 3)


CASES = list(_cases())


def _dense_reference(ei, w, s, batch, B, alpha, hosc_ortho, g):
    """hosc_oracle on to_dense_adj / to_dense_batch, and autograd's dS and d edge_weight."""
    wl, sl = w.clone().requires_grad_(True), s.clone().requires_grad_(True)
    adj, S, mask = SO.densify(ei, wl, sl, batch, B)
    losses = O.hosc_losses(adj, S, mask)
    keep = torch.tensor([alpha != 1.0, alpha != 0.0, hosc_ortho], dtype=torch.float64)
    losses = losses * keep
    (losses * torch.tensor(g, dtype=torch.float64)).sum().backward()
    return losses.detach(), sl.grad, wl.grad


@pytest.mark.parametrize("hosc_ortho", [False, True])
@pytest.mark.parametrize("alpha", [0.0, 0.5, 1.0])
@pytest.mark.parametrize("name,case", CASES, ids=[c[0] for c in CASES])
def test_sparse_restatement_matches_dense_oracle(name, case, alpha, hosc_ortho):
    ei, w, s, batch, B = case
    g = (0.7, -1.3, 0.9)
    terms = (1 if alpha != 1.0 else 0) | (2 if alpha != 0.0 else 0) | (4 if hosc_ortho else 0)
    exp_l, exp_ds, exp_dw = _dense_reference(ei, w, s, batch, B, alpha, hosc_ortho, g)
    got_l, got_ds, got_dw = SO.forward_backward(ei.numpy(), w.numpy(), s.numpy(), batch.numpy(), B, g, terms)
    assert np.all(np.isfinite(got_l))
    np.testing.assert_allclose(got_l, exp_l.numpy(), rtol=1e-10, atol=1e-12)
    np.testing.assert_allclose(got_ds, exp_ds.numpy(), rtol=1e-9, atol=1e-12)
    np.testing.assert_allclose(got_dw, exp_dw.numpy(), rtol=1e-9, atol=1e-12)


def test_hand_values():
    """Disjoint triangles with a one-hot S: L1 = L2 = -1, O = 0; a 4-cycle split in two pairs: L1 = -1/2, L2 = 0."""
    tri = [(i, j) for comp in ([0, 1, 2], [3, 4, 5]) for i in comp for j in comp if i != j]
    s = np.zeros((6, 2))
    s[:3, 0] = s[3:, 1] = 1.0
    got, _, _ = SO.forward_backward(np.array(tri).T, None, s, np.zeros(6, dtype=np.int64), 1)
    np.testing.assert_allclose(got, [-1.0, -1.0, 0.0], atol=1e-7)
    cyc = [(i, (i + 1) % 4) for i in range(4)] + [((i + 1) % 4, i) for i in range(4)]
    s = np.zeros((4, 2))
    s[:2, 0] = s[2:, 1] = 1.0
    got, _, _ = SO.forward_backward(np.array(cyc).T, None, s, np.zeros(4, dtype=np.int64), 1)
    np.testing.assert_allclose(got[:2], [-0.5, 0.0], atol=1e-7)


def test_motif_weights_of_a_directed_triangle():
    """A directed 3-cycle 0 -> 1 -> 2 -> 0 has no (A A) . A mass (paths of length 2 run against the edges); adding
    the chord 0 -> 2 gives P(0, 2) = w01 w12 and nothing else."""
    row, col, w = np.array([0, 1, 2]), np.array([1, 2, 0]), np.array([2.0, 3.0, 5.0])
    P, wM = SO.motif_weights(row, col, w, 3)
    assert np.all(P == 0) and np.all(wM == 0)
    row, col, w = np.array([0, 0, 1, 2]), np.array([1, 2, 2, 0]), np.array([2.0, 7.0, 3.0, 5.0])
    P, wM = SO.motif_weights(row, col, w, 3)
    np.testing.assert_array_equal(P, [0.0, 6.0, 0.0, 0.0])
    np.testing.assert_array_equal(wM, [0.0, 42.0, 0.0, 0.0])


def test_sparse_ops_registered_and_cpu_raises():
    from tgp_b200 import ops, unbatched

    for name in ("hosc_losses_sparse", "hosc_losses_sparse_bwd"):
        assert name in ops.OP_NAMES and hasattr(torch.ops.tgp_b200, name)
    ei, w, s, batch, B = CASES[0][1]
    with pytest.raises(RuntimeError, match="CUDA"):
        unbatched.hosc_losses_unbatched(ei, w.float(), s.float(), batch)
    with pytest.raises(RuntimeError, match="CUDA"):
        unbatched.hosc_pool_unbatched(torch.randn(s.size(0), 4), ei, w.float(), s.float(), batch)
    i64, i32 = torch.zeros(4, dtype=torch.long), torch.zeros(5, dtype=torch.int32)
    with pytest.raises(NotImplementedError):  # no CPU kernel behind the op
        torch.ops.tgp_b200.hosc_losses_sparse(i64, i64, torch.zeros(4), i32, i32, i32[:4], torch.zeros(1, 4, 2), None,
                                              3, 1e-8)


def test_abi_size_queries_grow_with_the_work_they_carve():
    from tgp_b200 import _lib as L

    lib = L.load()
    base = lib.tgpb200_hosc_sparse_loss_saved_bytes(2, 100, 16, 1000, 1)
    assert lib.tgpb200_hosc_sparse_loss_saved_bytes(2, 100, 16, 1000, 3) >= base + 2 * 4 * 1000
    f32 = lib.tgpb200_hosc_sparse_loss_fwd_workspace_bytes(2, 100, 16, 1000, 3, L.F32)
    assert f32 > lib.tgpb200_hosc_sparse_loss_fwd_workspace_bytes(2, 100, 16, 1000, 1, L.F32) > 0
    assert lib.tgpb200_hosc_sparse_loss_fwd_workspace_bytes(2, 100, 16, 1000, 3, L.BF16) < f32
    full = lib.tgpb200_hosc_sparse_loss_bwd_workspace_bytes(2, 100, 16, 1000, 3, L.F32, 1, 1)
    assert full > lib.tgpb200_hosc_sparse_loss_bwd_workspace_bytes(2, 100, 16, 1000, 3, L.F32, 0, 0) > 0
