"""Float64 restatement of HOSC pooling on a sparse adjacency (``tgp_b200.unbatched.hosc_losses_unbatched``) with scipy
sparse matrices and explicit forward and backward formulas: the motif weights ``P = (A A)`` on A's pattern and
``A_M = P . A``, the two cuts, the orthogonality term, ``dS`` and the gradient of every input edge weight.  It is
checked against ``hosc_oracle`` plus torch autograd on the densified inputs (tests/test_hosc_unbatched_cpu.py), so
the GPU tests can use it where the dense adjacency would not fit.

Layout: node i of graph b is row ``b * nmax + (i - ptr[b])`` of a padded ``[B * nmax]`` index space; duplicates add
up (``to_dense_adj``), self loops and zero-weight entries stay on the pattern."""
import math

import numpy as np
import scipy.sparse as sp
import torch

EPS = 1e-8


def layout(batch: np.ndarray, B: int):
    """(slot [N], counts [B], nmax): each node's row in the padded layout."""
    counts = np.bincount(batch, minlength=B)
    ptr = np.concatenate([[0], np.cumsum(counts)])
    nmax = max(int(counts.max()) if len(batch) else 1, 1)
    slot = batch * nmax + (np.arange(len(batch)) - ptr[batch])
    return slot, counts, nmax


def coalesce(edge_index: np.ndarray, edge_weight: np.ndarray, slot: np.ndarray, R: int):
    """(row, col, w, inv): the coalesced edges sorted by (row, col), duplicates summed, and each input edge's run."""
    r, c = slot[edge_index[0]], slot[edge_index[1]]
    keys, inv = np.unique(r.astype(np.int64) * R + c, return_inverse=True)
    w = np.bincount(inv, weights=edge_weight.astype(np.float64), minlength=len(keys))
    return keys // R, keys % R, w, inv.reshape(-1)


def _mat(row, col, val, R):
    return sp.csr_matrix((val, (row, col)), shape=(R, R))


def _at(M, row, col):
    """M[row_e, col_e] for every e (0 off M's stored pattern)."""
    return np.asarray(M[row, col]).reshape(-1) if len(row) else np.zeros(0)


def motif_weights(row, col, w, R):
    """(P_e, wM_e) = ((A A)_ij, (A A)_ij w_e) on A's pattern."""
    A = _mat(row, col, w, R)
    P = _at(A @ A, row, col)
    return P, P * w


def forward_backward(edge_index, edge_weight, s, batch, B, g=(1.0, 1.0, 1.0), terms=7, eps=EPS, grads=True):
    """Float64 [L1, L2, O], dS [N, K] and d edge_weight [E] for the upstream loss gradients ``g``; a term outside
    ``terms`` (1 first order, 2 motif, 4 orthogonality) is 0 and contributes nothing.  ``grads=False`` returns the
    losses only (dS and d edge_weight None)."""
    ei = np.asarray(edge_index, dtype=np.int64).reshape(2, -1)
    ew = np.ones(ei.shape[1]) if edge_weight is None else np.asarray(edge_weight, dtype=np.float64)
    S_in = np.asarray(s, dtype=np.float64)
    batch = np.asarray(batch, dtype=np.int64)
    N, K = S_in.shape
    slot, counts, nmax = layout(batch, B)
    R = B * nmax
    row, col, w, inv = coalesce(ei, ew, slot, R)
    S = np.zeros((R, K))
    S[slot] = S_in
    gof = np.arange(R) // nmax  # graph of every padded row

    def per_graph(v):  # [R, K] -> [B, K]
        return v.reshape(B, nmax, -1).sum(1)

    A = _mat(row, col, w, R)
    P = _at(A @ A, row, col)
    wM = P * w
    AM = _mat(row, col, wM, R)
    out, dS = np.zeros(3), np.zeros((R, K))
    gA = np.zeros(len(w))
    sq = per_graph(S * S)
    for t, (M, gt) in enumerate(((A, g[0]), (AM, g[1]))):
        if not terms & (1 << t):
            continue
        d = np.asarray(M.sum(1)).reshape(-1)
        MS = M @ S
        n = per_graph(S * MS)
        m = per_graph(d[:, None] * S * S) + eps
        out[t] = float(np.mean(-(n / m).sum(1) / K))
        if not grads:
            continue
        alpha = -gt / (K * B * m)  # dL/dn
        beta = gt * n / (K * B * m * m)  # dL/dm
        Sx = S * alpha[gof]
        dS += M @ Sx + M.T @ Sx + 2.0 * d[:, None] * S * beta[gof]
        r = (S * S * beta[gof]).sum(1)
        G = (Sx[row] * S[col]).sum(1) + r[row]  # dL/dM_ij on the pattern
        if t == 0:
            gA += G
        else:  # A_M = (A A) . A:  dA_ij = G_ij P_ij + (H A^T)_ij + (A^T H)_ij with H = G . A
            H = _mat(row, col, G * w, R)
            gA += G * P + _at(H @ A.T, row, col) + _at(A.T @ H, row, col)
    if terms & 4:
        norms = np.sqrt(sq)
        nb = counts.astype(np.float64)
        out[2] = float(np.mean((math.sqrt(K) - norms.sum(1) / np.sqrt(nb)) / (math.sqrt(K) - 1)))
        with np.errstate(divide="ignore", invalid="ignore"):
            coef = np.where(norms > 0, g[2] / (B * np.sqrt(nb)[:, None] * (math.sqrt(K) - 1) * norms), 0.0)
        dS -= S * coef[gof]
    if not grads:
        return out, None, None
    return out, dS[slot], gA[inv]


def densify(edge_index, edge_weight, s, batch, B):
    """Torch float64 (adj [B, nmax, nmax], S [B, nmax, K], mask) of ``to_dense_adj`` / ``to_dense_batch``, built
    differentiably from ``edge_weight`` and ``s``."""
    bt = torch.as_tensor(np.asarray(batch), dtype=torch.long)
    slot, counts, nmax = layout(bt.numpy(), B)
    slot = torch.as_tensor(slot)
    ei = torch.as_tensor(np.asarray(edge_index), dtype=torch.long).reshape(2, -1)
    w = edge_weight if edge_weight is not None else torch.ones(ei.size(1), dtype=torch.float64)
    r, c = slot[ei[0]], slot[ei[1]]
    adj = torch.zeros(B * nmax * nmax, dtype=torch.float64).index_put(
        ((r // nmax) * nmax * nmax + (r % nmax) * nmax + (c % nmax),), w, accumulate=True).view(B, nmax, nmax)
    S = torch.zeros(B * nmax, s.size(1), dtype=torch.float64).index_put((slot,), s).view(B, nmax, -1)
    mask = torch.arange(nmax)[None, :] < torch.as_tensor(counts)[:, None]
    return adj, S, mask


def random_case(sizes, avg_deg, K, seed, directed=False, dup=0.15, self_loops=0.05, zero=0.03, neg=0.05,
                bf16_weights=False):
    """(edge_index [2, E], edge_weight [E], s [N, K], batch [N], B): graphs of the given node counts with edges inside
    each graph; a share of duplicates, self loops, zero- and negative-weight edges; undirected (both directions, the
    same weight) unless ``directed``.  s is a softmax with a planted community per node."""
    g = torch.Generator().manual_seed(seed)
    rows, cols = [], []
    base = 0
    for n in sizes:
        e = int(avg_deg * n / (1 if directed else 2))
        if n > 0 and e > 0:
            r = torch.randint(0, n, (e,), generator=g) + base
            c = torch.randint(0, n, (e,), generator=g) + base
            loop = torch.rand(e, generator=g) < self_loops
            c = torch.where(loop, r, c)
            rows.append(r)
            cols.append(c)
        base += n
    r = torch.cat(rows) if rows else torch.zeros(0, dtype=torch.long)
    c = torch.cat(cols) if cols else torch.zeros(0, dtype=torch.long)
    w = torch.rand(r.numel(), generator=g, dtype=torch.float64) + 0.5
    w = torch.where(torch.rand(r.numel(), generator=g) < neg, -0.3 * w, w)
    w = torch.where(torch.rand(r.numel(), generator=g) < zero, torch.zeros_like(w), w)
    if not directed:
        r, c, w = torch.cat([r, c]), torch.cat([c, r]), torch.cat([w, w])
    nd = int(dup * r.numel())
    if nd:
        pick = torch.randint(0, r.numel(), (nd,), generator=g)
        r, c = torch.cat([r, r[pick]]), torch.cat([c, c[pick]])
        w = torch.cat([w, torch.rand(nd, generator=g, dtype=torch.float64) + 0.25])
    if bf16_weights:
        w = w.to(torch.bfloat16).double()
    N, B = sum(sizes), len(sizes)
    batch = torch.repeat_interleave(torch.arange(B), torch.tensor(sizes))
    comm = torch.randint(0, K, (N,), generator=g)
    s = torch.softmax(3.0 * torch.nn.functional.one_hot(comm, K).double() + torch.randn(N, K, generator=g,
                                                                                           dtype=torch.float64), -1)
    return torch.stack([r, c]), w, s, batch, B
