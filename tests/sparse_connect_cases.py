"""Cases, launch rules and float64 oracle of the sparse connect (``csrc/sparse_connect.cu``, ``csrc/sparse_coalesce.cu``).

``expected_paths`` restates in plain Python how the host code picks the kernels of a ``sparse_connect`` call, each rule
with the line it comes from, and ``CASES`` puts every rule on both sides of its threshold:

* branch (``functional.py:206-211``): kept-node when ``len(node_index) < num_nodes``, cluster otherwise;
* kept-node forward (``sparse_connect.cu:835``): one block (``small``) when ``N <= 32768``, ``kept <= 32768`` and
  ``ceil(E / 2048) + 2 <= 4096`` state words, the one-pass compaction otherwise; backward (``sparse_connect.cu:873``):
  ``k_unfilter_small`` when ``E <= 32768`` and ``num_out <= 32768``;
* cluster (``functional.py:214``, ``ops.py:273``): row-bucketed when the input rows are sorted and
  ``E + N < 2^31 - 1``, the remap (global radix sort) otherwise;
* remap (``sparse_connect.cu:781``): 32-bit keys when ``2 cb <= 32`` (``cb`` = bits of ``K - 1``), 64-bit otherwise;
  the sort runs ``ceil(2 cb / 8)`` passes (``prims.cuh:442``), whose parity decides the buffer the keys end in;
* bucketed (``sparse_coalesce.cu:732``): packed 32-bit rank keys when ``K < 2^21``; coarse rows of more than 512
  virtual entries go to the hub path (``:98``), hub runs of more than 4096 members to ``k_hub_long_runs`` (``:462``);
  exact launch sizes when ``E >= 2^20`` and the call is not padded (``ops.py:281``);
* coalesce backward (``sparse_connect.cu:915``): sum / mean through ``k_coalesce_bwd4`` plus a scalar tail when
  ``E % 4 != 0``, every other op through ``k_coalesce_bwd``; max / min count the ties first;
* mul gradient (``ops.py:295``): exact product rule from ``run_aux`` on the bucketed path, the quotient
  ``g out / w`` on the remap path;
* degree backward (``sparse_connect.cu:985``): the one-pass prepare kernel when the coarse rows are sorted (always, on
  both branches here), two grouped sums otherwise;
* ``k_dsum_spine``: one round of 1024 tiles of 2048 positions, or several when a normalised list has more than
  2,097,152 edges.

``oracle`` computes what the reference computes (``R.sparse_connect_so`` and its autograd) in float64, with the
semantics ``oracle/pyg_shim.py`` restates: the max / min coalesce gradient split evenly among ties, the max-weight
normalisation's gradient through the first occurrence of the maximum, the degree clamp passing the gradient where
``deg >= EPS``.  The maximum of the max-weight normalisation is picked among the float32 values the kernels compare
(``decision32``); its float64 value then enters the oracle.  For every output element the oracle also returns the sum
of the absolute values of its terms (``*_terms``), which the component-wise bounds of the GPU tests scale with.

How the terms are counted.  A float32 result that is a sum of exactly given terms errs by a few units of roundoff u
times the sum of the |terms|; the bound ``|err| <= 1e-5 * terms`` (about 170 u) leaves room for those roundings and
nothing else.  A factor that the forward derives from other sums carries their error with it, and to first order
the relative error of a product is the sum of its factors' relative errors.  So every derived factor f gets a
condition c_f (its relative error in units of u beyond its own rounding) and a product ``t = f_1 f_2 ...`` counts
``|t| (1 + sum c_i)``; a sum counts the sum of its terms'.  The conditions:

* the degree ``deg_v = sum_e wc_e`` has terms ``D_v = sum_e A_e`` (A_e the terms of the coalesced weight: the sum
  of its members' |w|, divided by L for mean; |wc| for max / min / mul and the kept-node branch), so its relative
  error is ``kappa_v = D_v / |deg_v|`` times that of its inputs; ``dinv = deg^(-1/2)`` halves it:
  ``c = kappa / 2``, which is 1/2 when nothing cancels; ``dinv^3`` has ``3 kappa / 2``; a degree under the EPS
  clamp makes ``dinv`` a constant, ``c = 0``;
* ``y = wc dinv_r dinv_c`` counts ``|y| (A / |wc| + c_r + c_c)``: 2 |y| when nothing cancels;
* the maximum ``m = |y_arg|`` of a graph has ``c_m = terms(y_arg) / m - 1``; ``z = y / m`` counts
  ``|z| (1 + c_y + c_m)``, ``1 / m^2`` has ``2 c_m``;
* the backward reuses these factors term by term: ``g / m``, ``acc / m^2`` with ``acc = sum g y`` (terms
  ``sum |g| terms(y)``), ``g dinv_r dinv_c``, ``gdinv_v = sum g wc dinv_other`` and ``0.5 gdinv dinv^3``; then the
  coalesce backward (``/ L`` for mean, ``/ ties`` for max / min, the product of the other members for mul).
"""
from __future__ import annotations

import zlib
from typing import Dict, NamedTuple, Optional

import torch
from torch import Tensor

EPS = 1e-8
OPS = ("sum", "mean", "max", "min", "mul")
SMALL_LIMIT = 32768          # k_kept_init_small / k_unfilter_small
SMALL_STATE_WORDS = 4096     # compaction state words of the one-block kept-node forward
DS_TILE = 2048               # positions per tile of the deterministic sums
SPINE_ROUND = 1024           # tiles per round of k_dsum_spine
PACKED_K = 1 << 21           # k_bucket_tiles<true> below this K
HUB_ENTRIES = 512            # kBkHub
LONG_RUN = 4096              # kBkLongRun
PLAN_SYNC_MIN_EDGES = 1 << 20


class Case(NamedTuple):
    branch: str            # "kept" / "cluster"
    N: int                 # fine nodes
    K: int                 # supernodes (cluster) / kept nodes (kept)
    E: int                 # input edges (approximate for the structured graphs)
    graph: str             # "rand", "tiles", "hub", "dyn"
    values: str            # "none", "rand", "tri" ({0.5, 1, 1.5}), "unit", "signed", "zeros", "dyn"
    op: str = "sum"
    rsl: bool = True
    dn: bool = False
    ewn: bool = False
    sorted_rows: bool = True
    G: int = 4             # graphs of the pooled nodes (max-weight normalisation)
    twice: bool = False    # also run twice and compare bitwise (C4 / C5-shaped)
    seed: int = 0

    @property
    def id(self) -> str:
        flags = "".join(n for n, on in (("rsl", self.rsl), ("dn", self.dn), ("ewn", self.ewn)) if on) or "plain"
        return (f"{self.branch}-{self.graph}-N{self.N}-K{self.K}-E{self.E}-{self.values}-{self.op}-{flags}"
                f"-{'sorted' if self.sorted_rows else 'shuffled'}" + ("-twice" if self.twice else ""))

    @property
    def weighted(self) -> bool:
        return self.values != "none"


def _cases():
    cs = []
    C = lambda *a, **k: Case("cluster", *a, **k)  # noqa: E731
    kept = lambda *a, **k: Case("kept", *a, **k)  # noqa: E731
    # remap path: K on both sides of every key-width / pass-parity threshold, E % 4 in {0, 1, 3}
    for K, E in ((2, 4001), (256, 6000), (257, 6003), (65536, 70001), (65537, 70000), (PACKED_K - 1, 60003),
                 (PACKED_K + 1, 60001)):
        cs.append(C(max(2 * K, 3000) if K < 65536 else 120000, K, E, "rand", "tri", "max", sorted_rows=False))
    # bucketed path: both rank-key forms, E % 4 in {0, 1, 3}
    for K, E in ((256, 6000), (257, 6003), (65537, 70001), (PACKED_K - 1, 60003), (PACKED_K + 1, 60001)):
        cs.append(C(max(2 * K, 3000) if K < 65536 else 120000, K, E, "rand", "tri", "max"))
    # every op on both coalesce paths, weighted with ties and unweighted, with and without self loops, both norms
    for op in OPS:
        for srt in (True, False):
            cs.append(C(3000, 700, 20001, "rand", "tri", op, sorted_rows=srt))
            cs.append(C(3000, 700, 20003, "rand", "tri", op, rsl=False, dn=True, ewn=True, sorted_rows=srt))
            cs.append(C(3000, 700, 20000, "rand", "zeros", op, sorted_rows=srt))
        cs.append(C(3000, 700, 20001, "rand", "none", op, dn=True, sorted_rows=op != "sum"))
        cs.append(C(3000, 700, 20003, "rand", "rand", op, rsl=False, dn=True))
        cs.append(C(3000, 700, 20000, "rand", "unit", op, ewn=True, sorted_rows=op in ("max", "min")))
        # hub rows (more than 512 entries) and a run of more than 4096 duplicates
        cs.append(C(20000, 3001, 60001, "hub", "tri", op))
    cs.append(C(20000, 3001, 60003, "hub", "rand", "sum", rsl=False, dn=True, ewn=True))
    cs.append(C(3000, 700, 20001, "rand", "signed", "max", dn=True, ewn=True))
    cs.append(C(3000, 700, 20001, "rand", "signed", "min", dn=True, sorted_rows=False))
    # exact launch sizes (E >= 2^20, unpadded) against capacity launches (padded)
    cs.append(C(400000, 150001, 1100001, "rand", "rand", "sum", dn=True))
    # several spine rounds: about 3e6 coarse edges, sorted rows, both norms
    cs.append(C(1500000, 1000003, 3000001, "rand", "rand", "sum", dn=True, ewn=True, G=16))
    # kept-node branch: one-block and one-pass forward, small and large backward, tile-aligned segments
    cs.append(kept(3000, 1700, 20003, "rand", "tri", dn=True, ewn=True))
    cs.append(kept(3000, 1700, 20001, "rand", "unit", rsl=False, dn=True, ewn=True))
    cs.append(kept(3000, 1700, 20000, "rand", "none", dn=True))
    cs.append(kept(3000, 1700, 20001, "rand", "signed", dn=True, ewn=True))
    cs.append(kept(32768, 30001, 120001, "rand", "rand", dn=True))
    cs.append(kept(32769, 30001, 120003, "rand", "rand", dn=True, ewn=True))
    cs.append(kept(20000, 19999, 0, "tiles", "tri", rsl=False, dn=True, ewn=True))
    cs.append(kept(20000, 19999, 0, "tiles", "signed", dn=True))
    cs.append(kept(1200000, 1000000, 4500001, "rand", "rand", dn=True, ewn=True, G=16))
    # dynamic range: about 1e5 heavy edges (1e4) sorted first, then light rows (1e-3 .. 1e-4)
    cs.append(kept(60000, 59999, 0, "dyn", "dyn", dn=True, ewn=True))
    cs.append(C(60000, 30000, 0, "dyn", "dyn", "sum", dn=True, ewn=True))
    # C4-shaped (matching-style clusters, mean) and C5-shaped (TopK 50 %, degree norm), run twice
    cs.append(C(40000, 22003, 400001, "rand", "rand", "mean", dn=True, twice=True))
    cs.append(kept(70001, 35001, 700003, "rand", "rand", dn=True, twice=True))
    return cs


CASES = _cases()


# --------------------------------------------------------------------------- #
# inputs
# --------------------------------------------------------------------------- #
def _gen(case: Case) -> torch.Generator:
    return torch.Generator().manual_seed(zlib.crc32(case.id.encode()) + case.seed)


def _tile_rows(N: int):
    """Row lengths whose runs start and end on 2048-position tile and 256-position warp boundaries, and some that
    straddle them."""
    lens = [2048, 256, 256, 256, 256, 256, 256, 256, 256, 4096, 1, 2047, 255, 1, 1792, 2049, 2047, 256, 3, 253,
            6144, 7, 9, 17, 223, 1792]
    lens = lens + [5] * 300 + [1] * 100 + [2048, 2048, 256]
    assert len(lens) <= N - 1
    return lens


def _graph(case: Case, g: torch.Generator):
    """(row, col) of the input edge list in row order."""
    N = case.N
    if case.graph == "rand":
        row = torch.randint(0, N, (case.E,), generator=g)
        col = torch.randint(0, N, (case.E,), generator=g)
        row = torch.sort(row).values
        return row, col
    if case.graph == "hub":
        E = case.E
        row = torch.randint(0, N, (E,), generator=g)
        col = torch.randint(0, N, (E,), generator=g)
        # node 0: 5000 edges into node 1 (one coarse run of more than 4096 duplicates), node 2: 800 distinct columns
        row[:5000], col[:5000] = 0, 1
        row[5000:5800], col[5000:5800] = 2, torch.randperm(N, generator=g)[:800]
        return torch.sort(row, stable=True).values, col[torch.sort(row, stable=True).indices]
    if case.graph == "tiles":
        lens = torch.tensor(_tile_rows(N))
        row = torch.repeat_interleave(torch.arange(lens.numel()), lens)
        col = torch.randint(0, N - 1, (row.numel(),), generator=g)
        return row, col
    if case.graph == "dyn":
        heavy_rows, heavy_per_row = 1000, 100
        light_rows = N // 2 - heavy_rows
        rh = torch.repeat_interleave(torch.arange(heavy_rows), heavy_per_row)
        per = 1 + torch.randint(0, 3, (light_rows,), generator=g)
        rl = torch.repeat_interleave(torch.arange(heavy_rows, heavy_rows + light_rows), per)
        row = torch.cat([rh, rl])
        col = torch.randint(0, N - 1, (row.numel(),), generator=g)
        return row, col
    raise ValueError(case.graph)


def _weights(case: Case, row: Tensor, g: torch.Generator) -> Optional[Tensor]:
    E = row.numel()
    v = case.values
    if v == "none":
        return None
    if v == "rand":
        return torch.rand(E, generator=g) + 0.5
    if v == "unit":
        return torch.ones(E)
    if v in ("tri", "zeros"):
        w = torch.tensor([0.5, 1.0, 1.5])[torch.randint(0, 3, (E,), generator=g)]
        if v == "zeros":
            w[torch.randperm(E, generator=g)[: E // 50]] = 0.0
        return w
    if v == "signed":
        w = (torch.rand(E, generator=g) + 0.5) * torch.where(torch.rand(E, generator=g) < 0.3, -1.0, 1.0)
        return w
    if v == "dyn":
        heavy = row < 1000
        light = 10.0 ** -(3 + torch.rand(E, generator=g))
        return torch.where(heavy, torch.full((E,), 1e4), light).float()
    raise ValueError(v)


def _signed_rows(case: Case, row: Tensor, col: Tensor, w: Tensor, node: Tensor) -> None:
    """Signed weights on the kept-node branch: one kept row whose degree cancels to exactly 0 and one whose degree
    the EPS clamp catches (the cluster branch takes max / min of signed weights, no cancellation)."""
    kept = torch.zeros(case.N, dtype=torch.bool)
    kept[node] = True
    counts = torch.bincount(row, minlength=case.N)
    starts = torch.cumsum(counts, 0) - counts
    two = torch.nonzero((counts == 2) & kept).flatten()
    for v, (x, y) in zip(two[:2].tolist(), ((0.75, -0.75), (3e-8, -2.5e-8))):
        e = int(starts[v])
        col[e], col[e + 1] = node[(v + 1) % node.numel()], node[(v + 2) % node.numel()]
        col[e] = node[0] if int(col[e]) == v else col[e]
        col[e + 1] = node[1] if int(col[e + 1]) == v else col[e + 1]
        w[e], w[e + 1] = x, y


def inputs(case: Case) -> Dict[str, Optional[Tensor]]:
    """CPU inputs: edge_index [2, E] (rows sorted unless the case shuffles them), weight [E] or None, and the
    selection: ``node_index`` (kept) or ``cluster`` (cluster), ``batch_pooled`` [K] (sorted, G graphs)."""
    g = _gen(case)
    row, col = _graph(case, g)
    w = _weights(case, row, g)
    out = {"node_index": None, "cluster": None}
    if case.branch == "kept":
        if case.graph in ("tiles", "dyn"):
            # every node but the last (which has no edges): the output keeps every edge
            out["node_index"] = torch.arange(case.K)
        else:
            out["node_index"] = torch.sort(torch.randperm(case.N, generator=g)[: case.K]).values
    else:
        if case.graph == "dyn":
            out["cluster"] = torch.arange(case.N) // 2  # monotone: the heavy rows stay first
        elif case.graph == "hub":
            cl = torch.randint(0, case.K, (case.N,), generator=g)
            cl[0], cl[1], cl[2] = 0, 1, 2
            out["cluster"] = cl
        else:
            cl = torch.randint(0, case.K, (case.N,), generator=g)
            if case.K > PACKED_K:  # columns above 2^21 (the unpacked key's high bits)
                cl[: case.N // 2] = PACKED_K - 5 + torch.randint(0, 6, (case.N // 2,), generator=g)
            out["cluster"] = cl
    if case.values == "signed" and case.branch == "kept":
        _signed_rows(case, row, col, w, out["node_index"])
    out["edge_index"], out["w"] = torch.stack([row, col]), w
    if out["edge_index"].size(1) >= 3_000_000:
        _straddle_spine_rounds(case, out, g)
    if not case.sorted_rows:
        p = torch.randperm(out["edge_index"].size(1), generator=g)
        out["edge_index"] = out["edge_index"][:, p]
        out["w"] = None if w is None else out["w"][p]
    bp = torch.randint(0, case.G, (case.K,), generator=g)
    bp[: min(case.G, case.K)] = torch.arange(min(case.G, case.K))
    out["batch_pooled"] = torch.sort(bp).values
    return out


def _straddle_spine_rounds(case: Case, out: Dict, g: torch.Generator) -> None:
    """Give the output row at position 1024 * 2048 (the first edge of the second spine round) 5000 more edges, so that
    its run straddles the boundary between two rounds of the spine."""
    row, col = out["edge_index"]
    b = SPINE_ROUND * DS_TILE
    if case.branch == "kept":
        node = out["node_index"]
        table = torch.full((case.N,), -1, dtype=torch.long)
        table[node] = torch.arange(node.numel())
        surv = (table[row] >= 0) & (table[col] >= 0) & (row != col)
        v = int(row[surv][b])
        cols = node[torch.randint(0, node.numel(), (5000,), generator=g)]
    else:
        cl = out["cluster"]
        cr = torch.sort(cl[row][cl[row] != cl[col]]).values
        c_b = int(cr[b])
        v = int(torch.nonzero(cl == c_b)[0])
        cols = torch.randint(0, case.N, (5000,), generator=g)
        cols = cols[cl[cols] != c_b]
    cols = cols[cols != v]
    row = torch.cat([row, torch.full((cols.numel(),), v, dtype=torch.long)])
    col = torch.cat([col, cols])
    order = torch.sort(row, stable=True).indices
    out["edge_index"] = torch.stack([row[order], col[order]])
    if out["w"] is not None:
        extra = torch.rand(cols.numel(), generator=g) + 0.5
        out["w"] = torch.cat([out["w"], extra])[order]


def cotangent(case: Case, n_out: int) -> Tensor:
    return torch.randn(n_out, generator=torch.Generator().manual_seed(zlib.crc32(case.id.encode()) + 7))


# --------------------------------------------------------------------------- #
# the launch rules
# --------------------------------------------------------------------------- #
def _cb(K: int) -> int:
    return max(1, (K - 1 if K > 1 else 1).bit_length())


def radix_passes(bits: int) -> int:
    return 1 if bits < 1 else (bits + 7) // 8


def expected_paths(case: Case, inp: Optional[Dict] = None, n_out: Optional[int] = None, padded: bool = False):
    """What the library runs for the case: a dict of rule -> path.  ``inp`` / ``n_out`` (the coarse edge count) are
    needed for the data-dependent rules (hub rows, long runs, the unfilter, the spine); without them those read
    None."""
    p: Dict[str, Optional[str]] = {"branch": case.branch}
    E = case.E if inp is None else inp["edge_index"].size(1)
    if case.branch == "kept":
        state_words = -(-max(E, 1) // 2048) + 2
        small = case.N <= SMALL_LIMIT and case.K <= SMALL_LIMIT and state_words <= SMALL_STATE_WORDS
        p["kept_fwd"] = "small" if small else "onepass"
        if n_out is not None and case.weighted:
            p["kept_bwd"] = "unfilter_small" if E <= SMALL_LIMIT and n_out <= SMALL_LIMIT else "unfilter"
    else:
        bucketed = case.sorted_rows and E + case.N < 2 ** 31 - 1
        p["cluster"] = "bucketed" if bucketed else "remap"
        cb = _cb(case.K)
        if bucketed:
            p["bucket_key"] = "packed" if case.K < PACKED_K else "unpacked"
            p["launch"] = "exact" if (E >= PLAN_SYNC_MIN_EDGES and not padded) else "capacity"
            if inp is not None:
                hub, long_run = _hub_stats(case, inp)
                p["hub"] = "hub" if hub else "tiles"
                p["long_run"] = "long" if long_run else "short"
        else:
            p["key"] = "u32" if 2 * cb <= 32 else "u64"
            p["passes"] = "odd" if radix_passes(2 * cb) % 2 else "even"
        if case.weighted:
            if case.op in ("sum", "mean"):
                p["coalesce_bwd"] = "bwd4_tail" if E % 4 else "bwd4"
            else:
                p["coalesce_bwd"] = "scalar"
            if case.op == "mul":
                p["mul_grad"] = "run_aux" if bucketed else "quotient"
    if case.dn and case.weighted:
        p["deg_bwd"] = "prepare"  # coarse rows are sorted on both branches of these cases
    if (case.dn or (case.ewn and case.weighted)) and n_out is not None:
        p["spine"] = "several" if -(-n_out // DS_TILE) > SPINE_ROUND else "one"
    return p


def _hub_stats(case: Case, inp: Dict):
    """(a coarse row has more than 512 virtual entries, a hub run has more than 4096 members)."""
    row, col = inp["edge_index"]
    cl = inp["cluster"]
    deg = torch.bincount(row, minlength=case.N)
    cost = deg.clamp(min=1)
    per_row = torch.zeros(case.K, dtype=torch.long).index_add_(0, cl, cost)
    hub_rows = per_row > HUB_ENTRIES
    hub = bool(hub_rows.any())
    key = cl[row] * case.K + cl[col]
    in_hub = hub_rows[cl[row]]
    _, counts = torch.unique(key[in_hub], return_counts=True)
    long_run = bool((counts > LONG_RUN).any()) if counts.numel() else False
    return hub, long_run


# --------------------------------------------------------------------------- #
# oracle
# --------------------------------------------------------------------------- #
def _so(case: Case, inp: Dict):
    from oracle import ref_path as R

    if case.branch == "kept":
        node = inp["node_index"]
        return R.OracleSelectOutput(node_index=node, num_nodes=case.N, cluster_index=torch.arange(node.numel()),
                                    num_supernodes=node.numel())
    return R.OracleSelectOutput(cluster_index=inp["cluster"], num_nodes=case.N, num_supernodes=case.K)


def reference(case: Case, inp: Dict, dtype=torch.float32, w: Optional[Tensor] = None):
    """``R.sparse_connect_so`` in ``dtype`` (the weight may be given, e.g. as a leaf that requires grad)."""
    from oracle import ref_path as R

    if w is None and inp["w"] is not None:
        w = inp["w"].to(dtype)
    return R.sparse_connect_so(inp["edge_index"], _so(case, inp), edge_weight=w,
                               batch_pooled=inp["batch_pooled"] if case.ewn else None, remove_self_loops=case.rsl,
                               reduce_op=case.op, degree_norm=case.dn, edge_weight_norm=case.ewn)


def _membership(case: Case, inp: Dict, ei_out: Tensor):
    """Per input edge: the output edge it went into (-1 if none)."""
    row, col = inp["edge_index"]
    if case.branch == "kept":
        node = inp["node_index"]
        table = torch.full((case.N,), -1, dtype=torch.long)
        table[node] = torch.arange(node.numel())
        r, c = table[row], table[col]
        keep = (r >= 0) & (c >= 0)
        if case.rsl:
            keep &= r != c
        if inp["w"] is not None:
            keep &= inp["w"].abs() > EPS
        slot = torch.full((row.numel(),), -1, dtype=torch.long)
        slot[keep] = torch.arange(int(keep.sum()))
        assert int(keep.sum()) == ei_out.size(1)
        return slot
    cl = inp["cluster"]
    K = case.K
    key = cl[row] * K + cl[col]
    okey = ei_out[0] * K + ei_out[1]
    pos = torch.searchsorted(okey, key).clamp(max=max(okey.numel() - 1, 0))
    hit = okey[pos] == key if okey.numel() else torch.zeros_like(key, dtype=torch.bool)
    return torch.where(hit, pos, torch.full_like(pos, -1))


def decision32(case: Case, inp: Dict):
    """The float32 values the kernels decide on: coalesced weights (sequential float32 combine, float32 of the exact
    sum for hub runs of more than 4096 members), the degree-normalised weights as ``k_deg_apply`` rounds them, and
    the first position of each graph's maximum of |w| among them."""
    from oracle import ref_path as R

    ei32, w32 = R.sparse_connect_so(inp["edge_index"], _so(case, inp), edge_weight=inp["w"],
                                    remove_self_loops=case.rsl, reduce_op=case.op)
    if w32 is None:
        w32 = torch.ones(ei32.size(1))
    if case.branch == "cluster" and case.op in ("sum", "mean") and inp["w"] is not None:
        slot = _membership(case, inp, ei32)
        ok = slot >= 0
        cnt = torch.bincount(slot[ok], minlength=ei32.size(1))
        if bool((cnt > LONG_RUN).any()):  # whole-block runs: double partials, one rounding
            s64 = torch.zeros(ei32.size(1), dtype=torch.float64).index_add_(0, slot[ok], inp["w"].double()[ok])
            if case.op == "mean":
                s64f = (s64.float() / cnt.clamp(min=1).float())
            else:
                s64f = s64.float()
            w32 = torch.where(cnt > LONG_RUN, s64f, w32)
    wd = w32
    if case.dn:
        deg = torch.zeros(case.K if case.branch == "cluster" else inp["node_index"].numel(),
                          dtype=torch.float64).index_add_(0, ei32[0], w32.double()).float()
        dinv = 1.0 / torch.sqrt(deg.clamp(min=EPS))
        wd = (w32 * dinv[ei32[0]]) * dinv[ei32[1]]
    arg = None
    if case.ewn and inp["w"] is not None:
        eb = inp["batch_pooled"][ei32[0]]
        mx = torch.zeros(case.G).scatter_reduce_(0, eb, wd.abs(), "amax", include_self=True)
        n = wd.numel()
        cand = torch.where(wd.abs() == mx[eb], torch.arange(n), torch.full((n,), n))
        arg = torch.full((case.G,), n).scatter_reduce_(0, eb, cand, "amin", include_self=True)
    return ei32, w32, wd, arg


def oracle(case: Case, inp: Dict) -> Dict[str, Tensor]:
    """Float64 forward and weight gradient of the whole ``sparse_connect`` with the sums of |terms|.

    Keys: ``edge_index``, ``w`` (output weights, None unweighted), ``w_terms``, ``w32`` (the float32 coalesced weights
    the kernels produce for max / min, None otherwise), ``run_len`` (members of every output edge), ``dw``,
    ``dw_terms`` (None unweighted), ``g`` (the cotangent of the output weights)."""
    from oracle import ref_path as R

    ei32, w32, wd32, arg = decision32(case, inp)
    row, col = inp["edge_index"]
    w_in = inp["w"]
    n_out = ei32.size(1)
    res = {"edge_index": ei32, "w": None, "w_terms": None, "dw": None, "dw_terms": None,
           "w32": w32 if case.op in ("max", "min") else None}
    slot = _membership(case, inp, ei32)
    ok = slot >= 0
    run_len = torch.bincount(slot[ok], minlength=n_out)
    res["run_len"] = run_len
    if w_in is None and not case.dn:
        return res
    g = cotangent(case, n_out).double()
    res["g"] = g
    # ---- forward in float64 through the reference (coalesce / filter, self loops, tiny weights, degree norm)
    w64 = None if w_in is None else w_in.double().requires_grad_(True)
    ei64, wdn = R.sparse_connect_so(inp["edge_index"], _so(case, inp), edge_weight=w64, remove_self_loops=case.rsl,
                                    reduce_op=case.op, degree_norm=case.dn)
    assert torch.equal(ei64, ei32), "float64 and float32 runs of the reference keep different edges"
    # ---- |terms| of the coalesced weights
    if w_in is None:
        wc = torch.ones(n_out, dtype=torch.float64)
        ac = wc.clone()
    else:
        wa = w_in.double().abs()
        if case.branch == "kept" or case.op in ("max", "min"):
            with torch.no_grad():
                ac = torch.zeros(n_out, dtype=torch.float64).index_add_(0, slot[ok], wa[ok]) / run_len.clamp(min=1)
                if case.op in ("max", "min") and case.branch == "cluster":
                    ac = w32.double().abs()
        elif case.op == "mul":
            ac = torch.ones(n_out, dtype=torch.float64).index_reduce_(0, slot[ok], wa[ok], "prod")
        else:
            ac = torch.zeros(n_out, dtype=torch.float64).index_add_(0, slot[ok], wa[ok])
            if case.op == "mean":
                ac = ac / run_len.clamp(min=1)
        wc = None
    wout = wdn
    aout = ac
    K = case.K if case.branch == "cluster" else inp["node_index"].numel()
    r_o, c_o = ei32[0], ei32[1]
    if case.dn:
        with torch.no_grad():
            wcv = torch.ones(n_out, dtype=torch.float64) if w_in is None else _coalesced64(case, inp, slot, run_len)
            _, dinv, cd = _degree_terms(case, r_o, wcv, ac, K)
            # y = wc d_r d_c: terms |y| (A_c / |wc| + c_r + c_c)
            aout = dinv[r_o] * dinv[c_o] * (ac + wcv.abs() * (cd[r_o] + cd[c_o]))
    if case.ewn and w_in is not None:
        eb = inp["batch_pooled"][r_o]
        n = n_out
        arg_c = arg.clamp(max=max(n - 1, 0))
        has = arg < n
        m = torch.where(has, wout[arg_c].abs(), torch.ones(case.G, dtype=torch.float64))
        m = torch.where(m == 0, torch.ones_like(m), m)
        wfin = wout / m[eb]
        with torch.no_grad():
            m_d = m.detach()
            cm = _max_condition(has, aout, arg_c, m_d)
            # z = y / m: terms |z| (1 + c_y + c_m) = (terms(y) + |y| c_m) / m
            a_fin = (aout + wout.detach().abs() * cm[eb]) / m_d[eb]
    else:
        wfin, a_fin = wout, aout
    res["w"] = wfin.detach()
    res["w_terms"] = a_fin
    if w_in is None:
        return res
    (wfin * g).sum().backward()
    res["dw"] = w64.grad.detach().clone()
    res["dw_terms"] = _grad_terms(case, inp, slot, run_len, ac, g, aout, (m.detach() if case.ewn else None), arg,
                                  K, w32)
    return res


def _coalesced64(case: Case, inp: Dict, slot: Tensor, run_len: Tensor) -> Tensor:
    """Coalesced weights in float64 (what enters the degree)."""
    ok = slot >= 0
    n_out = run_len.numel()
    w = inp["w"].double()
    if case.branch == "kept":
        return torch.zeros(n_out, dtype=torch.float64).index_add_(0, slot[ok], w[ok])
    if case.op in ("sum", "mean"):
        s = torch.zeros(n_out, dtype=torch.float64).index_add_(0, slot[ok], w[ok])
        return s / run_len.clamp(min=1) if case.op == "mean" else s
    if case.op == "mul":
        return torch.ones(n_out, dtype=torch.float64).index_reduce_(0, slot[ok], w[ok], "prod")
    red = "amax" if case.op == "max" else "amin"
    return torch.zeros(n_out, dtype=torch.float64).index_reduce_(0, slot[ok], w[ok], red, include_self=False)


def _degree_terms(case: Case, rows: Tensor, wc: Tensor, ac: Tensor, K: int):
    """(deg, dinv, c) per pooled node: c = kappa / 2 with kappa = sum of the row's terms / |deg|, the condition of
    dinv = deg^(-1/2) (0 where the EPS clamp makes dinv a constant)."""
    deg = torch.zeros(K, dtype=torch.float64).index_add_(0, rows, wc)
    dterms = torch.zeros(K, dtype=torch.float64).index_add_(0, rows, ac)
    live = deg >= EPS
    cd = torch.where(live, 0.5 * dterms / deg.abs().clamp(min=EPS), torch.zeros_like(deg))
    return deg, deg.clamp(min=EPS).pow(-0.5), cd


def _max_condition(has: Tensor, terms: Tensor, arg: Tensor, m: Tensor) -> Tensor:
    """Condition c_m of each graph's maximum m = |y_arg|: terms(y_arg) / m - 1 (0 for a graph without edges)."""
    return torch.where(has, terms[arg] / m - 1.0, torch.zeros_like(m))


def _grad_terms(case, inp, slot, run_len, ac, g, adn, m, arg, K, w32) -> Tensor:
    """Sum of |terms| of the weight gradient: the backward of every stage with absolute values, each factor that the
    forward derives carrying its condition (module docstring)."""
    n_out = run_len.numel()
    ga = g.abs()
    # max-weight normalisation backward: g / m, and acc / m^2 at the first maximum of each graph
    if m is not None:
        eb = inp["batch_pooled"][_out_rows(case, inp, slot, n_out)]
        valid = arg < n_out
        cm = _max_condition(valid, adn, arg.clamp(max=max(n_out - 1, 0)), m)
        acc_t = torch.zeros(case.G, dtype=torch.float64).index_add_(0, eb, ga * adn)  # acc = sum g y
        ga = ga * (1 + cm[eb]) / m[eb]
        hit = torch.zeros(n_out, dtype=torch.bool)
        hit[arg[valid]] = True
        ga = ga + torch.where(hit, acc_t[eb] * (1 + 2 * cm[eb]) / (m[eb] * m[eb]), torch.zeros_like(ga))
    # degree normalisation backward: g d_r d_c, and -0.5 gdinv_r d_r^3 with gdinv_v = sum g wc d_other
    if case.dn:
        r_o = _out_rows(case, inp, slot, n_out)
        c_o = _out_cols(case, inp, slot, n_out)
        wcv = ac if inp["w"] is None else _coalesced64(case, inp, slot, run_len)
        deg, d, cd = _degree_terms(case, r_o, wcv, ac, K)
        gd = (torch.zeros(K, dtype=torch.float64).index_add_(0, r_o, ga * ac * d[c_o] * (1 + cd[c_o]))
              .index_add_(0, c_o, ga * ac * d[r_o] * (1 + cd[r_o])))
        gdeg = torch.where(deg >= EPS, 0.5 * gd * d ** 3 * (1 + 3 * cd), torch.zeros_like(gd))
        ga = ga * d[r_o] * d[c_o] * (1 + cd[r_o] + cd[c_o]) + gdeg[r_o]
    # coalesce / filter backward
    ok = slot >= 0
    w = inp["w"].double()
    out = torch.zeros(w.numel(), dtype=torch.float64)
    s = slot[ok]
    if case.branch == "kept" or case.op == "sum":
        out[ok] = ga[s]
    elif case.op == "mean":
        out[ok] = ga[s] / run_len[s]
    elif case.op in ("max", "min"):
        hit = w.float()[ok] == w32[s]
        ties = torch.zeros(n_out, dtype=torch.float64).index_add_(0, s, hit.double())
        out[ok] = torch.where(hit, ga[s] / ties[s].clamp(min=1), torch.zeros_like(ga[s]))
    else:  # mul: g times the product of the other members (|prod| / |w| when w != 0)
        wa = w.abs()[ok]
        out[ok] = torch.where(wa > 0, ga[s] * ac[s] / wa.clamp(min=1e-300), torch.zeros_like(ga[s]))
    return out


def _out_rows(case, inp, slot, n_out):
    return _out_ends(case, inp, slot, n_out, 0)


def _out_cols(case, inp, slot, n_out):
    return _out_ends(case, inp, slot, n_out, 1)


def _out_ends(case, inp, slot, n_out, k):
    ok = slot >= 0
    end = inp["edge_index"][k]
    lab = (torch.searchsorted(inp["node_index"], end) if case.branch == "kept" else inp["cluster"][end])
    out = torch.zeros(n_out, dtype=torch.long)
    out[slot[ok]] = lab[ok]
    return out


# --------------------------------------------------------------------------- #
# the summation of the deterministic segment sums, emulated in float64
# --------------------------------------------------------------------------- #
def prefix_difference_sums(keys: Tensor, vals: Tensor, K: int) -> Tensor:
    """Each segment's sum as the difference of two values of one running float64 prefix sum over all positions (the
    form that makes a segment's error scale with everything sorted before it)."""
    pre = torch.cumsum(torch.cat([torch.zeros(1, dtype=torch.float64), vals.double()]), 0)
    out = torch.zeros(K, dtype=torch.float64)
    n = keys.numel()
    first = torch.ones(n, dtype=torch.bool)
    first[1:] = keys[1:] != keys[:-1]
    last = torch.ones(n, dtype=torch.bool)
    last[:-1] = keys[1:] != keys[:-1]
    out[keys[last]] = pre[1:][last] - pre[:-1][first]
    return out


def segmented_sums(keys: Tensor, vals: Tensor, K: int) -> Tensor:
    """Each segment summed on its own in float64 (the segmented scan)."""
    return torch.zeros(K, dtype=torch.float64).index_add_(0, keys, vals.double())
