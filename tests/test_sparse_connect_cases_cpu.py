"""CPU checks of the sparse-connect case table (``sparse_connect_cases``): every launch path is reached by some case,
the thresholds are met on both sides, the float64 oracle reproduces the reference's own float32 connect and autograd,
and the dynamic-range cases are not vacuous.  ``pytest -rP`` prints which cases reach each path."""
import functools

import pytest
import torch

import sparse_connect_cases as S


@functools.lru_cache(maxsize=None)
def _paths():
    out = {}
    for c in S.CASES:
        inp = S.inputs(c) if c.branch == "cluster" and c.sorted_rows else None
        out[c] = S.expected_paths(c, inp)
    return out


def _combos():
    combos = [("branch", "kept"), ("branch", "cluster"), ("kept_fwd", "small"), ("kept_fwd", "onepass"),
              ("deg_bwd", "prepare")]
    for op in S.OPS:
        for path in ("bucketed", "remap"):
            combos.append(("cluster", path, op))
    for key in ("u32", "u64"):
        for par in ("odd", "even"):
            combos.append(("key+passes", key, par))
    combos += [("bucket_key", "packed"), ("bucket_key", "unpacked"), ("hub", "hub"), ("hub", "tiles"),
               ("long_run", "long"), ("launch", "exact"), ("launch", "capacity"), ("mul_grad", "run_aux"),
               ("mul_grad", "quotient"), ("coalesce_bwd", "bwd4"), ("coalesce_bwd", "bwd4_tail"),
               ("coalesce_bwd", "scalar")]
    for br in ("kept", "cluster"):
        for norm in ("dn", "ewn"):
            combos.append(("norm", br, norm))
    return combos


def _reaching(combo):
    out = []
    for c, p in _paths().items():
        if combo[0] == "cluster":
            hit = p.get("cluster") == combo[1] and c.op == combo[2] and c.weighted
        elif combo[0] == "key+passes":
            hit = p.get("key") == combo[1] and p.get("passes") == combo[2]
        elif combo[0] == "norm":
            hit = c.branch == combo[1] and (c.dn if combo[2] == "dn" else (c.ewn and c.weighted))
        else:
            hit = p.get(combo[0]) == combo[1]
        if hit:
            out.append(c)
    return out


@pytest.mark.parametrize("combo", _combos(), ids=["-".join(c) for c in _combos()])
def test_launch_path_reached(combo):
    cases = _reaching(combo)
    print(f"{combo}: " + ", ".join(c.id for c in cases))
    assert cases, f"no case runs {combo}"


def test_thresholds_on_both_sides():
    Ks = {c.K for c in S.CASES if c.branch == "cluster"}
    for K in (2, 256, 257, 65536, 65537, S.PACKED_K - 1, S.PACKED_K + 1):
        assert K in Ks, K
    assert {c.E % 4 for c in S.CASES if c.branch == "cluster" and c.E} >= {0, 1, 3}
    for op in S.OPS:
        for w in ("none", "tri", "zeros", "unit"):
            assert any(c.op == op and c.values == w for c in S.CASES if c.branch == "cluster"), (op, w)
        assert any(c.op == op and c.rsl for c in S.CASES) and any(c.op == op and not c.rsl for c in S.CASES)
    kept = [c for c in S.CASES if c.branch == "kept"]
    assert any(c.N == S.SMALL_LIMIT for c in kept) and any(c.N == S.SMALL_LIMIT + 1 for c in kept)
    for v in ("tri", "unit", "signed", "dyn", "none"):
        assert any(c.values == v for c in kept), v
    assert any(c.values == "dyn" for c in S.CASES if c.branch == "cluster")


def test_spine_takes_several_rounds():
    """The largest normalised cases have more than 1024 tiles of 2048 edges, with a coarse row that straddles the
    boundary between the first two spine rounds (the carry between rounds matters)."""
    for c in S.CASES:
        if c.E < 3_000_000:
            continue
        inp = S.inputs(c)
        ei32, _, _, _ = S.decision32(c, inp)
        n = ei32.size(1)
        assert S.expected_paths(c, inp, n)["spine"] == "several", c.id
        b = S.SPINE_ROUND * S.DS_TILE
        assert n > b and int(ei32[0, b - 1]) == int(ei32[0, b]), f"{c.id}: no row straddles the spine round boundary"


def test_tile_aligned_segments():
    c = next(c for c in S.CASES if c.graph == "tiles")
    row = S.inputs(c)["edge_index"][0]
    starts = torch.nonzero(torch.cat([torch.ones(1, dtype=torch.bool), row[1:] != row[:-1]])).flatten()
    ends = torch.cat([starts[1:], torch.tensor([row.numel()])])
    assert bool((starts % S.DS_TILE == 0).sum() >= 3) and bool((ends % S.DS_TILE == 0).sum() >= 3)
    assert bool(((starts % 256 == 0) & (starts % S.DS_TILE != 0)).sum() >= 3)
    long = (ends - starts) > S.DS_TILE
    assert bool(long.any()), "a run longer than a tile"


def _small_cases():
    out = []
    for op in S.OPS:
        for srt in (True, False):
            out.append(S.Case("cluster", 300, 70, 2001, "rand", "tri", op, sorted_rows=srt))
            out.append(S.Case("cluster", 300, 70, 2003, "rand", "rand", op, rsl=False, dn=True, ewn=True,
                              sorted_rows=srt))
        out.append(S.Case("cluster", 300, 70, 2000, "rand", "zeros", op))
        out.append(S.Case("cluster", 300, 70, 2000, "rand", "unit", op, ewn=True))
    out.append(S.Case("cluster", 300, 70, 2001, "rand", "none", "sum", dn=True))
    out.append(S.Case("cluster", 300, 70, 2001, "rand", "signed", "max", dn=True, ewn=True))
    out.append(S.Case("kept", 300, 170, 2001, "rand", "tri", dn=True, ewn=True))
    out.append(S.Case("kept", 300, 170, 2001, "rand", "unit", rsl=False, dn=True, ewn=True))
    out.append(S.Case("kept", 300, 170, 2001, "rand", "signed", dn=True, ewn=True))
    return out


@pytest.mark.parametrize("case", _small_cases(), ids=[c.id for c in _small_cases()])
def test_oracle_matches_reference_fp32(case):
    """The oracle against ``R.sparse_connect_so`` and its autograd at float32: indices and order bit-exact, weights
    and the weight gradient to rtol 1e-6 (the terms bound every difference)."""
    inp = S.inputs(case)
    ref = S.oracle(case, inp)
    w = None if inp["w"] is None else inp["w"].clone().requires_grad_(True)
    ei, wo = S.reference(case, inp, torch.float32, w)
    assert torch.equal(ei, ref["edge_index"])
    if wo is None:
        assert ref["w"] is None
        return
    assert bool((ref["w_terms"] >= ref["w"].abs() * (1 - 1e-12)).all())
    err = (wo.detach().double() - ref["w"]).abs()
    assert bool((err <= 1e-6 * ref["w_terms"] + 1e-30).all()), float((err / ref["w_terms"]).max())
    if case.op in ("max", "min") and case.branch == "cluster" and not (case.dn or case.ewn):
        assert torch.equal(wo.detach(), ref["w32"])
    if w is None:
        return
    (wo * ref["g"].float()).sum().backward()
    gerr = (w.grad.double() - ref["dw"]).abs()
    assert bool((ref["dw_terms"] >= ref["dw"].abs() * (1 - 1e-9) - 1e-300).all())
    assert bool((gerr <= 1e-6 * ref["dw_terms"] + 1e-30).all()), float((gerr / (ref["dw_terms"] + 1e-30)).max())


def test_oracle_holds_ties_and_clamps():
    """The tie regimes tie: max / min coalesce runs with several members at the extreme, graphs whose maximum |w| is
    shared; the signed kept-node case has a degree of exactly 0 and one below EPS."""
    c = next(c for c in S.CASES if c.branch == "cluster" and c.values == "tri" and c.op == "max" and c.K == 700)
    inp = S.inputs(c)
    ref = S.oracle(c, inp)
    slot = S._membership(c, inp, ref["edge_index"])
    ok = slot >= 0
    hit = inp["w"][ok] == ref["w32"][slot[ok]]
    ties = torch.bincount(slot[ok][hit], minlength=ref["edge_index"].size(1))
    assert int((ties > 1).sum()) > 10
    c = next(c for c in S.CASES if c.branch == "kept" and c.values == "signed" and c.graph == "rand")
    inp = S.inputs(c)
    ei, _, _, _ = S.decision32(c, inp)
    w64 = S._coalesced64(c, inp, S._membership(c, inp, ei), torch.ones(ei.size(1), dtype=torch.long))
    deg = torch.zeros(c.K, dtype=torch.float64).index_add_(0, ei[0], w64)
    assert bool((deg == 0).any() & ((deg > 0) & (deg < S.EPS)).any())


@pytest.mark.parametrize("branch", ["kept", "cluster"])
def test_dynamic_range_case_not_vacuous(branch):
    """The degrees of the dynamic-range case: a float64 prefix difference (each segment's sum as the difference of two
    running sums over everything before it) misses the 1e-5 bound on some light row; summing each segment on its own
    stays far inside it."""
    c = next(c for c in S.CASES if c.graph == "dyn" and c.branch == branch)
    inp = S.inputs(c)
    ei, w32, _, _ = S.decision32(c, inp)
    K = c.K
    keys, vals = ei[0], w32.double()
    exact = torch.zeros(K, dtype=torch.float64).index_add_(0, keys, vals)
    terms = torch.zeros(K, dtype=torch.float64).index_add_(0, keys, vals.abs())
    bound = 1e-5 * terms
    heavy = float(vals[: 100000].sum())
    assert heavy >= 9e8 and float(vals[-1000:].abs().max()) <= 1e-3
    pre = S.prefix_difference_sums(keys, vals, K)
    seg = S.segmented_sums(keys, vals, K)
    bad = (pre - exact).abs() > bound
    assert int(bad.sum()) > 100, "the prefix difference would pass: the case is vacuous"
    assert bool(((seg - exact).abs() <= 1e-12 * terms).all())
