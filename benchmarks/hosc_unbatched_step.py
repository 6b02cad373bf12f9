"""HOSC pooling on a sparse adjacency (``unbatched.hosc_pool_unbatched``) against the batched dense ``hosc_pool``.

One forward + backward step (alpha = 0.5, MinCut's orthogonality term, upstream gradients on x_pool, adj_pool and
both losses; S, x and the edge weights requiring grad) per workload, eager (the sparse path reads the coalesced edge
count back once per call, so it is not captured as a CUDA graph; the dense arm runs eager too).  Two arms alternate
over timed windows of at least 100 ms each, after a warm-up; the median window is reported.

* a: ragged batch at the C2 shape, B = 512 graphs of N <= 256 nodes, K = 64, F = 128, density 0.1: sparse against
  dense on ``to_dense_adj`` of the same graphs;
* b: one graph, N = 16 384, E ~ 540 k (uniform, symmetric): dense against sparse;
* c: the C4 graph, N = 1 M, E = 20 M power-law (``bench.powerlaw_graph``), K = 64, F = 128: the sparse step, the
  motif pass alone (the forward ``k_hosc_isect_*`` launches), a per-kernel table of one step, and the intersection
  work -- sum over the coalesced edges of the shorter list each one walks -- with its rate.

Each workload prints one JSON line with the card name and power limit.

    python benchmarks/hosc_unbatched_step.py [--workload {a,b,c,all}] [--windows W] [--out FILE]
"""
import argparse
import json
import os
import subprocess
import sys

sys.path.insert(0, os.getcwd())
sys.path.insert(0, os.path.join(os.getcwd(), "torch-geometric-pool_b200"))
import torch

import bench
import tgp_b200 as T
from tgp_b200 import _lib as L
from tgp_b200 import functional as F_
from tgp_b200 import unbatched as U

K, F = 64, 128
MU, ALPHA = 0.1, 0.5
FLAGS = dict(remove_self_loops=True, degree_norm=True, edge_weight_norm=False)


def _power_limit():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
        return out or "unknown"
    except (OSError, subprocess.SubprocessError):
        return "unknown"


def _symmetric(rows, cols, n_total, seed):
    g = torch.Generator(device="cuda").manual_seed(seed)
    w = torch.rand(rows.numel(), device="cuda", generator=g) + 0.5
    return torch.stack([torch.cat([rows, cols]), torch.cat([cols, rows])]), torch.cat([w, w])


def _ragged_batch(B, nmax, density, seed):
    g = torch.Generator(device="cuda").manual_seed(seed)
    sizes = torch.tensor([nmax - (7 * b) % (nmax // 3) for b in range(B)], device="cuda")
    ptr = torch.cat([torch.zeros(1, dtype=torch.long, device="cuda"), torch.cumsum(sizes, 0)])
    batch = torch.repeat_interleave(torch.arange(B, device="cuda"), sizes)
    pairs = (sizes * (sizes - 1) // 2 * density).long()  # expected undirected edges per graph
    gb = torch.repeat_interleave(torch.arange(B, device="cuda"), pairs)
    n = sizes[gb]
    r = (torch.rand(gb.numel(), device="cuda", generator=g) * n).long() + ptr[gb]
    c = (torch.rand(gb.numel(), device="cuda", generator=g) * n).long() + ptr[gb]
    keep = r != c
    ei, w = _symmetric(r[keep], c[keep], int(ptr[-1]), seed)
    return ei, w, batch, B


def _inputs(n, ei, w, batch, B, nmax, seed):
    g = torch.Generator(device="cuda").manual_seed(seed)
    s = torch.softmax(torch.randn(n, K, device="cuda", generator=g), -1).requires_grad_(True)
    x = torch.randn(n, F, device="cuda", generator=g).requires_grad_(True)
    w = w.clone().requires_grad_(True)
    gx = torch.randn(B, K, F, device="cuda", generator=g)
    ga = torch.randn(B, K, K, device="cuda", generator=g)
    return s, x, w, gx, ga


def _run_step(fn, leaves, gx, ga):
    one = torch.ones((), device="cuda")

    def run():
        for t in leaves:
            t.grad = None
        xp, ap, loss = fn()
        torch.autograd.backward([xp, ap, loss["hosc_loss"], loss["ortho_loss"]], [gx, ga, one, one])

    return run


def _window(run, reps):
    start, stop = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    start.record()
    for _ in range(reps):
        run()
    stop.record()
    stop.synchronize()
    return start.elapsed_time(stop) / reps


def _alternate(arms, windows):
    reps = {}
    for key, run in arms.items():  # warm-up, then size each window to at least 100 ms
        _window(run, 3)
        reps[key] = max(3, int(100.0 / _window(run, 3)) + 1)
    times = {key: [] for key in arms}
    for _ in range(windows):
        for key, run in arms.items():
            times[key].append(_window(run, reps[key]))
    med = {key: sorted(v)[len(v) // 2] for key, v in times.items()}
    return med, times, reps


def _sparse_arm(ei, w, s, x, batch, B, gx, ga):
    return _run_step(lambda: U.hosc_pool_unbatched(x, ei, w, s, batch, B, MU, ALPHA, False, **FLAGS), (s, x, w), gx, ga)


def _dense_arm(ei, w, s, x, batch, B, nmax, gx, ga):
    """hosc_pool on to_dense_adj / to_dense_batch of the same graphs (built once, outside the step)."""
    adj = F_.to_dense_adj(ei, batch, w.detach(), B, nmax).requires_grad_(True)
    s3 = F_.to_dense_batch(s.detach(), batch, B, nmax)[0].contiguous().requires_grad_(True)
    x3 = F_.to_dense_batch(x.detach(), batch, B, nmax)[0].contiguous().requires_grad_(True)
    mask = F_.to_dense_batch(s.detach(), batch, B, nmax)[1]
    fn = lambda: T.hosc_pool(x3, adj, s3, mask, MU, ALPHA, False, adj_transpose=False, **FLAGS)  # noqa: E731
    return _run_step(fn, (s3, x3, adj), gx, ga)


def _outputs_agree(ei, w, s, x, batch, B, nmax):
    """max relative difference of (x_pool, adj_pool, hosc_loss) between the two paths on these inputs."""
    xs, as_, ls = U.hosc_pool_unbatched(x, ei, w, s, batch, B, MU, ALPHA, False, **FLAGS)
    adj = F_.to_dense_adj(ei, batch, w.detach(), B, nmax)
    s3, mask = F_.to_dense_batch(s.detach(), batch, B, nmax)
    x3 = F_.to_dense_batch(x.detach(), batch, B, nmax)[0]
    xd, ad, ld = T.hosc_pool(x3, adj, s3, mask, MU, ALPHA, False, adj_transpose=False, **FLAGS)
    rel = lambda a, b: float((a - b).detach().abs().max() / b.detach().abs().max().clamp(min=1e-30))  # noqa: E731
    return {"x_pool": rel(xs, xd), "adj_pool": rel(as_, ad), "hosc_loss": rel(ls["hosc_loss"], ld["hosc_loss"])}


def workload_a(windows):
    B, nmax = 512, 256
    ei, w, batch, B = _ragged_batch(B, nmax, 0.1, seed=1)
    n = batch.numel()
    s, x, w, gx, ga = _inputs(n, ei, w, batch, B, nmax, seed=2)
    arms = {"sparse": _sparse_arm(ei, w, s, x, batch, B, gx, ga),
            "dense": _dense_arm(ei, w, s, x, batch, B, nmax, gx, ga)}
    med, times, reps = _alternate(arms, windows)
    return {"workload": "a", "shape": {"B": B, "Nmax": nmax, "nodes": n, "edges": ei.size(1), "K": K, "F": F},
            "sparse_ms": med["sparse"], "dense_ms": med["dense"], "sparse_over_dense": med["sparse"] / med["dense"],
            "rel_diff": _outputs_agree(ei, w, s, x, batch, B, nmax), "ms_all": times, "reps_per_window": reps}


def workload_b(windows):
    n, pairs = 16384, 270_000
    g = torch.Generator(device="cuda").manual_seed(3)
    r = torch.randint(0, n, (pairs,), device="cuda", generator=g)
    c = torch.randint(0, n, (pairs,), device="cuda", generator=g)
    keep = r != c
    ei, w = _symmetric(r[keep], c[keep], n, 3)
    batch = torch.zeros(n, dtype=torch.long, device="cuda")
    s, x, w, gx, ga = _inputs(n, ei, w, batch, 1, n, seed=4)
    arms = {"dense": _dense_arm(ei, w, s, x, batch, 1, n, gx, ga), "sparse": _sparse_arm(ei, w, s, x, batch, 1, gx, ga)}
    med, times, reps = _alternate(arms, windows)
    return {"workload": "b", "shape": {"N": n, "edges": ei.size(1), "K": K, "F": F}, "sparse_ms": med["sparse"],
            "dense_ms": med["dense"], "dense_over_sparse": med["dense"] / med["sparse"],
            "rel_diff": _outputs_agree(ei, w, s, x, batch, 1, n), "ms_all": times, "reps_per_window": reps}


def workload_c(windows):
    n, e = 1 << 20, 20_000_000
    ei = bench.powerlaw_graph(n, e, "cuda", seed=5)
    g = torch.Generator(device="cuda").manual_seed(6)
    w = torch.rand(ei.size(1), device="cuda", generator=g) + 0.5
    batch = torch.zeros(n, dtype=torch.long, device="cuda")
    s, x, w, gx, ga = _inputs(n, ei, w, batch, 1, n, seed=7)
    run = _sparse_arm(ei, w, s, x, batch, 1, gx, ga)
    med, times, reps = _alternate({"sparse": run}, windows)
    torch.cuda.synchronize()
    L.time_kernel("*")  # one traced step: every launch of the library with its CUDA-event time
    run()
    torch.cuda.synchronize()
    trace = L.kernel_trace()
    L.time_kernel(None)
    table = {}
    for name, ms in trace:
        t = table.setdefault(name, [0.0, 0])
        t[0] += ms
        t[1] += 1
    fwd_isect = [ms for name, ms in trace if "k_hosc_isect" in name][:2]  # the forward's warp + heavy launches
    # intersection work of the forward: per coalesced edge, the length of the shorter of out(i) and in(j)
    ei_c = torch.unique(ei[0] * n + ei[1])
    row, col = ei_c // n, ei_c % n
    deg_out = torch.bincount(row, minlength=n)
    deg_in = torch.bincount(col, minlength=n)
    walk = torch.minimum(deg_out[row], deg_in[col])
    work = int(walk.sum())
    heavy = int((walk > 1024).sum())
    motif_ms = sum(fwd_isect)
    return {"workload": "c", "shape": {"N": n, "edges": ei.size(1), "coalesced_edges": int(ei_c.numel()), "K": K,
                                       "F": F},
            "step_ms": med["sparse"], "motif_pass_ms": motif_ms, "motif_pass_launches_ms": fwd_isect,
            "intersection_work_entries": work, "heavy_edges": heavy,
            "intersection_rate_entries_per_s": work / (motif_ms * 1e-3) if motif_ms > 0 else None,
            "kernels_ms_and_launches": {k: [round(v[0], 4), v[1]] for k, v in sorted(table.items(), key=lambda kv: -kv[1][0])},
            "ms_all": times["sparse"], "reps_per_window": reps}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--workload", choices=["a", "b", "c", "all"], default="all")
    ap.add_argument("--windows", type=int, default=7)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    head = {"device": torch.cuda.get_device_name(0), "power_limit": _power_limit()}
    lines = []
    for name, fn in (("a", workload_a), ("b", workload_b), ("c", workload_c)):
        if args.workload not in (name, "all"):
            continue
        lines.append(json.dumps({**head, **fn(args.windows)}))
        print(lines[-1], flush=True)
        torch.cuda.empty_cache()
    if args.out:
        with open(args.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
