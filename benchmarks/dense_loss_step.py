"""Cost of the dense poolers with losses of their own against MinCut at the C2 shape (B = 512, N = 256, K = 64,
F = 128).

For each pooler, its step and the MinCut step (forward + backward with MinCut's connector flags, only x and S
requiring grad) are each captured as one CUDA graph; the two graphs run in one process, alternating, over timed
windows of at least 100 ms each.

* dmon (fp32, adjacency density 0.05): the fused ``dense_pool`` call with loss_kind 3 (graph_nodes = N) against
  loss_kind 1, the losses vector taking upstream gradient (1, 1, 1, 0).
* acc (fp32 and bf16, density 0.05): ``acc_pool`` (the loss-free fused dense call plus the ``acc_losses`` kernels)
  against ``mincut_pool``.  Also the ``k_acc_*`` kernels alone, from CUDA events around each launch in eager forward +
  backward passes, and the eager torch restatement of the two losses (``tests/acc_oracle.py``: ``totvar_loss`` +
  ``asym_norm_loss``, forward + backward) on the same inputs: its time and its peak memory above the inputs.
* hosc (fp32 and bf16, density 0.1: more triangles): ``hosc_pool`` (alpha = 0.5, MinCut's orthogonality term: the
  fused dense call plus the ``hosc_losses`` products and kernels) against ``mincut_pool``.  Also every launch named
  *hosc* alone (the ``k_hosc_*`` kernels and ``k_tc_gemm:hosc:*`` products) with its launches per pass, and the eager
  restatement of the two cut losses (``tests/hosc_oracle.py``: ``cut_loss`` of A and of ``motif_adjacency(A)``).

Each pooler prints one JSON line, with the card name and power limit beside its numbers.

    python benchmarks/dense_loss_step.py --pooler {dmon,acc,hosc,all} [--windows W] [--eager-reps R] [--out FILE]
"""
import argparse
import json
import os
import subprocess
import sys

sys.path.insert(0, os.getcwd())
sys.path.insert(0, os.path.join(os.getcwd(), "torch-geometric-pool_b200"))
sys.path.insert(0, os.path.join(os.getcwd(), "tests"))
import torch

import acc_oracle as A
import hosc_oracle as O
import tgp_b200 as T
from tgp_b200 import _lib as L
from tgp_b200 import functional as F_

B, N, K, F = 512, 256, 64, 128
FLAGS = dict(remove_self_loops=True, degree_norm=True, adj_transpose=True)
DTYPES = {"fp32": torch.float32, "bf16": torch.bfloat16}
TRACE_PASSES = 20


def _power_limit():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
        return out or "unknown"
    except (OSError, subprocess.SubprocessError):
        return "unknown"


def _inputs(density, dtype):
    dev = "cuda"
    g = torch.Generator().manual_seed(0)
    a = (torch.rand(B, N, N, generator=g) < density).float()
    a = torch.triu(a, 1)
    a = (a + a.transpose(1, 2)).to(dev, dtype)
    x = torch.randn(B, N, F, generator=g).to(dev, dtype).requires_grad_(True)
    s = torch.softmax(torch.randn(B, N, K, generator=g), -1).to(dev, dtype).requires_grad_(True)
    gx = torch.randn(B, K, F, generator=g).to(dev, dtype)
    ga = torch.randn(B, K, K, generator=g).to(dev, dtype)
    return x, a, s, gx, ga


def _dmon_steps(x, a, s, gx, ga):
    """(MinCut step, DMoN step) through ``dense_pool`` and its losses vector."""
    gl = torch.tensor([1.0, 1.0, 1.0, 0.0], device=x.device)
    gn = torch.full((B,), float(N), device=x.device)

    def step(loss_kind, graph_nodes):
        def run():
            xp, ap, losses = F_.dense_pool(x, a, s, loss_kind=loss_kind, graph_nodes=graph_nodes, **FLAGS)
            torch.autograd.backward([xp, ap, losses], [gx, ga, gl])
            return xp, ap, losses

        return run

    return step(F_.LOSS_MINCUT, None), step(F_.LOSS_DMON, gn)


def _pool_steps(pool):
    """(MinCut step, ``pool`` step) through the ``*_pool`` functions, each loss of the dict with upstream gradient 1."""
    def steps(x, a, s, gx, ga):
        one = torch.ones((), device=x.device)

        def step(fn):
            def run():
                xp, ap, loss = fn(x, a, s)
                losses = list(loss.values())
                torch.autograd.backward([xp, ap, *losses], [gx, ga] + [one] * len(losses))
                return xp, ap, *losses

            return run

        return step(lambda x, a, s: T.mincut_pool(x, a, s, **FLAGS)), step(pool)

    return steps


def _graph(run, x, s):
    def step():
        x.grad = None
        s.grad = None
        return run()

    return T.GraphedStep(step)


def _window(graph, reps):
    start, stop = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    start.record()
    for _ in range(reps):
        graph.replay()
    stop.record()
    stop.synchronize()
    return start.elapsed_time(stop) / reps


def _trace(pattern, run, s):
    """{name: [ms of each launch]} of the launches whose name contains ``pattern`` over ``TRACE_PASSES`` eager passes
    of ``run(s)`` (forward + backward), after one untimed pass."""
    s = s.detach().requires_grad_(True)
    run(s)
    torch.cuda.synchronize()
    L.time_kernel(pattern)
    for _ in range(TRACE_PASSES):
        s.grad = None
        run(s)
    torch.cuda.synchronize()
    per = {}
    for name, ms in L.kernel_trace():
        per.setdefault(name, []).append(ms)
    L.time_kernel(None)
    return per


def _eager(loss, s, reps):
    """The restated torch ``loss(s)``, forward + backward: mean ms and the peak memory (GB) above the inputs."""
    s = s.detach().requires_grad_(True)

    def run():
        s.grad = None
        loss(s).backward()

    try:
        run()
        torch.cuda.synchronize()
        torch.cuda.reset_peak_memory_stats()
        base = torch.cuda.memory_allocated()
        start, stop = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        start.record()
        for _ in range(reps):
            run()
        stop.record()
        stop.synchronize()
        ms, gb = start.elapsed_time(stop) / reps, (torch.cuda.max_memory_allocated() - base) / 1e9
    except torch.cuda.OutOfMemoryError:
        ms, gb = None, None
    finally:
        s.grad = None
        torch.cuda.empty_cache()
    return {"eager_losses_ms": ms, "eager_losses_peak_gb": gb}


def _acc_sections(a, s, eager_reps):
    per = _trace("k_acc", lambda s: F_.acc_losses(a, s).sum().backward(), s)
    return {"acc_loss_kernels_ms": {name: sum(v) / len(v) for name, v in per.items()},
            **_eager(lambda s: A.totvar_loss(s, a) + A.asym_norm_loss(s), s, eager_reps)}


def _hosc_sections(a, s, eager_reps):
    def run(s):
        losses = F_.hosc_losses(a, s, 0.5, False)
        (0.5 * losses[0] + 0.5 * losses[1]).backward()

    per = _trace("hosc", run, s)
    return {"hosc_kernels_ms_and_launches": {name: [sum(v) / len(v), len(v) / TRACE_PASSES]
                                             for name, v in per.items()},
            **_eager(lambda s: 0.5 * O.cut_loss(a, s) + 0.5 * O.cut_loss(O.motif_adjacency(a), s), s, eager_reps)}


# name: (adjacency density, dtypes, (MinCut step, pooler step) builder, extra sections or None)
POOLERS = {
    "dmon": (0.05, ("fp32",), _dmon_steps, None),
    "acc": (0.05, ("fp32", "bf16"), _pool_steps(lambda x, a, s: T.acc_pool(x, a, s, **FLAGS)), _acc_sections),
    "hosc": (0.1, ("fp32", "bf16"), _pool_steps(lambda x, a, s: T.hosc_pool(x, a, s, None, 0.1, 0.5, False, **FLAGS)),
             _hosc_sections),
}


def _run(name, dtype, windows, eager_reps):
    density, _, steps, sections = POOLERS[name]
    x, a, s, gx, ga = _inputs(density, DTYPES[dtype])
    graphs = {key: _graph(run, x, s) for key, run in zip(("mincut", name), steps(x, a, s, gx, ga))}
    reps = {}
    for key, gr in graphs.items():  # warm-up, then size each window to at least 100 ms
        _window(gr, 20)
        reps[key] = max(50, int(100.0 / _window(gr, 50)) + 1)
    times = {key: [] for key in graphs}
    for _ in range(windows):
        for key, gr in graphs.items():
            times[key].append(_window(gr, reps[key]))
    med = {key: sorted(v)[len(v) // 2] for key, v in times.items()}
    del graphs
    extra = sections(a, s, eager_reps) if sections else {}
    return {"mincut_ms": med["mincut"], f"{name}_ms": med[name], "ratio": med[name] / med["mincut"], **extra,
            "mincut_ms_all": times["mincut"], f"{name}_ms_all": times[name], "reps_per_window": reps}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--pooler", choices=[*POOLERS, "all"], required=True)
    ap.add_argument("--windows", type=int, default=10)
    ap.add_argument("--eager-reps", type=int, default=5)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    head = {"device": torch.cuda.get_device_name(0), "power_limit": _power_limit(), "shape": [B, N, K, F]}
    lines = []
    for name in POOLERS if args.pooler == "all" else [args.pooler]:
        dtypes = POOLERS[name][1]
        if len(dtypes) == 1:  # one dtype: its results at the top level
            res = {**head, "dtype": dtypes[0], **_run(name, dtypes[0], args.windows, args.eager_reps)}
        else:
            res = dict(head)
            for dtype in dtypes:
                res[dtype] = _run(name, dtype, args.windows, args.eager_reps)
                torch.cuda.empty_cache()
        lines.append(json.dumps(res))
        print(lines[-1])
    if args.out:
        with open(args.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
