"""Cost of HOSC pooling against MinCut at the C2 shape (B = 512, N = 256, K = 64, F = 128), fp32 and bf16.

* HOSC step: ``hosc_pool`` forward + backward (alpha = 0.5, MinCut's orthogonality term: the fused dense call plus the
  ``hosc_losses`` products and kernels), MinCut step: ``mincut_pool`` forward + backward, both with MinCut's connector
  flags, only x and S requiring grad, captured as one CUDA graph each.  The two graphs run in one process,
  alternating, over timed windows of at least 100 ms each.
* The HOSC kernels and products alone (``k_hosc_*`` and the ``k_tc_gemm:hosc:*`` products), from CUDA events around
  each launch in an eager forward + backward pass, with the count of launches of each name per pass.
* The eager torch restatement of the two cut losses (``tests/hosc_oracle.py``: ``cut_loss`` of A and of
  ``motif_adjacency(A)``, forward + backward) on the same inputs: its time and its peak memory above the inputs.

The script prints the card name and power limit beside the numbers, one JSON line.

    python benchmarks/hosc_step.py [--windows W] [--eager-reps R] [--out FILE]
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

import hosc_oracle as O
import tgp_b200 as T
from tgp_b200 import _lib as L
from tgp_b200 import functional as F_

B, N, K, F = 512, 256, 64, 128
FLAGS = dict(remove_self_loops=True, degree_norm=True, adj_transpose=True)


def _power_limit():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
        return out or "unknown"
    except (OSError, subprocess.SubprocessError):
        return "unknown"


def _graph(pool, x, a, s, gx, ga):
    one = torch.ones((), device=x.device)

    def step():
        x.grad = None
        s.grad = None
        xp, ap, loss = pool(x, a, s)
        losses = list(loss.values())
        torch.autograd.backward([xp, ap, *losses], [gx, ga] + [one] * len(losses))
        return xp, ap, *losses

    return T.GraphedStep(step)


def _window(graph, reps):
    start, stop = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    start.record()
    for _ in range(reps):
        graph.replay()
    stop.record()
    stop.synchronize()
    return start.elapsed_time(stop) / reps


def _hosc(x, a, s):
    return T.hosc_pool(x, a, s, None, 0.1, 0.5, False, **FLAGS)


def _mincut(x, a, s):
    return T.mincut_pool(x, a, s, **FLAGS)


def _loss_kernels(a, s, reps=20):
    """{name: [mean ms, launches per pass]} of each launch named *hosc* over eager forward + backward passes of
    hosc_losses (alpha = 0.5)."""
    s = s.detach().requires_grad_(True)

    def run():
        s.grad = None
        losses = F_.hosc_losses(a, s, 0.5, False)
        (0.5 * losses[0] + 0.5 * losses[1]).backward()

    run()
    torch.cuda.synchronize()
    L.time_kernel("hosc")
    for _ in range(reps):
        run()
    torch.cuda.synchronize()
    per = {}
    for name, ms in L.kernel_trace():
        per.setdefault(name, []).append(ms)
    L.time_kernel(None)
    return {name: [sum(v) / len(v), len(v) / reps] for name, v in per.items()}


def _eager(a, s, reps):
    """The restated torch losses, forward + backward: mean ms and the peak memory (GB) above the inputs."""
    s = s.detach().requires_grad_(True)

    def run():
        s.grad = None
        (0.5 * O.cut_loss(a, s) + 0.5 * O.cut_loss(O.motif_adjacency(a), s)).backward()

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
        return start.elapsed_time(stop) / reps, (torch.cuda.max_memory_allocated() - base) / 1e9
    except torch.cuda.OutOfMemoryError:
        return None, None
    finally:
        s.grad = None
        torch.cuda.empty_cache()


def _run(dtype, windows, eager_reps):
    dev = "cuda"
    g = torch.Generator().manual_seed(0)
    a = (torch.rand(B, N, N, generator=g) < 0.1).float()
    a = torch.triu(a, 1)
    a = (a + a.transpose(1, 2)).to(dev, dtype)
    x = torch.randn(B, N, F, generator=g).to(dev, dtype).requires_grad_(True)
    s = torch.softmax(torch.randn(B, N, K, generator=g), -1).to(dev, dtype).requires_grad_(True)
    gx = torch.randn(B, K, F, generator=g).to(dev, dtype)
    ga = torch.randn(B, K, K, generator=g).to(dev, dtype)
    graphs = {"mincut": _graph(_mincut, x, a, s, gx, ga), "hosc": _graph(_hosc, x, a, s, gx, ga)}
    reps = {}
    for name, gr in graphs.items():  # warm-up, then size each window to at least 100 ms
        _window(gr, 20)
        reps[name] = max(50, int(100.0 / _window(gr, 50)) + 1)
    times = {name: [] for name in graphs}
    for _ in range(windows):
        for name, gr in graphs.items():
            times[name].append(_window(gr, reps[name]))
    med = {name: sorted(v)[len(v) // 2] for name, v in times.items()}
    del graphs
    kernels = _loss_kernels(a, s)
    eager_ms, eager_gb = _eager(a, s, eager_reps)
    return {
        "mincut_ms": med["mincut"], "hosc_ms": med["hosc"], "ratio": med["hosc"] / med["mincut"],
        "hosc_kernels_ms_and_launches": kernels, "eager_losses_ms": eager_ms, "eager_losses_peak_gb": eager_gb,
        "mincut_ms_all": times["mincut"], "hosc_ms_all": times["hosc"], "reps_per_window": reps,
    }


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--windows", type=int, default=10)
    ap.add_argument("--eager-reps", type=int, default=5)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    res = {"device": torch.cuda.get_device_name(0), "power_limit": _power_limit(), "shape": [B, N, K, F]}
    for name, dtype in (("fp32", torch.float32), ("bf16", torch.bfloat16)):
        res[name] = _run(dtype, args.windows, args.eager_reps)
        torch.cuda.empty_cache()
    line = json.dumps(res)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
