"""Cost of DMoN on the fused dense path against MinCut at the C2 shape (B = 512, N = 256, K = 64, F = 128, fp32).

Each step is the fused forward + backward of ``dense_pool`` (loss_kind 3 vs 1, MinCut's connector flags), captured as
one CUDA graph.  The two graphs run in one process, alternating, over timed windows of at least 100 ms each; the
script prints the card name and power limit beside the per-step medians and their ratio.

    python benchmarks/dmon_step.py [--windows W] [--out FILE]
"""
import argparse
import json
import os
import subprocess
import sys

sys.path.insert(0, os.getcwd())
sys.path.insert(0, os.path.join(os.getcwd(), "torch-geometric-pool_b200"))
import torch

import tgp_b200 as T
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


def _graph(loss_kind, x, a, s, gx, ga, gl, gn):
    def step():
        x.grad = None
        s.grad = None
        xp, ap, losses = F_.dense_pool(x, a, s, loss_kind=loss_kind, graph_nodes=gn, **FLAGS)
        torch.autograd.backward([xp, ap, losses], [gx, ga, gl])
        return xp, ap, losses

    return T.GraphedStep(step)


def _window(graph, reps):
    start, stop = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    start.record()
    for _ in range(reps):
        graph.replay()
    stop.record()
    stop.synchronize()
    return start.elapsed_time(stop) / reps


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--windows", type=int, default=10)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    dev = "cuda"
    g = torch.Generator().manual_seed(0)
    a = (torch.rand(B, N, N, generator=g) < 0.05).float()
    a = torch.triu(a, 1)
    a = (a + a.transpose(1, 2)).to(dev)
    x = torch.randn(B, N, F, generator=g).to(dev).requires_grad_(True)
    s = torch.softmax(torch.randn(B, N, K, generator=g), -1).to(dev).requires_grad_(True)
    gx, ga = torch.randn(B, K, F, generator=g).to(dev), torch.randn(B, K, K, generator=g).to(dev)
    gl = torch.tensor([1.0, 1.0, 1.0, 0.0], device=dev)
    gn = torch.full((B,), float(N), device=dev)
    graphs = {"mincut": _graph(F_.LOSS_MINCUT, x, a, s, gx, ga, gl, None),
              "dmon": _graph(F_.LOSS_DMON, x, a, s, gx, ga, gl, gn)}
    reps = {}
    for name, gr in graphs.items():  # warm-up, then size each window to at least 100 ms
        _window(gr, 20)
        reps[name] = max(50, int(100.0 / _window(gr, 50)) + 1)
    times = {name: [] for name in graphs}
    for _ in range(args.windows):
        for name, gr in graphs.items():
            times[name].append(_window(gr, reps[name]))
    med = {name: sorted(v)[len(v) // 2] for name, v in times.items()}
    res = {
        "device": torch.cuda.get_device_name(0), "power_limit": _power_limit(), "shape": [B, N, K, F], "dtype": "fp32",
        "mincut_ms": med["mincut"], "dmon_ms": med["dmon"], "ratio": med["dmon"] / med["mincut"],
        "mincut_ms_all": times["mincut"], "dmon_ms_all": times["dmon"], "reps_per_window": reps,
    }
    line = json.dumps(res)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
