"""Times the per-graph epilogue / backward-assembly kernels of the dense path for several strip plans.

    python benchmarks/per_graph_kernels.py [c2|c3l1]

TGPB200_STRIP_ELEMS = matrix elements per CTA (the cluster size follows).
"""
import os
import sys

sys.path.insert(0, os.getcwd())
sys.path.insert(0, os.path.join(os.getcwd(), "torch-geometric-pool_b200"))
import torch

import bench
from tgp_b200 import _lib


def main():
    name = sys.argv[1] if len(sys.argv) > 1 else "c3l1"
    w = bench.WORKLOADS[name]
    a, s, x = (t.cuda() for t in bench.make_inputs(w, "cuda", 0))
    from tgp_b200 import functional as F_
    B, N, K, F = w["B"], w["N"], w["K"], w["F"]
    s.requires_grad_(True)
    x.requires_grad_(True)
    g_xp = torch.ones(B, K, F, dtype=a.dtype, device="cuda")
    g_ap = torch.ones(B, K, K, dtype=a.dtype, device="cuda")
    g_l = torch.zeros(4, dtype=torch.float32, device="cuda")
    kind = F_.LOSS_MINCUT if w["pooler"] == "mincut" else F_.LOSS_DIFFPOOL
    g_l[0 if w["pooler"] == "mincut" else 2] = 1.0
    g_l[1 if w["pooler"] == "mincut" else 3] = 1.0

    def step():
        s.grad = None
        x.grad = None
        xp, ap, losses = F_.dense_pool(x, a, s, remove_self_loops=True, degree_norm=True, adj_transpose=True,
                                       loss_kind=kind, ent_div=float(B * N))
        torch.autograd.backward([xp, ap, losses], [g_xp, g_ap, g_l])

    for elems in [2048, 4096, 8192, 16384, 32768, 1 << 20]:
        os.environ["TGPB200_STRIP_ELEMS"] = str(elems)
        row = [f"elems={elems:8d}"]
        for kern in ("k_graph_epilogue", "k_graph_bwd"):
            for _ in range(3):
                step()
            torch.cuda.synchronize()
            _lib.time_kernel(kern)
            for _ in range(10):
                step()
            torch.cuda.synchronize()
            ms, n = _lib.kernel_time_ms()
            _lib.time_kernel(None)
            row.append(f"{kern}: {ms * 1e3:8.1f} us (n={n})")
        print("  ".join(row), flush=True)


if __name__ == "__main__":
    main()
