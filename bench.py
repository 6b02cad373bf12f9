#!/usr/bin/env python
"""bench.py -- coarsened graphs/s of the Reduce + Connect hot path (forward + backward).

Headline workload (BASELINE.json configs[1], "C2"): MinCutPooling dense, 64 clusters, batch 512 graphs x 256
nodes x 128 feats, fp32, S^T X + S^T A S + mincut/ortho losses + post-processing, fwd+bwd.  One "step" = one pass
of the path over one batch of 512 graphs per GPU (weak scaling: every rank owns its own 512 graphs, no data-path
collective).  The step runs as ONE CUDA graph (tgp_b200.GraphedStep: the dense path never synchronises), so the
timed region holds no Python / allocator / launch overhead; the eager time is reported beside it.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--workload all|c1|c2|c3|c4|c5]
                    [--dump-outputs DIR]

Prints ONE JSON line (rank 0).  `value` = graphs/s with inputs resident in HBM over exactly K timed steps;
`long_run` repeats the measurement over a >= 100 ms region; `e2e` = the same metric through the public API from
pinned HOST buffers (edge list + features copied in every step, densified on the device, losses read back);
`roofline` = algorithmic bytes of the dominant kernel / its CUDA-event duration / MEASURED_PEAKS.json;
`kernels` = per-kernel time of one step (separate eager pass) and `host_gap_ms` = ms_per_step - their sum;
`configs` = a measured entry (ms_per_step, roofline, ...) for every BASELINE.json config (C1..C5) that the
launch can run; `cpu_baseline` = the CPU oracle (restated reference path) on a bounded sample.

`--dump-outputs DIR` writes what the last timed step of the headline (dense) workload computed on rank 0 as
DIR/<name>.npy in float32: the last level's pooled features `x_pool` and adjacency `adj_pool`, the `losses`
([mincut, ortho, link, entropy], one row per level when there are several), and the gradients `grad_x` and `grad_s<i>`
of X and of each level's assignment.  The inputs depend only on the workload and the rank, so two builds can be compared
array for array.  Per-graph arrays are a fixed, seeded sample of the batch's graphs when all of them would exceed 64 MB.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
for p in (ROOT, os.path.join(ROOT, "torch-geometric-pool_b200")):
    if p not in sys.path:
        sys.path.insert(0, p)

import torch  # noqa: E402

METRIC = "coarsened graphs/s (Reduce+Connect fwd+bwd)"
DUMP_BYTES = 64 * 10**6  # upper bound of what --dump-outputs writes

DENSE = {
    "c2": dict(B=512, levels=[(256, 64)], F=128, dtype="f32", p=0.05, pooler="mincut", scaling="weak",
               desc="MinCutPooling dense, K=64, 512 graphs x 256 nodes x 128 feats, fp32, fwd+bwd"),
    "c3": dict(B=1024, levels=[(512, 256), (256, 64), (64, 16)], F=256, dtype="bf16", p=0.02, pooler="diff",
               scaling="strong",
               desc="DiffPool dense, 3 chained levels (512->256->64->16 clusters), 1024 graphs x 512 nodes x 256 "
                    "feats, bf16, fwd+bwd"),
}
SPARSE = {
    "c1": dict(kind="topk", graphs=128, n_lo=24, n_hi=36, p=0.1, F=64,
               desc="TopK ratio 0.5 + sum reduce + kept-node connect, 128 ER graphs (~30 nodes, 64 feats), fwd+bwd"),
    "c4": dict(kind="cluster", N=1_000_000, E=20_000_000, F=128,
               desc="cluster connect (remap + coalesce sum + self-loop removal) + mean reduce, 1M nodes / 20M edges "
                    "power-law, 128 feats, matching-style cluster map (K ~ 0.55 N), fwd+bwd"),
    "c5": dict(kind="topk_big", N=16_000_000, E=400_000_000, F=128,
               desc="TopK 50% kept-node connect (degree-normalised) + sum reduce on one 16M-node / 400M-edge graph, "
                    "128 feats, fwd+bwd, edge-sharded over the GPUs"),
}


def config_of(name, gpus):
    """The `config` object: identical for the b200 and the reference arm of one launch."""
    if name in DENSE:
        w = DENSE[name]
        return {"workload": w["desc"], "graphs_per_step": w["B"], "loss": "x_pool.sum()+adj_pool.sum()+aux losses",
                "gpus": gpus, "scaling": w["scaling"]}
    w = SPARSE[name]
    return {"workload": w["desc"], "gpus": gpus}


def peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.isfile(path):
        d = json.load(open(path))
        return float(d["hbm_gbs"]), float(d.get("bf16_tflops_sustained", d.get("bf16_tflops", 1400.0))), "measured"
    return 6650.0, 1400.0, "fallback"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def __enter__(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100", "-i",
                 str(self.index)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None
        return self

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def __exit__(self, *exc):
        if self.proc is not None:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=2)
            except Exception:
                self.proc.kill()

    def summary(self):
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[1]))
                mx.append(float(r[2]))
                for n, v in zip(names, r[4:8]):
                    if v.lower().startswith("active"):
                        reasons.add(n)
            except Exception:
                continue
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        return {"sm_mhz": statistics.median(sm), "sm_max_mhz": max(mx), "reasons": sorted(reasons), "samples": len(sm)}


# --------------------------------------------------------------------------------------------------------------
# timing helpers
# --------------------------------------------------------------------------------------------------------------
def bind_to_gpu_numa_node(local_rank):
    """Run this rank (and first-touch its pinned host buffers) on the NUMA node its GPU hangs off: the end-to-end leg is
    bound by host -> device DMA, and a pinned buffer on the other socket crosses the inter-socket link first.  Best
    effort: returns a description, or None when the topology is not exposed (single node, container without sysfs)."""
    try:
        bus = torch.cuda.get_device_properties(local_rank).pci_bus_id
        dom = getattr(torch.cuda.get_device_properties(local_rank), "pci_domain_id", 0)
        dev_id = getattr(torch.cuda.get_device_properties(local_rank), "pci_device_id", 0)
        path = f"/sys/bus/pci/devices/{dom:04x}:{bus:02x}:{dev_id:02x}.0/numa_node"
        node = int(open(path).read().strip())
        if node < 0:
            return None
        cpus = set()
        for part in open(f"/sys/devices/system/node/node{node}/cpulist").read().strip().split(","):
            lo, _, hi = part.partition("-")
            cpus.update(range(int(lo), int(hi or lo) + 1))
        cpus &= os.sched_getaffinity(0)
        if not cpus:
            return None
        os.sched_setaffinity(0, cpus)
        return {"numa_node": node, "cpus": len(cpus)}
    except Exception:
        return None


class Ctx:
    def __init__(self, args):
        self.args = args
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.rank = int(os.environ.get("RANK", "0"))
        self.local_rank = int(os.environ.get("LOCAL_RANK", "0"))
        self.dist = None
        torch.cuda.set_device(self.local_rank)
        self.dev = torch.device("cuda", self.local_rank)
        self.numa = bind_to_gpu_numa_node(self.local_rank) if self.world > 1 else None
        if self.world > 1:
            import torch.distributed as dist_

            self.dist = dist_
            self.dist.init_process_group("nccl", device_id=self.dev)

    def barrier(self):
        if self.dist is not None:
            self.dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(self, v):
        if self.dist is None:
            return v
        t = torch.tensor([v], dtype=torch.float64, device=self.dev)
        self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return float(t.item())

    def timed(self, fn, steps):
        """ms per step over exactly `steps` calls, barrier + synchronize on both sides, max over ranks."""
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        self.barrier()
        e0.record()
        for _ in range(steps):
            fn()
        e1.record()
        self.barrier()
        return self.max_over_ranks(e0.elapsed_time(e1)) / steps

    def long_run(self, fn, target_ms=150.0, lo=5, hi=4000):
        """A second measurement whose timed region lasts >= ~target_ms (the step count is the same on all ranks)."""
        probe = self.timed(fn, 3)
        steps = int(min(hi, max(lo, target_ms / max(probe, 1e-4))))
        if self.dist is not None:
            t = torch.tensor([steps], dtype=torch.int64, device=self.dev)
            self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
            steps = int(t.item())
        return {"steps": steps, "ms_per_step": self.timed(fn, steps)}


def kernel_table(fn, steps=5):
    """Per-kernel CUDA-event times of `fn` (eager, a separate pass outside every headline region):
    ({name: {"launches_per_step", "ms_per_step"}}, sum of kernel ms per step, first-occurrence trace of one step)."""
    from tgp_b200 import _lib

    fn()
    torch.cuda.synchronize()
    _lib.time_kernel("*")
    for _ in range(steps):
        fn()
    torch.cuda.synchronize()
    trace = _lib.kernel_trace()
    _lib.time_kernel(None)
    agg = {}
    for name, ms in trace:
        a = agg.setdefault(name, [0, 0.0])
        a[0] += 1
        a[1] += ms
    table = {k: {"launches_per_step": v[0] / steps, "ms_per_step": round(v[1] / steps, 5)} for k, v in agg.items()}
    one_step = trace[: len(trace) // steps] if steps > 0 else trace
    return table, sum(v[1] for v in agg.values()) / steps, one_step


# --------------------------------------------------------------------------------------------------------------
# dense workloads (C2, C3)
# --------------------------------------------------------------------------------------------------------------
def dense_inputs(w, B, dev, seed):
    g = torch.Generator(device=dev).manual_seed(seed)
    N, K0 = w["levels"][0]
    dt = torch.float32 if w["dtype"] == "f32" else torch.bfloat16
    a = (torch.rand(B, N, N, device=dev, generator=g) < w["p"]).float()
    a = torch.triu(a, 1)
    a = (a + a.transpose(1, 2)).to(dt).contiguous()
    x = torch.randn(B, N, w["F"], device=dev, generator=g).to(dt)
    s = [torch.softmax(torch.randn(B, n, k, device=dev, generator=g), -1).to(dt) for n, k in w["levels"]]
    return a, x, s


def dense_alg_bytes(w, B):
    """SURVEY 8(d) per level: fwd = es B (N^2 + NK + NF + KF + K^2); bwd re-reads A, S, X and the two upstream
    gradients and writes dS, dX: es B (N^2 + 2NK + 2NF + KF + K^2)."""
    es = 4 if w["dtype"] == "f32" else 2
    F = w["F"]
    fwd = bwd = 0
    for (N, K) in w["levels"]:
        fwd += es * B * (N * N + N * K + N * F + K * F + K * K)
        bwd += es * B * (N * N + 2 * N * K + 2 * N * F + K * F + K * K)
    return fwd, bwd


class DenseStep:
    """fwd + bwd of the (chained) dense pooling levels on static device tensors, as explicit upstream gradients:
    loss = x_pool.sum() + adj_pool.sum() + aux losses (examples/time_and_mem_test.py:380-383, plus the pooled
    adjacency so that the connect backward is exercised)."""

    def __init__(self, w, B, dev, seed):
        from tgp_b200 import functional as F_

        self.F_, self.w, self.B = F_, w, B
        self.a, self.x, self.s = dense_inputs(w, B, dev, seed)
        self.x.requires_grad_(True)
        for t in self.s:
            t.requires_grad_(True)
        Kl = w["levels"][-1][1]
        dt = self.a.dtype
        self.g_xp = torch.ones(B, Kl, w["F"], dtype=dt, device=dev)
        self.g_ap = torch.ones(B, Kl, Kl, dtype=dt, device=dev)
        self.g_l = torch.zeros(4, dtype=torch.float32, device=dev)
        if w["pooler"] == "mincut":
            self.g_l[0] = self.g_l[1] = 1.0
            self.kind = F_.LOSS_MINCUT
        else:
            self.g_l[2] = self.g_l[3] = 1.0
            self.kind = F_.LOSS_DIFFPOOL

    def run(self, a=None, x=None, s=None):
        a = self.a if a is None else a
        x = self.x if x is None else x
        s = self.s if s is None else s
        x.grad = None
        for t in s:
            t.grad = None
        xl, al, outs, grads = x, a, [], []
        for (n, k), sl in zip(self.w["levels"], s):
            xl, al, losses = self.F_.dense_pool(xl, al, sl, remove_self_loops=True, degree_norm=True,
                                                adj_transpose=True, loss_kind=self.kind, ent_div=float(self.B * n))
            outs.append(losses)
            grads.append(self.g_l)
        torch.autograd.backward([xl, al] + outs, [self.g_xp, self.g_ap] + grads)
        return xl, al, outs[0] if len(outs) == 1 else torch.stack(outs)

    def outputs(self, step_out):
        """What the caller of one step receives (`step_out` = what `run` returned; the gradients are read from X and S),
        as float32 arrays for --dump-outputs.  Per-graph arrays keep a fixed, seeded sample of the graphs when all of
        them would exceed DUMP_BYTES."""
        xl, al, losses = step_out
        per_graph = {"x_pool": xl, "adj_pool": al, "grad_x": self.x.grad}
        per_graph.update({f"grad_s{i}": t.grad for i, t in enumerate(self.s)})
        graph_bytes = sum(4 * t[0].numel() for t in per_graph.values())
        n = min(self.B, (DUMP_BYTES - 4 * losses.numel()) // graph_bytes)
        keep = torch.randperm(self.B, generator=torch.Generator().manual_seed(0))[:n].sort().values.to(xl.device)
        out = {k: t.detach().index_select(0, keep).float() for k, t in per_graph.items()}
        out["losses"] = losses.detach().float().clone()
        return out


def run_dense(ctx, name, headline):
    import tgp_b200 as T
    from tgp_b200 import _lib

    args, w = ctx.args, DENSE[name]
    B = w["B"] if w["scaling"] == "weak" else max(w["B"] // ctx.world, 1)
    st = DenseStep(w, B, ctx.dev, 1000 + ctx.rank)
    total_graphs = B * ctx.world
    warm = max(args.warmup, 3)
    for _ in range(warm):
        st.run()
    ctx.barrier()
    eager_ms = ctx.timed(st.run, min(args.steps, 50))
    graphed = T.GraphedStep(st.run, warmup=1)
    for _ in range(warm):
        graphed.replay()
    ctx.barrier()
    out = {}
    if headline:
        # nvidia-smi samples every 100 ms while a step takes < 1 ms: the sampler also covers a soak of the same
        # graph replay right before and after the timed region (same load, same clocks)
        with ClockSampler(ctx.local_rank) as clk:
            t_soak = time.perf_counter() + 1.0
            while time.perf_counter() < t_soak:
                for _ in range(50):
                    graphed.replay()
                torch.cuda.synchronize()
            ms = ctx.timed(graphed.replay, args.steps)
            if args.dump_outputs:
                out["_dump"] = st.outputs(graphed.outputs)
            long = ctx.long_run(graphed.replay)
            t_soak = time.perf_counter() + 0.3
            while time.perf_counter() < t_soak:
                graphed.replay()
            torch.cuda.synchronize()
        out["clocks"] = clk.summary()
    else:
        ms = ctx.timed(graphed.replay, max(args.steps, 10))
        long = ctx.long_run(graphed.replay)
    table, ksum, trace = kernel_table(st.run)
    hbm, tf, src = peaks()
    fwd_b, bwd_b = dense_alg_bytes(w, B)
    roof = {"peak_source": f"{src} (MEASURED_PEAKS.json)", "algorithmic_bytes_step": fwd_b + bwd_b,
            "step_frac_hbm": (fwd_b + bwd_b) / (long["ms_per_step"] * 1e-3) / 1e9 / hbm}
    if name == "c2":
        # dominant launch: the larger of the two fused kernels -- the forward main kernel (one pass over A, X, S per graph,
        # algorithmic bytes = the forward's) or the fused backward (W = A S in tensor memory -> dS, dX; algorithmic bytes =
        # the backward's).  Both are listed under "fused_kernels".  If the shape took neither, the roofline is the step's.
        cand = {}
        for k in table:
            if k.startswith("k_dense_fwd_fused"):
                cand[k] = fwd_b
            elif k.startswith("k_dense_bwd_fused"):
                cand[k] = bwd_b
        dom = sorted(cand, key=lambda k: -table[k]["ms_per_step"])
        if dom:
            tpath = os.path.join(ROOT, "profiles", "r2_traffic.json")
            tr = json.load(open(tpath)) if os.path.isfile(tpath) else {}
            per = {}
            for k in dom:
                kms = table[k]["ms_per_step"] / max(table[k]["launches_per_step"], 1)
                ach = cand[k] / (kms * 1e-3) / 1e9
                per[k] = {"kernel_ms": kms, "algorithmic_bytes": cand[k], "achieved": ach, "frac": ach / hbm,
                          "traffic": tr.get(k)}
            d0 = per[dom[0]]
            roof.update({"bound": "hbm", "achieved": d0["achieved"], "peak": hbm, "unit": "GB/s", "frac": d0["frac"],
                         "traffic": d0["traffic"], "traffic_source": "profiles/r2_traffic.json (ncu --set full, per launch)",
                         "kernel": dom[0], "kernel_ms": d0["kernel_ms"], "algorithmic_bytes": d0["algorithmic_bytes"],
                         "fused_kernels": per})
        else:
            ach = (fwd_b + bwd_b) / (long["ms_per_step"] * 1e-3) / 1e9
            roof.update({"bound": "hbm", "achieved": ach, "peak": hbm, "unit": "GB/s", "frac": ach / hbm,
                         "traffic": None, "kernel": "whole step", "algorithmic_bytes": fwd_b + bwd_b})
    else:
        # C3 level 1 is tensor-bound: S^T A S = T = S^T A (2 B K N^2) and A_raw = T S (2 B K^2 N), timed as the first
        # launches of those two products in the step (level 1)
        N, K = w["levels"][0]
        t_ms = sum(next((ms_ for nm, ms_ in trace if nm == tag), 0.0)
                   for tag in ("k_tc_gemm:T=StA", "k_tc_gemm:Araw=TS"))
        fl = 2.0 * B * K * N * N + 2.0 * B * K * K * N
        ach = fl / (t_ms * 1e-3) / 1e12 if t_ms > 0 else 0.0
        roof.update({"bound": "tensor", "achieved": ach, "peak": tf, "unit": "TFLOP/s", "frac": ach / tf,
                     "traffic": None, "kernel": "S^T A S of level 1 (k_tc_gemm:T=StA + k_tc_gemm:Araw=TS)",
                     "kernel_ms": t_ms, "flops": fl})
    out.update({
        "ms_per_step": ms, "value": total_graphs / (ms * 1e-3), "unit": "graphs/s", "graphs_per_gpu": B,
        "scaling": w["scaling"], "dtype": w["dtype"], "steps": args.steps if headline else max(args.steps, 10),
        "mode": "one CUDA graph per step (tgp_b200.GraphedStep)", "eager_ms_per_step": eager_ms,
        "long_run": long, "gpu_launches_per_step": graphed.kernels_per_replay,
        "kernel_ms_sum": ksum, "host_gap_ms": long["ms_per_step"] - ksum, "eager_host_gap_ms": eager_ms - ksum,
        "kernels": table, "roofline": roof,
        "l2_policy": "inputs + saved tensors larger than L2 (126 MB), no flush",
    })
    out["_step"] = st
    out["_graphed"] = graphed
    return out


def dense_e2e(ctx, name):
    """End to end through the public API from pinned HOST buffers, the way a PyG pipeline feeds a dense pooler
    (tgp/src.py:374-452): per step the batch's edge list, node features and batch vector are copied host -> device,
    densified on the device (to_dense_adj / to_dense_batch kernels), the assignment comes from a linear + softmax
    select on the device (MLPSelect's role; torch ops, outside the path), then the fused pool runs fwd + bwd and the
    losses are read back.  Two buffer sets / two captured graphs: the copy of step i+1 overlaps the compute of step i."""
    import tgp_b200 as T
    from tgp_b200 import functional as F_

    w = DENSE[name]
    B, (N, K), F = w["B"], w["levels"][0], w["F"]
    dev = ctx.dev
    a, x, _ = dense_inputs(w, B, dev, 2000 + ctx.rank)
    nz = a.float().nonzero()  # (b, i, j) row-major = PyG block-diagonal order
    ei_h = torch.stack([nz[:, 0] * N + nz[:, 1], nz[:, 0] * N + nz[:, 2]]).cpu().pin_memory()
    x_h = x.float().reshape(B * N, F).cpu().pin_memory()
    batch_h = torch.arange(B).repeat_interleave(N).pin_memory()
    del a, x, nz
    wsel = torch.randn(F, K, device=dev) / F ** 0.5
    kind = F_.LOSS_MINCUT if w["pooler"] == "mincut" else F_.LOSS_DIFFPOOL
    g_xp = torch.ones(B, K, F, device=dev)
    g_ap = torch.ones(B, K, K, device=dev)
    g_l = torch.zeros(4, device=dev)
    g_l[0] = g_l[1] = 1.0

    copy_stream = torch.cuda.Stream(device=dev)
    main_stream = torch.cuda.current_stream(dev)
    sets = []
    for _ in range(2):
        bufs = (torch.empty_like(ei_h, device=dev), torch.empty_like(x_h, device=dev),
                torch.empty_like(batch_h, device=dev))

        def step(bufs=bufs):
            ei, xf, batch = bufs
            adj = F_.to_dense_adj(ei, batch, None, num_graphs=B, max_num_nodes=N)
            x3, _ = F_.to_dense_batch(xf, batch, B, N)
            s = torch.softmax(x3 @ wsel, -1).requires_grad_(True)
            x3 = x3.requires_grad_(True)
            xp, ap, losses = F_.dense_pool(x3, adj, s, remove_self_loops=True, degree_norm=True, adj_transpose=True,
                                           loss_kind=kind, ent_div=float(B * N))
            torch.autograd.backward([xp, ap, losses], [g_xp, g_ap, g_l])
            return losses

        for dst, src in zip(bufs, (ei_h, x_h, batch_h)):
            dst.copy_(src)
        sets.append((bufs, T.GraphedStep(step, warmup=2)))
    consumed = [None, None]

    def stage(j):
        with torch.cuda.stream(copy_stream):
            if consumed[j] is not None:
                copy_stream.wait_event(consumed[j])
            for dst, src in zip(sets[j][0], (ei_h, x_h, batch_h)):
                dst.copy_(src, non_blocking=True)
            done = torch.cuda.Event()
            done.record(copy_stream)
        return done

    def loop(n):
        ready = stage(0)
        for i in range(n):
            j = i & 1
            main_stream.wait_event(ready)
            if i + 1 < n:
                ready = stage(j ^ 1)
            losses = sets[j][1].replay()
            consumed[j] = torch.cuda.Event()
            consumed[j].record(main_stream)
            losses.cpu()  # device -> host read of the step's result

    loop(3)
    steps = max(5, min(ctx.args.steps, 40))
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ctx.barrier()
    e0.record()
    loop(steps)
    e1.record()
    ctx.barrier()
    ms = ctx.max_over_ranks(e0.elapsed_time(e1)) / steps
    h2d = sum(t.numel() * t.element_size() for t in (ei_h, x_h, batch_h))
    return {"value": ctx.world * B / (ms * 1e-3), "unit": "graphs/s", "h2d_bytes_per_step": h2d,
            "d2h_bytes_per_step": 16, "ms_per_step": ms, "steps": steps,
            "inputs": "pinned host edge_index [2,E] int64 + x [B*N,F] fp32 + batch [B*N] int64 per step",
            "pipeline": "H2D of step i+1 on a copy stream overlaps the graph replay of step i; on-device "
                        "to_dense_adj / to_dense_batch + linear-softmax select + fused pool fwd+bwd; losses read back",
            "host_numa_binding": ctx.numa}


# --------------------------------------------------------------------------------------------------------------
# sparse workloads (C1, C4, C5)
# --------------------------------------------------------------------------------------------------------------
def powerlaw_graph(n, e, device, seed):
    """Chung-Lu style power-law graph (exponent 2.3), symmetric, no self loops, sorted by (row, col)."""
    g = torch.Generator(device=device).manual_seed(seed)
    w = (torch.arange(1, n + 1, device=device, dtype=torch.float32)) ** (-1.0 / 1.3)
    cdf = torch.cumsum(w.double(), 0)
    cdf = (cdf / cdf[-1]).float()
    half = e // 2
    src = torch.searchsorted(cdf, torch.rand(half, device=device, generator=g)).clamp_(max=n - 1)
    dst = torch.randint(0, n, (half,), device=device, generator=g)
    keep = src != dst
    src, dst = src[keep], dst[keep]
    perm = torch.randperm(n, device=device, generator=g)  # hubs are spread over the id range
    src, dst = perm[src], perm[dst]
    key = torch.cat([src * n + dst, dst * n + src])
    del src, dst, keep, perm
    key = torch.sort(key)[0]
    return torch.stack([key // n, key % n])


def er_batch(w, seed):
    gc = torch.Generator().manual_seed(seed)
    eis, bs, off = [], [], 0
    for gi in range(w["graphs"]):
        n = int(torch.randint(w["n_lo"], w["n_hi"] + 1, (1,), generator=gc))
        up = torch.triu(torch.rand(n, n, generator=gc) < w["p"], 1)
        r, c = up.nonzero(as_tuple=True)
        eis.append(torch.cat([torch.stack([r, c]), torch.stack([c, r])], 1) + off)
        bs.append(torch.full((n,), gi))
        off += n
    ei = torch.cat(eis, 1)
    ei = ei[:, torch.argsort(ei[0] * off + ei[1])]
    return ei, torch.cat(bs), off


def matching_clusters(N, dev, g):
    """Matching-style map: a random pairing along a permutation, ~45 % of the nodes paired -> K ~ 0.55 N."""
    perm = torch.randperm(N, device=dev, generator=g)
    paired = int(0.9 * N) // 2 * 2
    cl = torch.empty(N, dtype=torch.long, device=dev)
    cl[perm[:paired]] = torch.arange(paired // 2, device=dev).repeat_interleave(2)
    cl[perm[paired:]] = torch.arange(paired // 2, paired // 2 + N - paired, device=dev)
    return cl, paired // 2 + N - paired


def per_graph_topk(score, batch, dev):
    """Per-graph top half by score (selection is upstream of the path and timed separately)."""
    N = score.numel()
    order = torch.argsort(batch * 4.0 - score)  # graph asc, score desc
    ptr = torch.zeros(int(batch.max()) + 2, dtype=torch.long, device=dev)
    ptr[1:] = torch.bincount(batch).cumsum(0)
    rank_in = torch.arange(N, device=dev) - ptr[batch[order]]
    keep = rank_in < ((ptr[1:] - ptr[:-1] + 1) // 2)[batch[order]]
    return order[keep]


def sparse_alg_bytes(E, e_out, nnz, K, N, F, train):
    """SURVEY 8(d): edges in (2*8+4) + edges out (2*8+4) + index map + x rows in + x_pool out; the backward adds the
    feature gradients (x_pool grad in, x grad out) and the two edge-weight gradient vectors."""
    alg = 20 * E + 20 * e_out + 8 * nnz + 4 * F * (nnz + K)
    if train:
        alg += 4 * F * (N + K) + 4 * E + 4 * e_out
    return alg


def run_sparse(ctx, name):
    import tgp_b200 as T
    from tgp_b200 import _lib
    from tgp_b200 import functional as F_

    args, w = ctx.args, SPARSE[name]
    dev = ctx.dev
    g = torch.Generator(device=dev).manual_seed(0)
    F = w["F"]
    if w["kind"] == "topk":
        ei, batch, N = er_batch(w, 0)
        ei, batch = ei.to(dev), batch.to(dev)
        units, G = w["graphs"], w["graphs"]
    else:
        N = w["N"]
        ei = powerlaw_graph(N, w["E"], dev, 0)
        batch, units, G = None, 1, 1
    E = ei.size(1)
    x = torch.randn(N, F, device=dev, generator=g).requires_grad_(True)
    ew = (torch.rand(E, device=dev, generator=g) + 0.5).requires_grad_(True)
    if w["kind"] == "cluster":
        cl, K = matching_clusters(N, dev, g)
        so = T.SelectOutput(cluster_index=cl, num_nodes=N, num_supernodes=K)
        reduce_op, fresh_so, degree_norm = "mean", False, False
        F_.csr_of(so)  # pre-coarsened pipeline: the cluster CSR is cached on the SelectOutput and reused
    else:
        score = torch.tanh(torch.randn(N, device=dev, generator=g))
        node_index = torch.topk(score, N // 2).indices if batch is None else per_graph_topk(score, batch, dev)
        K = node_index.numel()
        so = T.SelectOutput(node_index=node_index, num_nodes=N, cluster_index=torch.arange(K, device=dev),
                            num_supernodes=K, weight=score[node_index])
        # TopK makes a new SelectOutput every step: the CSR build belongs to the step
        reduce_op, fresh_so, degree_norm = "sum", True, w["kind"] == "topk_big"
    torch.cuda.synchronize()
    e_out_box = [0]
    # upstream gradients (what the next layer hands back) live outside the step, as in the dense workloads
    up = {"xp": torch.ones(K, F, device=dev), "w": None}

    def eager():
        x.grad = None
        ew.grad = None
        if fresh_so:
            so._b200_csr = None
        xp, eo, wo, _ = T.sparse_pool(x, ei, so, edge_weight=ew, batch=batch, reduce_op=reduce_op,
                                      degree_norm=degree_norm)
        if up["w"] is None or up["w"].numel() != wo.numel():
            up["w"] = torch.ones_like(wo)
        torch.autograd.backward([xp, wo], [up["xp"], up["w"]])
        e_out_box[0] = eo.size(1)

    warm = max(args.warmup, 3)
    for _ in range(warm):
        eager()
    torch.cuda.synchronize()
    launches0 = _lib.kernel_launches()
    eager()
    torch.cuda.synchronize()
    launches = _lib.kernel_launches() - launches0
    e_out = e_out_box[0]
    eager_run = ctx.long_run(eager)
    out = {"mode": "eager public API (one host read of the coarse edge count per step)",
           "ms_per_step": eager_run["ms_per_step"], "long_run": eager_run, "gpu_launches_per_step": launches}
    if w["kind"] in ("topk", "cluster"):
        # the no-host-read form captured as one CUDA graph (launch-bound batch; for the 20 M-edge cluster connect it
        # removes the two host reads and the launch gaps of ~40 kernels, at the price of capacity-sized launches)
        g_xp = up["xp"]
        g_w = torch.ones(E, device=dev)

        def padded():
            x.grad = None
            ew.grad = None
            if fresh_so:
                so._b200_csr = None
            xp, eo, wo, _, cnt = T.sparse_pool_padded(x, ei, so, edge_weight=ew, batch=batch, reduce_op=reduce_op,
                                                      degree_norm=degree_norm, num_graphs=G)
            torch.autograd.backward([xp, wo], [g_xp, g_w])
            return cnt

        graphed = T.GraphedStep(padded, warmup=2)

        def replay_and_read():
            graphed.replay()

        gr = ctx.long_run(replay_and_read)
        out["eager_ms_per_step"] = eager_run["ms_per_step"]
        out["graph_ms_per_step"] = gr["ms_per_step"]
        if gr["ms_per_step"] < eager_run["ms_per_step"]:
            out.update({"mode": "one CUDA graph per step (tgp_b200.sparse_pool_padded + GraphedStep: device-side edge "
                                "count, no host read inside the step)",
                        "ms_per_step": gr["ms_per_step"], "long_run": gr,
                        "gpu_launches_per_step": graphed.kernels_per_replay})
        del graphed
    if w["kind"] == "topk":
        sel = ctx.long_run(lambda: T.topk(score, 0.5, batch, num_graphs=G), target_ms=30.0)
        out["select_ms"] = sel["ms_per_step"]  # TopK selection kernel (upstream of the path), incl. its host read
    table, ksum, _ = kernel_table(eager, steps=3)
    hbm, _, src = peaks()
    nnz = so.node_index.numel()
    alg = sparse_alg_bytes(E, e_out, nnz, K, N, F, True)
    ms = out["ms_per_step"]
    # the memory-bound kernels of the step against their OWN algorithmic bytes (what each must move at least once);
    # bytes and time are both per STEP for the kernel name (the coalesce backward is a main launch + an E % 4 tail)
    own = {
        "k_segment_reduce_fwd": 4 * F * (nnz + K) + 16 * nnz,            # gathered rows in, pooled rows out, index + weight
        "k_segment_reduce_bwd": 4 * F * (N + nnz) + 16 * nnz,            # pooled-gradient rows in, x-gradient rows out
        "k_compact_emit": 12 * e_out + 20 * e_out,                       # virtual coarse edges in, int64 edge list out
        "k_coalesce_bwd": 8 * E + 4 * e_out,                             # slot + gradient out per edge, coarse gradient in
    }
    if w["kind"] != "cluster":  # the cluster path uses this kernel only to compact the hub rows' members
        own["k_compact_onepass"] = 20 * E + 20 * e_out                   # kept-node filter: edges in, survivors out
    kroof = {}
    for kname, nbytes in own.items():
        if kname in table and table[kname]["ms_per_step"] > 0:
            t = table[kname]["ms_per_step"]
            kroof[kname] = {"algorithmic_bytes": nbytes, "kernel_ms": t, "achieved": nbytes / (t * 1e-3) / 1e9,
                            "frac": nbytes / (t * 1e-3) / 1e9 / hbm}
    out["kernel_rooflines"] = kroof
    out.update({
        "value": units / (ms * 1e-3), "unit": "graphs/s", "scaling": "weak", "dtype": "f32",
        "shape": {"N": N, "E": E, "K": K, "E_out": e_out, "F": F},
        "kernel_ms_sum": ksum, "host_gap_ms": ms - ksum,
        "eager_host_gap_ms": eager_run["ms_per_step"] - ksum, "kernels": table,
        "roofline": {"bound": "hbm", "achieved": alg / (ms * 1e-3) / 1e9, "peak": hbm, "unit": "GB/s",
                     "frac": alg / (ms * 1e-3) / 1e9 / hbm, "traffic": None, "kernel": "whole step",
                     "kernel_frac": alg / (ksum * 1e-3) / 1e9 / hbm if ksum > 0 else None,
                     "algorithmic_bytes": alg, "peak_source": f"{src} (MEASURED_PEAKS.json hbm_gbs)"},
        "l2_policy": ("working set fits L2 (latency-bound config)" if w["kind"] == "topk"
                      else "inputs larger than L2 (126 MB), no flush"),
    })
    return out


def run_c5_sharded(ctx):
    """One 16M-node / 400M-edge graph over N GPUs (strong scaling): edges in contiguous ranges (global edge order =
    rank order), kept nodes in contiguous node ranges.  Per step and rank: CSR + sum reduce of the local kept nodes,
    local kept-node filter + relabel, one all-reduce of the per-rank edge counts, degree normalisation with one
    all-reduce (sum) of the [K] degree partials in the forward and of the [K] gradient partials in the backward."""
    import tgp_b200 as T
    from tgp_b200 import _lib
    from tgp_b200 import distributed as D
    from tgp_b200 import functional as F_

    w = SPARSE["c5"]
    dev, world, rank = ctx.dev, ctx.world, ctx.rank
    N, F = w["N"], w["F"]
    g = torch.Generator(device=dev).manual_seed(0)
    ei_full = powerlaw_graph(N, w["E"], dev, 0)  # every rank builds the same graph, then keeps its shard
    E = ei_full.size(1)
    lo, hi = D.even_ranges(E, world)[rank]
    ei = ei_full[:, lo:hi].contiguous()
    del ei_full
    torch.cuda.empty_cache()
    score = torch.tanh(torch.randn(N, device=dev, generator=g))
    ew_full = torch.rand(E, device=dev, generator=g) + 0.5
    ew = ew_full[lo:hi].clone().requires_grad_(True)
    del ew_full
    node_index = torch.sort(torch.topk(score, N // 2).indices)[0]
    K = node_index.numel()
    k_lo, k_hi = D.even_ranges(K, world)[rank]
    n_lo = int(node_index[k_lo]) if k_hi > k_lo else 0
    n_hi = int(node_index[k_hi - 1]) + 1 if k_hi > k_lo else 0
    x = torch.randn(n_hi - n_lo, F, device=dev, generator=g).requires_grad_(True)  # the rank's node range only
    so = T.SelectOutput(node_index=node_index[k_lo:k_hi] - n_lo, num_nodes=n_hi - n_lo,
                        cluster_index=torch.arange(k_hi - k_lo, device=dev), num_supernodes=k_hi - k_lo,
                        weight=score[node_index[k_lo:k_hi]])
    F_.rows_sorted(ei)
    tot_box = [0, 0]

    def step():
        x.grad = None
        ew.grad = None
        so._b200_csr = None
        xp, _ = T.B200Reduce("sum")(x, so)
        eo, wo, off, tot = D.sharded_kept_node_connect(ei, ew, node_index, N, degree_norm=True, rows_sorted=True)
        torch.autograd.backward([xp, wo], [torch.ones_like(xp), torch.ones_like(wo)])
        tot_box[0], tot_box[1] = tot, eo.size(1)

    for _ in range(3):
        step()
    ctx.barrier()
    n0 = _lib.kernel_launches()
    step()
    torch.cuda.synchronize()
    launches = _lib.kernel_launches() - n0
    run = ctx.long_run(step, target_ms=200.0, lo=5)
    hbm, _, src = peaks()
    alg = sparse_alg_bytes(E, tot_box[0], K, K, N, F, True)
    ms = run["ms_per_step"]
    return {"mode": "eager public API, edge-sharded (tgp_b200.distributed.sharded_kept_node_connect)",
            "ms_per_step": ms, "long_run": run, "value": 1.0 / (ms * 1e-3), "unit": "graphs/s",
            "edges_per_s": E / (ms * 1e-3), "scaling": "strong", "dtype": "f32", "gpu_launches_per_step": launches,
            "shape": {"N": N, "E": E, "K": K, "E_out": tot_box[0], "E_local": hi - lo, "E_out_local": tot_box[1], "F": F},
            "collectives_per_step": {"all_reduce_counts_bytes": 8 * world, "all_reduce_degree_bytes": 4 * K,
                                     "all_reduce_grad_dinv_bytes": 4 * K},
            "roofline": {"bound": "hbm", "achieved": alg / (ms * 1e-3) / 1e9, "peak": hbm * world, "unit": "GB/s",
                         "frac": alg / (ms * 1e-3) / 1e9 / (hbm * world), "traffic": None, "kernel": "whole step",
                         "algorithmic_bytes": alg, "peak_source": f"{src} (MEASURED_PEAKS.json hbm_gbs) x {world} GPUs"},
            "l2_policy": "inputs larger than L2 (126 MB), no flush"}


# --------------------------------------------------------------------------------------------------------------
# CPU reference arm (oracle port: torch_geometric / torch_scatter are not installable offline)
# --------------------------------------------------------------------------------------------------------------
def oracle_dense_step(w, a, s, x):
    """Reference CPU path (restated; PyG unavailable offline): fwd + bwd of the same step."""
    from oracle import ref_path as R

    s = s.clone().requires_grad_(True)
    x = x.clone().requires_grad_(True)
    if w["pooler"] == "mincut":
        xp, ap, loss = R.mincut_pool(x, a, s)
    else:
        xp, ap, loss = R.diff_pool(x, a, s)
    (xp.sum() + ap.sum() + sum(loss.values())).backward()
    return float(sum(v.detach() for v in loss.values()))


def cpu_dense_inputs(w, B, seed):
    g = torch.Generator().manual_seed(seed)
    N, K = w["levels"][0]
    a = (torch.rand(B, N, N, generator=g) < w["p"]).float()
    a = torch.triu(a, 1)
    a = a + a.transpose(1, 2)
    s = torch.softmax(torch.randn(B, N, K, generator=g), -1)
    x = torch.randn(B, N, w["F"], generator=g)
    return a, s, x


def cpu_baseline(w, budget_s=12.0, sample_graphs=32, warmup=1):
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    a, s, x = cpu_dense_inputs(w, sample_graphs, 123)
    for _ in range(warmup):
        oracle_dense_step(w, a, s, x)
    times = []
    t_end = time.perf_counter() + budget_s
    while time.perf_counter() < t_end and len(times) < 30:
        t0 = time.perf_counter()
        oracle_dense_step(w, a, s, x)
        times.append(time.perf_counter() - t0)
    med = statistics.median(times)
    return {"value": sample_graphs / med, "unit": "graphs/s", "cores": cores, "kind": "port",
            "sample": f"{sample_graphs} graphs of the workload shape (level 1), fp32, fwd+bwd, median of {len(times)} "
                      "iterations; reference CPU path restated in oracle/ (PyG unavailable offline)"}


def cpu_sparse_baseline(name, budget_s=4.0):
    """The sparse configs on the host cores: C1 at full size, C4 / C5 on a 1/20 (1/80) scale sample."""
    from oracle import ref_path as R

    w = SPARSE[name]
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    g = torch.Generator().manual_seed(0)
    if w["kind"] == "topk":
        ei, batch, N = er_batch(w, 0)
        units, scale = w["graphs"], 1
    else:
        scale = 20 if name == "c4" else 80
        N = w["N"] // scale
        ei = powerlaw_graph(N, w["E"] // scale, "cpu", 0)
        batch, units = None, 1.0 / scale
    E = ei.size(1)
    x = torch.randn(N, w["F"], generator=g)
    ew = torch.rand(E, generator=g) + 0.5
    if w["kind"] == "cluster":
        cl, K = matching_clusters(N, "cpu", g)
        so = R.OracleSelectOutput(cluster_index=cl, num_supernodes=K)
    else:
        score = torch.tanh(torch.randn(N, generator=g))
        node_index = torch.topk(score, N // 2).indices if batch is None else per_graph_topk(score, batch, "cpu")
        so = R.OracleSelectOutput(node_index=node_index, num_nodes=N, cluster_index=torch.arange(node_index.numel()),
                                  num_supernodes=node_index.numel(), weight=score[node_index])

    def step():
        xx = x.clone().requires_grad_(True)
        ww = ew.clone().requires_grad_(True)
        if w["kind"] == "cluster":
            xp, _ = R.aggr_reduce(xx, so, op="mean")
            eo, wo = R.sparse_connect_so(ei, so, edge_weight=ww)
        else:
            xp, eo, wo, _ = R.topk_pool(xx, ei, ww, so, batch=batch, degree_norm=w["kind"] == "topk_big")
        (xp.sum() + wo.sum()).backward()

    step()
    times = []
    t_end = time.perf_counter() + budget_s
    while time.perf_counter() < t_end and len(times) < 20:
        t0 = time.perf_counter()
        step()
        times.append(time.perf_counter() - t0)
    med = statistics.median(times)
    return {"value": units / med, "unit": "graphs/s", "cores": cores, "kind": "port",
            "sample": (f"full-size batch, median of {len(times)}" if scale == 1 else
                       f"1/{scale}-scale graph (N={N}, E={E}); value = (1/{scale} graph)/time, i.e. assumes linear "
                       f"scaling to the full size; median of {len(times)}")}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    name = args.workload if args.workload in DENSE else "c2"
    w = DENSE[name]
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    sample = min(w["B"], 512)  # the full C2 batch per step (bounded for the larger workloads)
    a, s, x = cpu_dense_inputs(w, sample, 123)
    for _ in range(args.warmup):
        oracle_dense_step(w, a, s, x)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        oracle_dense_step(w, a, s, x)
    dt = (time.perf_counter() - t0) / args.steps
    value = sample / dt
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": "graphs/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt * 1e3,
        "higher_is_better": True, "scaling": w["scaling"], "vs_baseline": None,
        "dtype": "f32", "data": "synthetic", "config": config_of(name, args.gpus),
        "device": "host CPU",
        "cpu_baseline": {"value": value, "unit": "graphs/s", "cores": cores, "kind": "port",
                         "sample": f"{sample} graphs of the workload shape per step, fp32, fwd+bwd; reference CPU path "
                                   "restated in oracle/ (torch_geometric / torch_scatter are not installable offline)"},
        "e2e": {"value": value, "unit": "graphs/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line), flush=True)


def strip(d):
    return {k: v for k, v in d.items() if not k.startswith("_")}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="all", choices=["all"] + sorted(DENSE) + sorted(SPARSE))
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the last timed step's outputs as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "b200" or args.workload in SPARSE):
        ap.error("--dump-outputs writes the outputs of the dense headline step: --impl b200, --workload all, c2 or c3")
    if args.impl == "reference":
        run_reference(args)
        return
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device (the B200 path has no CPU fallback); use --impl reference")
    ctx = Ctx(args)
    world, rank = ctx.world, ctx.rank
    head_name = args.workload if args.workload in DENSE else "c2"
    configs = {}
    line = None
    dump = None

    def attempt(name, fn):
        try:
            configs[name] = strip(fn())
        except Exception as exc:  # a config that cannot run on this launch is reported, never silently dropped
            configs[name] = {"error": f"{type(exc).__name__}: {exc}"[:300]}
        configs[name]["config"] = config_of(name, world)
        torch.cuda.empty_cache()

    if args.workload in ("all",) + tuple(DENSE):
        head = run_dense(ctx, head_name, headline=True)
        e2e = dense_e2e(ctx, head_name) if head_name == "c2" else None
        w = DENSE[head_name]
        line = {
            "metric": METRIC, "value": head["value"], "unit": "graphs/s", "n_gpus": world, "steps": args.steps,
            "warmup": max(args.warmup, 3), "ms_per_step": head["ms_per_step"], "higher_is_better": True,
            "scaling": w["scaling"], "vs_baseline": None, "dtype": w["dtype"], "data": "synthetic",
            "config": config_of(head_name, world),
            "parallelism": f"graph-batch sharding x{world}, no data-path collective",
            "gpu_launches": head["gpu_launches_per_step"] * args.steps,
            "roofline": head["roofline"], "clocks": head["clocks"],
        }
        for k in ("mode", "eager_ms_per_step", "long_run", "gpu_launches_per_step", "kernel_ms_sum", "host_gap_ms",
                  "eager_host_gap_ms", "kernels", "l2_policy", "graphs_per_gpu"):
            line[k] = head[k]
        if e2e is not None:
            line["e2e"] = e2e
        configs[head_name] = {k: v for k, v in strip(head).items() if k not in ("kernels", "clocks")}
        configs[head_name]["config"] = config_of(head_name, world)
        dump = head.get("_dump")
        del head
        torch.cuda.empty_cache()
    if args.workload == "all":
        other_dense = [n for n in DENSE if n != head_name]
        for n in other_dense:
            attempt(n, lambda n=n: run_dense(ctx, n, headline=False))
        if world == 1:
            for n in ("c1", "c4", "c5"):
                attempt(n, lambda n=n: run_sparse(ctx, n))
        else:
            attempt("c5", lambda: run_c5_sharded(ctx))
            for n in ("c1", "c4"):
                configs[n] = {"skipped": "single-GPU config (measured at --gpus 1)", "config": config_of(n, world)}
    elif args.workload in SPARSE:
        if world > 1 and args.workload == "c5":
            res = run_c5_sharded(ctx)
        else:
            res = run_sparse(ctx, args.workload)
        res = strip(res)
        line = {"metric": METRIC, "value": res["value"], "unit": "graphs/s", "n_gpus": world, "steps": res["long_run"]["steps"],
                "warmup": max(args.warmup, 3), "ms_per_step": res["ms_per_step"], "higher_is_better": True,
                "scaling": res.get("scaling", "weak"), "vs_baseline": None, "dtype": "f32", "data": "synthetic",
                "config": config_of(args.workload, world),
                "gpu_launches": res["gpu_launches_per_step"] * res["long_run"]["steps"], "roofline": res["roofline"]}
        line.update({k: v for k, v in res.items() if k not in line})
    if rank == 0:
        if configs:
            if not args.no_cpu_baseline and world == 1:
                for n in ("c1", "c4", "c5"):
                    if n in configs and "error" not in configs[n]:
                        configs[n]["cpu_baseline"] = cpu_sparse_baseline(n)
            line["configs"] = configs
        if not args.no_cpu_baseline and world == 1 and args.workload in ("all",) + tuple(DENSE):
            line["cpu_baseline"] = cpu_baseline(DENSE[head_name])
        print(json.dumps(line), flush=True)
        if dump is not None:
            import numpy as np

            os.makedirs(args.dump_outputs, exist_ok=True)
            for name, t in dump.items():
                np.save(os.path.join(args.dump_outputs, f"{name}.npy"), t.cpu().numpy())
    if ctx.dist is not None:
        ctx.dist.barrier()
        ctx.dist.destroy_process_group()


if __name__ == "__main__":
    main()
