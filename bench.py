#!/usr/bin/env python
"""bench.py -- SGC-LL train throughput (graphs/s) on N B200s, one JSON line on rank 0.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

The result line goes to stdout without the per-kernel tables and descriptions; the full record follows on stderr as
one JSON line.  K is the number of timed steps of `value`.  --dump-outputs DIR writes what the last of them computed
(loss, gradients, parameters after Adam) as DIR/*.npy.

Headline workload (BASELINE.json configs[1], SURVEY.md section 8d "C2"): ToxCast-shape synthetic molecules,
B = 1024 graphs per GPU (weak scaling), Nmax = 132, 75 atom features, 617 tasks, K = 3, through the SimpleAGCN
stack (4 SGC_LL layers 75-64-128-128-64 + DenseMol 256 + GraphGather + 617 two-class heads), forward + backward +
gradient all-reduce + Adam.  One "step" = one such pass over one batch.

  value    graphs/s with the batch resident in HBM: the step (one agcn_stack_loss_grad call + all-reduce +
           agcn_adam_step) captured in a CUDA graph and replayed; CUDA events, max over ranks, L2 flushed between
           the timed steps
  e2e      graphs/s through the public API from pinned HOST buffers in the reference's zero-padded wire layout
           (graph_topology.py:84-98): every step builds its topology plan, the pack kernels read the pinned arrays
           in place (only the real rows cross PCIe) on a side stream while the previous step computes, the step
           runs eagerly, and its loss is read back to the host.  At every N.
  roofline the kernels of one layer forward (layer 3) timed live with CUDA events on their streams, each against its
           own algorithmic bytes / flops and MEASURED_PEAKS.json; the top-level entry is the slowest of them;
           `kernels` is the per-kernel table of one eager step
  configs  the other BASELINE.json shapes, each with its own graphs/s, e2e, kernel table and CPU baseline:
           C1 Tox21 (B = 256, 12 tasks), C3 ModelNet40 (B = 32 x 1024 points, 40 classes), C4 Sydney (ragged)
  cpu_baseline / --impl reference: the reference's algorithm as written (oracle port: per-graph Python loop with
           the interpreted O(n^2) metric block, autograd for the rest) on the host cores, on a bounded sample of
           the same workload; `cpu_vectorised` = the batched all-core torch restatement (BASELINE.md section 4).
"""
import argparse
import gc
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

FILTERS = (64, 128, 128, 64)
K_ORDER, FINAL = 3, 256
WORKLOADS = {
    "C1": dict(key="C1", gen="molecules", B=256, Nmax=132, F=75, n_tasks=12, loss="sigmoid_ce", seed=1234,
               name="C1 Tox21-shape synthetic molecules: B=256/GPU, Nmax=132, F=75, 12 tasks, K=3, SimpleAGCN "
                    "(4xSGC_LL 64-128-128-64 + DenseMol256 + Gather + heads), fwd+bwd+allreduce+Adam"),
    "C2": dict(key="C2", gen="molecules", B=1024, Nmax=132, F=75, n_tasks=617, loss="sigmoid_ce", seed=1235,
               name="C2 ToxCast-shape synthetic molecules: B=1024/GPU, Nmax=132, F=75, 617 tasks, K=3, SimpleAGCN "
                    "(4xSGC_LL 64-128-128-64 + DenseMol256 + Gather + heads), fwd+bwd+allreduce+Adam"),
    "C3": dict(key="C3", gen="modelnet", B=32, Nmax=1024, F=3, n_tasks=40, loss="softmax_ce", seed=1236,
               adj_rule="mean_distance",
               name="C3 ModelNet40-shape synthetic point clouds: B=32/GPU, N=1024 points, xyz, 40 classes, K=3, "
                    "SimpleAGCN stack (4xSGC_LL 64-128-128-64 + DenseMol256 + Gather + softmax head), "
                    "fwd+bwd+allreduce+Adam"),
    "C4": dict(key="C4", gen="sydney", B=128, Nmax=1024, F=4, n_tasks=26, loss="softmax_ce", seed=1237,
               adj_rule="cutoff",
               name="C4 Sydney-Urban-Objects-shape ragged point clouds: B=128/GPU, n~loguniform[13,1024] padded to "
                    "1024, xyz+intensity, 26 classes, K=3, SimpleAGCN stack, fwd+bwd+allreduce+Adam"),
}
WORKLOAD = WORKLOADS["C2"]["name"]


def load_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        p = json.load(open(path))
        return {"hbm_gbs": p["hbm_gbs"], "bf16_tflops": p["bf16_tflops"], "source": "measured"}
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "source": "fallback"}


class ClockSampler(object):
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""

    def __init__(self, index):
        self.index = index
        self.lines = []
        self.proc = None

    def start(self):
        q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + q,
                                          "--format=csv,noheader,nounits", "-lms", "100"], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._pump, daemon=True).start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def wait_first(self, timeout_s):
        t_end = time.time() + timeout_s
        while self.proc is not None and not self.lines and time.time() < t_end:
            time.sleep(0.02)

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for line in self.lines:
            parts = [p.strip() for p in line.split(",")]
            if len(parts) < 6:
                continue
            try:
                sm.append(float(parts[0])); mx.append(float(parts[1]))
            except ValueError:
                continue
            for name, val in zip(names, parts[2:6]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


# ------------------------------------------------------------------------------------------------
# workloads
# ------------------------------------------------------------------------------------------------
def make_inputs(cfg, rank, B=None):
    """Padded wire-layout batch of one rank (numpy) + labels: X [B,Nmax,F], L [B,Nmax,Nmax], n_nodes, targets, weights."""
    import numpy as np
    from agcn_b200 import synthetic
    B = B or cfg["B"]
    seed = cfg["seed"] + rank
    if cfg["gen"] == "molecules":
        X, L, n = synthetic.molecule_batch(B, cfg["Nmax"], seed=seed)
    elif cfg["gen"] == "modelnet":
        X, L, n = synthetic.modelnet_like_batch(B, cfg["Nmax"], seed=seed)
    elif cfg["gen"] == "sydney":
        X, L, n = synthetic.sydney_like_batch(B, cfg["Nmax"], seed=seed)
    else:
        raise ValueError(cfg["gen"])
    rng = np.random.default_rng(99 + rank)
    T = cfg["n_tasks"]
    if cfg["loss"] == "softmax_ce":
        tg = np.zeros((B, T), np.float32)
        tg[np.arange(B), rng.integers(0, T, B)] = 1.0
        w = np.ones(B, np.float32)
    else:
        y = rng.random((B, T)) < 0.1
        tg = np.zeros((B, T, 2), np.float32)
        tg[..., 0] = ~y
        tg[..., 1] = y
        tg = tg.reshape(B, 2 * T)
        w = np.ones((B, 2 * T), np.float32)
    return X, L, n, tg, w


def step_algorithmic(n_nodes, F0, filters, K, paper):
    """Algorithmic FLOPs and bytes of one fwd+bwd pass of the SGC_LL layers over a batch (SURVEY.md section 8d)."""
    import numpy as np
    n = n_nodes.astype(np.float64)
    dims = [F0] + list(filters)
    flops = bytes_ = 0.0
    for i in range(len(filters)):
        F, Fo = dims[i], dims[i + 1]
        f_fwd = 2 * K * n * n * F + 2 * n * K * F * Fo - (2 * n * n * F if not paper else 0)   # no Gram in literal mode
        f_bwd = 4 * n * K * F * Fo + 4 * (K - 1) * n * n * F
        if paper:
            f_fwd = f_fwd + 2 * n * F * F
            f_bwd = f_bwd + 2 * n * n * F + 4 * n * F * F
        flops += (f_fwd + f_bwd).sum()
        bytes_ += (4 * (n * F + n * n + n * Fo) + 4 * (2 * n * F + n * n + n * Fo)).sum()
    return flops, bytes_


# ------------------------------------------------------------------------------------------------
# CPU arms
# ------------------------------------------------------------------------------------------------
def _cpu_literal_worker(args):
    """Forward + backward of the SimpleAGCN stack over a shard of graphs with the oracle port of the reference as
    written (interpreted metric block in every layer's forward, graphconv.py:163-211)."""
    import numpy as np
    import torch
    from oracle import sgcll_oracle as O
    X, L, n_nodes, F0, Nt, seed = args
    torch.set_num_threads(1)
    dims = [F0] + list(FILTERS)
    params = [{k: v.requires_grad_(True) for k, v in O.make_params(dims[i], dims[i + 1], K_ORDER, "SGC_LL", seed=seed + i,
                                                                    dtype=torch.float32, perturb=False).items()}
              for i in range(4)]
    g = torch.Generator().manual_seed(seed)
    dW = (torch.rand(FILTERS[-1], FINAL, generator=g) * 0.2 - 0.1).requires_grad_(True)
    hW = (torch.randn(FINAL, Nt, generator=g) * 0.01).requires_grad_(True)
    loss = torch.zeros(())
    for b in range(len(n_nodes)):
        n = int(n_nodes[b])
        x = torch.from_numpy(X[b, :n])
        Lg = torch.from_numpy(L[b, :n, :n])
        for i in range(4):
            with torch.no_grad():
                O.metric_block_literal(x.detach().numpy(), params[i]["M_L"].detach().numpy())
            y, _, _, _ = O.sgc_ll_graph(x, Lg, params[i], K_ORDER, "SGC_LL", "reference_literal", "reference",
                                        compute_similarity=False)
            x = torch.relu(y)
        mol = torch.tanh((x @ dW).sum(0))
        logits = mol @ hW
        loss = loss + torch.nn.functional.binary_cross_entropy_with_logits(logits, torch.zeros_like(logits),
                                                                           reduction='sum')
    loss.backward()
    return float(loss.detach())


def cpu_literal(cfg, n_graphs, steps, warmup, procs):
    """graphs/s of the reference-as-written port on `procs` host processes (one core each)."""
    import multiprocessing as mp
    X, L, n_nodes, _, _ = make_inputs(cfg, 0, B=n_graphs + 1)
    X, L, n_nodes = X[1:], L[1:], n_nodes[1:]          # drop the forced maximum-size sample of slot 0
    Nt = cfg["n_tasks"] * (2 if cfg["loss"] == "sigmoid_ce" else 1)
    shards = [(X[i::procs], L[i::procs], n_nodes[i::procs], cfg["F"], Nt, 7) for i in range(procs)]
    ctx = mp.get_context("fork")
    times = []
    with ctx.Pool(procs) as pool:
        for it in range(warmup + steps):
            t0 = time.perf_counter()
            pool.map(_cpu_literal_worker, shards)
            if it >= warmup:
                times.append(time.perf_counter() - t0)
    total = sum(times)
    return n_graphs * len(times) / total, total / len(times) * 1e3, float(n_nodes.mean())


def cpu_vectorised(cfg, n_graphs, steps, warmup, paper):
    """graphs/s of the batched all-core torch restatement (oracle/vectorised_baseline.py): fwd + bwd + the same loss."""
    import numpy as np
    import torch
    from oracle import vectorised_baseline as VB
    threads = os.cpu_count() or 1
    torch.set_num_threads(threads)
    X, L, n, tg, w = make_inputs(cfg, 0, B=n_graphs)
    Nt = tg.shape[1]
    layers, head = VB.make_params([cfg["F"]] + list(FILTERS), K_ORDER, FINAL, Nt, seed=3)
    buckets = VB.prepare_buckets(X, L, n, tg, w)
    mode = ("paper", "full") if paper else ("reference_literal", "reference")
    times = []
    for it in range(warmup + steps):
        t0 = time.perf_counter()
        loss = VB.simple_agcn_loss(buckets, layers, head, K_ORDER, n_graphs, mode[0], mode[1], cfg["loss"])
        loss.backward()
        if it >= warmup:
            times.append(time.perf_counter() - t0)
    times.sort()
    med = times[len(times) // 2]
    return n_graphs / med, med * 1e3, threads, float(np.asarray(n).mean())


def run_reference(args):
    """--impl reference: the reference's own CPU implementation of the path (oracle port, all host cores) on OUR
    arm's config.  Rank 0 alone runs; the other ranks exit without work."""
    if int(os.environ.get("RANK", "0")) != 0:
        return
    cfg = WORKLOADS[args.workload]
    cores = os.cpu_count() or 1
    world = args.gpus
    if args.cpu_kind == "vectorised":
        n_graphs = args.ref_graphs or cfg["B"]
        steps, warmup = max(1, args.steps), max(0, args.warmup)
        gps, ms, procs, nbar = cpu_vectorised(cfg, n_graphs, steps, warmup, args.paper)
        kind = "port"
        sample = ("%d graphs/step of the %s workload (mean n=%.1f), %d step(s), batched torch restatement "
                  "(oracle/vectorised_baseline.py, %s semantics), %d threads"
                  % (n_graphs, cfg["key"], nbar, steps, "paper/full" if args.paper else "reference_literal", procs))
    else:
        procs = max(1, min(cores, 32))
        n_graphs = args.ref_graphs or min(cfg["B"], 1024)
        if cfg["gen"] != "molecules":
            n_graphs = args.ref_graphs or 2 * procs      # the interpreted O(n^2) block needs seconds per 1024-point cloud
        steps, warmup = max(1, args.steps), max(0, min(args.warmup, 2))
        # keep the whole run within a few minutes whatever K/W the driver passes
        est = 1.0 * n_graphs / 1200.0 if cfg["gen"] == "molecules" else 30.0
        steps = max(1, min(steps, int(150.0 / max(est, 1e-3))))
        gps, ms, nbar = cpu_literal(cfg, n_graphs, steps, warmup, procs)
        kind = "port"
        sample = ("%d graphs/step of the %s workload (mean n=%.1f), %d step(s), reference-as-written port "
                  "(interpreted metric block + autograd), %d processes" % (n_graphs, cfg["key"], nbar, steps, procs))
    line = {"impl": "reference", "metric": "sgc_ll_train_graphs_per_s", "value": gps, "unit": "graphs/s",
            "n_gpus": world, "steps": steps, "warmup": warmup, "ms_per_step": ms, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": bench_config(cfg, world),
            "cpu_baseline": {"value": gps, "unit": "graphs/s", "cores": procs, "kind": kind, "sample": sample},
            "e2e": {"value": gps, "unit": "graphs/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line))


def bench_config(cfg, world):
    """The `config` object of the JSON line: identical for both arms."""
    return {"workload": cfg["name"], "global_batch": world * cfg["B"], "parallelism": "dp%d" % world,
            "semantics": "laplacian=reference_literal, metric_grad=reference",
            "l2": "flushed between timed steps (256 MB fill)",
            "host_layout_e2e": "reference wire layout: zero-padded [B,Nmax,F] + [B,Nmax,Nmax] (pinned)"}


def cpu_leg(cfg, kind, steps, warmup, paper=False, graphs=0):
    """A CPU arm in a fresh interpreter (fork pools / thread settings must not meet CUDA)."""
    cmd = [sys.executable, os.path.abspath(__file__), "--impl", "reference", "--workload", cfg["key"], "--cpu-kind", kind,
           "--steps", str(steps), "--warmup", str(warmup)]
    if paper:
        cmd.append("--paper")
    if graphs:
        cmd += ["--ref-graphs", str(graphs)]
    try:
        out = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, timeout=400,
                             env=dict(os.environ, RANK="0", WORLD_SIZE="1"))
        ref = json.loads(out.stdout.strip().splitlines()[-1])
        return dict(ref["cpu_baseline"], ms_per_step=ref["ms_per_step"])
    except Exception as exc:
        return {"value": None, "unit": "graphs/s", "cores": 0, "kind": "port", "sample": "failed: %s" % str(exc)[:160]}


# ------------------------------------------------------------------------------------------------
# GPU arm
# ------------------------------------------------------------------------------------------------
class Runner(object):
    """One workload on this rank: host buffers, model, resident tensors, and the measurements."""

    def __init__(self, cfg, dev, rank, world, laplacian="reference_literal", metric_grad="reference", overlap=True):
        import torch
        import agcn_b200
        from agcn_b200.simple_agcn import SimpleAGCNStep
        self.torch, self.agcn = torch, agcn_b200
        self.cfg, self.dev, self.rank, self.world = cfg, dev, rank, world
        import numpy as np
        X, L, n, tg, w = make_inputs(cfg, rank)
        self.n_nodes = n
        self.B = cfg["B"]
        # the reference's wire layout (graph_topology.py:84-98), pinned
        self.Xpad_h, self.Lpad_h = torch.from_numpy(X).pin_memory(), torch.from_numpy(L).pin_memory()
        self.tg_h, self.w_h = torch.from_numpy(tg).pin_memory(), torch.from_numpy(w).pin_memory()
        # labels as the reference feeds them (multitask_classifier.py:147-152,171-185: bool [B, T] labels + float [B, T]
        # weights; the one-hot encoding happens inside the graph, :196-199): the e2e path copies these and expands
        # them on the device
        if cfg["loss"] == "sigmoid_ce":
            self.y_h = torch.from_numpy(np.ascontiguousarray(tg.reshape(self.B, -1, 2)[..., 1]).astype(np.uint8)).pin_memory()
            self.wc_h = torch.from_numpy(np.ascontiguousarray(w.reshape(self.B, -1, 2)[..., 0])).pin_memory()
        else:
            self.y_h = torch.from_numpy(tg.argmax(1).astype(np.int64)).pin_memory()
            self.wc_h = self.w_h
        self.model = SimpleAGCNStep(cfg["F"], FILTERS, FINAL, cfg["n_tasks"], K_ORDER, self.B, device=dev,
                                    world_size=world, laplacian=laplacian, metric_grad=metric_grad, loss=cfg["loss"],
                                    overlap_allreduce=overlap)
        self.batch = agcn_b200.GraphBatch(n, cfg["Nmax"], device=dev)
        self.Xd, self.Ld = self.batch.pack_nodes(self.Xpad_h), self.batch.pack_lap(self.Lpad_h)
        self.tg_d, self.w_d = self.tg_h.to(dev), self.w_h.to(dev)
        self.flush = torch.empty(256 * 1024 * 1024 // 4, dtype=torch.float32, device=dev)   # > 126 MB L2
        self.graph = None
        torch.cuda.synchronize()

    # ---- helpers
    def barrier(self):
        import torch.distributed as dist
        self.torch.cuda.synchronize()
        if self.world > 1:
            dist.barrier()
        self.torch.cuda.synchronize()

    def max_over_ranks(self, ms):
        import torch.distributed as dist
        t = self.torch.tensor([ms], device=self.dev, dtype=self.torch.float64)
        if self.world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t)

    def resident_step(self):
        self.loss = self.model.step(self.Xd, self.Ld, self.batch, self.tg_d, self.w_d)   # (a replayed graph rewrites it)
        return self.loss

    def timed(self, fn, steps, warmup):
        torch = self.torch
        for _ in range(warmup):
            fn()
        self.barrier()
        evs = []
        for _ in range(steps):
            self.flush.fill_(1.0)                              # evict L2 between timed steps (not timed)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            fn()
            e1.record()
            evs.append((e0, e1))
        self.barrier()
        return self.max_over_ranks(sum(a.elapsed_time(b) for a, b in evs)) / steps

    def capture(self):
        """The resident step as a CUDA graph (the step is ~60 small launches: replay removes the host launch path)."""
        torch = self.torch
        try:
            side = torch.cuda.Stream(device=self.dev)
            side.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(side):
                for _ in range(3):
                    self.resident_step()
            torch.cuda.current_stream().wait_stream(side)
            torch.cuda.synchronize()
            graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(graph):
                self.resident_step()
            self.graph = graph
            return "cuda_graph"
        except Exception as exc:
            self.graph = None
            torch.cuda.synchronize()
            return "eager (graph capture failed: %s)" % str(exc)[:120]

    def replay(self):
        self.graph.replay()

    def release(self):
        self.graph = None
        gc.collect()
        self.torch.cuda.synchronize()

    # ---- end to end
    def timed_e2e(self, steps, warmup, mode="zero_copy"):
        """Every step: plan of the batch, the padded pinned host arrays taken in, train step, loss back on the host.
        mode "zero_copy": the pack kernels read the pinned arrays in place (only real rows cross PCIe), packing of
        step i+1 on a side stream while step i computes, the loss of step i read after step i+1 is queued.
        mode "copy_engine": the padded arrays are staged through the copy engine first (same overlap).
        mode "serial": zero-copy, but pack, step and loss read strictly one after the other.
        mode "points" (point clouds): the host hands over the coordinates only; the threshold adjacency and the
        Laplacian (meshloader.py:264-285 / pointcloudloader.py:240-263 + graph_structure.py:85-130) are built on the
        device by agcn_point_laplacian inside the timed step."""
        torch, agcn = self.torch, self.agcn
        dev, model = self.dev, self.model
        torch.cuda.synchronize()
        # ingestion of the next batch runs beside the current step: the step's stream gets the higher priority so that
        # its kernels are scheduled ahead of the pack kernels' PCIe-stalled warps
        side = torch.cuda.Stream(device=dev, priority=0)
        main = torch.cuda.Stream(device=dev, priority=-1)
        # eager launches: ONE all-reduce of the flat gradient buffer after backward.  The bucketed all-reduce under the
        # backward pass pays off inside the replayed CUDA graph; launched eagerly, five c10d calls per step cost more host
        # time than the overlap saves (2 x B200, C2: 1.13 ms per step bucketed, 0.94 ms with one all-reduce)
        keep = model.overlap_allreduce
        model.overlap_allreduce = False
        try:
            with torch.cuda.stream(main):
                return self._timed_e2e(steps, warmup, mode, side, main)
        finally:
            model.overlap_allreduce = keep

    def _timed_e2e(self, steps, warmup, mode, side, main):
        torch, agcn = self.torch, self.agcn
        dev, model = self.dev, self.model
        loss_host = [torch.empty(1).pin_memory() for _ in range(2)]
        lab = [(torch.empty_like(self.tg_h, device=dev), torch.empty_like(self.w_h, device=dev)) for _ in range(2)]
        stage_bufs = None
        if mode == "copy_engine":
            stage_bufs = [(torch.empty_like(self.Xpad_h, device=dev), torch.empty_like(self.Lpad_h, device=dev))
                          for _ in range(2)]
        ready = [torch.cuda.Event() for _ in range(2)]
        consumed = [torch.cuda.Event() for _ in range(2)]

        def stage(i):
            slot = i % 2
            with torch.cuda.stream(side):
                side.wait_event(consumed[slot])
                b = agcn.GraphBatch(self.n_nodes, self.cfg["Nmax"], device=dev)
                if mode == "points":
                    # only the coordinates cross PCIe; adjacency + Laplacian are built on the device
                    X = b.pack_nodes(self.Xpad_h)
                    L = b.point_laplacians(X, rule=self.cfg["adj_rule"])
                elif stage_bufs is not None:
                    stage_bufs[slot][0].copy_(self.Xpad_h, non_blocking=True)
                    stage_bufs[slot][1].copy_(self.Lpad_h, non_blocking=True)
                    X, L = b.pack_nodes(stage_bufs[slot][0]), b.pack_lap(stage_bufs[slot][1])
                else:
                    X, L = b.pack_nodes(self.Xpad_h), b.pack_lap(self.Lpad_h)     # zero-copy reads of pinned memory
                self.labels_to_device(lab[slot])
                ready[slot].record(side)
            X.record_stream(main)
            L.record_stream(main)
            return b, X, L

        def run_pipelined(n_steps):
            losses, pending = [], None
            nxt = stage(0)
            for i in range(n_steps):
                cur = nxt
                if i + 1 < n_steps:
                    nxt = stage(i + 1)
                slot = i % 2
                main.wait_event(ready[slot])
                b, X, L = cur
                loss = model.step(X, L, b, lab[slot][0], lab[slot][1])
                host = loss_host[slot]
                host.copy_(loss, non_blocking=True)
                consumed[slot].record(main)
                done = torch.cuda.Event()
                done.record(main)
                if pending is not None:
                    pending[1].synchronize()
                    losses.append(float(pending[0]))
                pending = (host, done)
            pending[1].synchronize()
            losses.append(float(pending[0]))
            return losses

        def run_serial(n_steps):
            losses = []
            for i in range(n_steps):
                b = agcn.GraphBatch(self.n_nodes, self.cfg["Nmax"], device=dev)
                X, L = b.pack_nodes(self.Xpad_h), b.pack_lap(self.Lpad_h)
                self.labels_to_device(lab[0])
                losses.append(float(model.step(X, L, b, lab[0][0], lab[0][1])))   # device -> host read of the loss
            return losses

        def run_graphed(n_steps):
            """mode "graph": batch i+1 is staged by a feeder thread (plan, zero-copy pack, labels on the side stream) while
            the main thread captures step i, updates the executable graph of step i-1 in place and launches it."""
            import queue
            q, err = queue.Queue(maxsize=1), []

            def feeder():
                try:
                    torch.cuda.set_device(dev)
                    for i in range(n_steps):
                        q.put(stage(i))
                except BaseException as exc:      # surfaces in the main thread
                    err.append(exc)
                    q.put(None)

            th = threading.Thread(target=feeder, daemon=True)
            th.start()
            losses, pending = [], None
            for i in range(n_steps):
                cur = q.get()
                if cur is None:
                    raise err[0]
                slot = i % 2
                main.wait_event(ready[slot])
                b, X, L = cur
                loss = model.step_graphed(X, L, b, lab[slot][0], lab[slot][1])
                host = loss_host[slot]
                host.copy_(loss, non_blocking=True)
                consumed[slot].record(main)
                done = torch.cuda.Event()
                done.record(main)
                if pending is not None:
                    pending[1].synchronize()
                    losses.append(float(pending[0]))
                pending = (host, done)
            pending[1].synchronize()
            losses.append(float(pending[0]))
            th.join()
            return losses

        run = run_serial if mode == "serial" else (run_graphed if mode == "graph" else run_pipelined)
        for ev in consumed:
            ev.record(main)
        run(warmup)
        self.barrier()
        self.flush.fill_(1.0)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(main)
        losses = run(steps)
        e1.record(main)
        self.barrier()
        import numpy as np
        assert len(losses) == steps and all(np.isfinite(losses))
        return self.max_over_ranks(e0.elapsed_time(e1)) / steps

    def labels_to_device(self, dst):
        """Compact host labels -> the one-hot targets / per-logit weights the loss kernel reads (current stream)."""
        torch = self.torch
        if self.cfg["loss"] == "sigmoid_ce":
            # one kernel reads the pinned labels / weights in place and writes tf.one_hot(label, 2) + per-logit weights
            from agcn_b200.simple_agcn import expand_labels
            expand_labels(self.y_h, self.wc_h, dst[0], dst[1])
        else:
            y = self.y_h.to(self.dev, non_blocking=True)
            dst[0].zero_()
            dst[0].scatter_(1, y.unsqueeze(1), 1.0)
            dst[1].copy_(self.wc_h, non_blocking=True)

    def label_bytes(self):
        return int(self.y_h.numel() * self.y_h.element_size() + self.wc_h.numel() * 4)

    def h2d_bytes(self, zero_copy):
        side = self.label_bytes() + self.n_nodes.nbytes * 8
        if zero_copy:      # the real rows the pack kernels read over PCIe (sector granularity adds a little)
            return int(self.batch.total_nodes * self.cfg["F"] * 4 + self.batch.total_lap * 4 + side)
        return int(self.Xpad_h.numel() * 4 + self.Lpad_h.numel() * 4 + side)

    # ---- per-kernel table of one eager step
    def kernel_table(self, steps=3):
        from agcn_b200 import _lib
        torch = self.torch
        for _ in range(2):
            self.resident_step()
        torch.cuda.synchronize()
        _lib.profile_enable(True)
        t_total = 0.0
        for _ in range(steps):
            self.flush.fill_(1.0)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            self.resident_step()
            e1.record()
            torch.cuda.synchronize()
            t_total += e0.elapsed_time(e1)
        table = _lib.profile_read()
        _lib.profile_enable(False)
        out = {k: {"launches_per_step": n / float(steps), "ms_per_step": ms / steps} for k, (n, ms) in table.items()}
        return dict(sorted(out.items(), key=lambda kv: -kv[1]["ms_per_step"])), t_total / steps


def measure_peaks(dev):
    """TF32-dense (cuBLAS, torch.matmul with allow_tf32) and fp32-FMA (own probe kernel) peaks, measured in this run:
    MEASURED_PEAKS.json records only HBM and bf16 (SURVEY.md section 8d asks for these two)."""
    import ctypes
    import torch
    from agcn_b200 import _lib
    out = {}
    try:
        old = torch.backends.cuda.matmul.allow_tf32
        torch.backends.cuda.matmul.allow_tf32 = True
        a = torch.randn(8192, 8192, device=dev)
        b = torch.randn(8192, 8192, device=dev)
        best = 1e9
        for i in range(6):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            torch.matmul(a, b)
            e1.record()
            torch.cuda.synchronize()
            if i:
                best = min(best, e0.elapsed_time(e1))
        torch.backends.cuda.matmul.allow_tf32 = old
        out["tf32_tflops"] = 2 * 8192.0 ** 3 / (best * 1e-3) / 1e12
        del a, b
    except Exception as exc:
        out["tf32_error"] = str(exc)[:100]
    try:
        sink = torch.zeros(148 * 8 * 256, device=dev)
        iters = 1 << 14
        best = 1e9
        for i in range(4):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            _lib.check(_lib.lib().agcn_probe_fp32_fma(ctypes.c_void_p(sink.data_ptr()), iters,
                                                      ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)))
            e1.record()
            torch.cuda.synchronize()
            if i:
                best = min(best, e0.elapsed_time(e1))
        out["fp32_fma_tflops"] = 148 * 8 * 256 * 8.0 * 2 * iters / (best * 1e-3) / 1e12
    except Exception as exc:
        out["fp32_error"] = str(exc)[:100]
    out["how"] = ("tf32: torch.matmul 8192^3 with allow_tf32 (cuBLAS), best of 5; fp32: 148x8 CTAs x 256 threads x 8 "
                  "independent FMA chains (agcn_probe_fp32_fma), best of 3; CUDA events")
    return out


def layer3_roofline(r, peaks, tf32_peak):
    """Kernels of one layer forward (layer 3: 128 -> 128, K = 3) over this batch, each timed alone with the L2 flushed
    before the layer, CUDA events on the launching streams recorded by the library (agcn_profile_*).  Every kernel gets
    ITS OWN algorithmic bytes / flops (DESIGN.md section 4); `roofline` is the one that takes longest, `layer` the
    SURVEY section 8d figure of the whole layer forward over the sum of its kernels."""
    import torch
    from agcn_b200 import _lib
    from agcn_b200.functional import sgc_ll_packed
    import numpy as np
    layer = r.model.layers[2]
    F, Fo, K = layer.n_atom_feature, layer.nb_filter, layer.K
    X = torch.relu(torch.randn(r.batch.total_nodes, F, device=r.dev))
    cfg = layer._cfg('relu')
    p = {k: v.detach() for k, v in layer.vars.items()}
    with torch.no_grad():
        for it in range(13):
            r.flush.fill_(0.0)
            if it == 3:
                torch.cuda.synchronize()
                _lib.profile_enable(True)
            sgc_ll_packed(X, r.Ld, None, p, r.batch, cfg)
        torch.cuda.synchronize()
        table = _lib.profile_read()
        _lib.profile_enable(False)
    n = r.n_nodes.astype(np.float64)
    R, LL = float(n.sum()), float((n * n).sum())
    small, mid = n[n <= 64], n[(n > 64) & (n <= 144)]
    if not table:
        return {"bound": "hbm", "kernel": None, "achieved": None, "peak": peaks["hbm_gbs"], "unit": "GB/s", "frac": None,
                "traffic": None, "note": "no profiled launch"}
    # algorithmic work of each kernel of the layer forward
    work = {
        # recurrences of the tiled graphs: read X and L once, write T_1 .. T_{K-1}
        "ct::cheb_tile_fwd_kernel": {"bytes": 4.0 * (K * small.sum() * F + (small * small).sum()),
                                     "flops": 2.0 * (K - 1) * (small * small).sum() * F},
        "ct::cheb_tile_fwd_kernel(mid)": {"bytes": 4.0 * (K * mid.sum() * F + (mid * mid).sum()),
                                          "flops": 2.0 * (K - 1) * (mid * mid).sum() * F},
        # contraction over every packed row: read T_0 .. T_{K-1}, the weights once, write Y
        "pt::rows_gemm_kernel(fwd)": {"bytes": 4.0 * (K * R * F + R * Fo + K * F * Fo + Fo), "flops": 2.0 * R * K * F * Fo},
        "pt::pre_tile_kernel(fwd)": {"bytes": 4.0 * (K * R * F + R * Fo + K * F * Fo + Fo), "flops": 2.0 * R * K * F * Fo},
        # one Chebyshev product L T over the graphs above 144 nodes (point clouds)
        "bt::grouped_tc_kernel": {"bytes": 4.0 * (LL + 2 * R * F), "flops": 2.0 * LL * F},
        "bt::grouped_tcu_kernel": {"bytes": 4.0 * (LL + 2 * R * F), "flops": 2.0 * LL * F},
    }
    rows = {}
    for k, v in table.items():
        per = v[1] / v[0]
        row = {"launches": v[0], "ms_per_launch": per}
        if k in work:
            w = work[k]
            row.update({"algorithmic_bytes_per_launch": w["bytes"], "achieved_gbs": w["bytes"] / (per * 1e-3) / 1e9,
                        "hbm_frac": w["bytes"] / (per * 1e-3) / 1e9 / peaks["hbm_gbs"],
                        "algorithmic_flops_per_launch": w["flops"], "achieved_tflops": w["flops"] / (per * 1e-3) / 1e12,
                        "tensor_frac": w["flops"] / (per * 1e-3) / 1e12 / tf32_peak})
        rows[k] = row
    name, (launches, ms) = max(table.items(), key=lambda kv: kv[1][1] / kv[1][0])
    per = ms / launches
    traffic, traffic_src = None, None
    tpath = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(tpath):
        t = json.load(open(tpath))
        traffic, traffic_src = t.get(name + "/" + r.cfg["key"]), t.get("source")
    # the layer as a whole: SURVEY section 8d bytes / flops over the chain recurrences -> contraction
    chain = sum(v["ms_per_launch"] for k, v in rows.items() if "(mid)" not in k)
    layer_bytes = 4.0 * (R * F + LL + R * Fo) + 4.0 * (K * F * Fo + Fo)
    layer_flops = 2.0 * (K - 1) * LL * F + 2.0 * R * K * F * Fo
    layer_row = {"algorithmic_bytes": layer_bytes, "algorithmic_flops": layer_flops, "ms_chain": chain,
                 "achieved_gbs": layer_bytes / (chain * 1e-3) / 1e9, "hbm_frac": layer_bytes / (chain * 1e-3) / 1e9 / peaks["hbm_gbs"],
                 "achieved_tflops": layer_flops / (chain * 1e-3) / 1e12,
                 "tensor_frac": layer_flops / (chain * 1e-3) / 1e12 / tf32_peak,
                 "note": "layer 3 forward (F=128 -> Fo=128, K=3): SURVEY section 8d work over the sum of its kernels "
                         "(mid-size graphs run beside the tiles)"}
    w = work.get(name)
    if w is not None and (name.startswith("bt::grouped_tc") or w["flops"] / max(w["bytes"], 1.0) > tf32_peak * 1e12 / (peaks["hbm_gbs"] * 1e9)):
        ach = w["flops"] / (per * 1e-3) / 1e12
        return {"bound": "tensor", "kernel": name + ", layer 3 forward, whole-batch launch", "achieved": ach,
                "peak": tf32_peak, "unit": "TFLOP/s", "frac": ach / tf32_peak, "traffic": traffic,
                "traffic_source": traffic_src, "algorithmic_flops_per_launch": w["flops"],
                "algorithmic_bytes_per_launch": w["bytes"], "ms_per_launch": per, "launches_timed": launches,
                "peak_source": "tf32 dense measured in this run (cuBLAS); the kernel issues 3x these flops (3xTF32)",
                "kernels_of_the_layer_forward": rows, "layer": layer_row}
    bytes_k = w["bytes"] if w else layer_bytes
    achieved = bytes_k / (per * 1e-3) / 1e9
    return {"bound": "hbm", "kernel": name + ", layer 3 forward (F=128 -> Fo=128, K=3), whole-batch launch",
            "achieved": achieved, "peak": peaks["hbm_gbs"], "unit": "GB/s", "frac": achieved / peaks["hbm_gbs"],
            "traffic": traffic, "traffic_source": traffic_src, "peak_source": peaks["source"],
            "algorithmic_bytes_per_launch": bytes_k, "ms_per_launch": per, "launches_timed": launches,
            "kernels_of_the_layer_forward": rows, "layer": layer_row}


def dump_outputs(r, out_dir):
    """What the last timed step hands its caller: the loss, every parameter's gradient and the parameters after Adam
    (flat, in the model's parameter order), as float32 DIR/{loss,grads,params}.npy.  The inputs, the initial
    parameters and the number of steps run before are fixed by the arguments, so two builds can be compared."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    for name, t in (("loss", r.loss), ("grads", r.model.flat_grad), ("params", r.model.flat_params.flat)):
        np.save(os.path.join(out_dir, name + ".npy"), t.detach().float().cpu().numpy())


# what only describes or breaks down a number: left out of the result line, kept in the full record on stderr
DETAIL_KEYS = {"kernels", "kernels_of_the_layer_forward", "layer", "pipeline", "note", "how", "sample",
               "traffic_source", "peak_source"}


def result_line(rec):
    """The record without its detail and with each secondary config cut to its rates, small enough (~4 KB) for a
    reader that keeps only the end of the output to parse."""
    def strip(o):
        return {k: strip(v) for k, v in o.items() if k not in DETAIL_KEYS} if isinstance(o, dict) else o

    def rates(res):
        out = {k: res[k] for k in ("value", "ms_per_step", "error") if k in res}
        out.update({k: res[k]["value"] for k in ("e2e", "cpu_baseline") if k in res})
        if "roofline" in res:
            out["roofline_frac"] = res["roofline"]["frac"]
        return out
    return strip(dict(rec, configs={k: rates(v) for k, v in rec["configs"].items()}))


def measure_workload(cfg, dev, rank, world, args, peaks, tf32_peak, full):
    """graphs/s (resident, CUDA-graph replay), e2e (host buffers), kernel table, dominant-kernel roofline for one
    workload.  full=True adds the secondary e2e modes and the paper-semantics co-headline (the C2 headline)."""
    import numpy as np
    import torch
    from agcn_b200 import _lib
    r = Runner(cfg, dev, rank, world, overlap=not args.no_overlap)
    steps, warmup = args.steps, args.warmup
    if not full:
        steps, warmup = max(5, min(args.steps, 10)), 3
    res = {"workload": cfg["name"], "mean_nodes": float(r.n_nodes.mean()), "parameters": r.model.n_parameters()}
    l0 = _lib.launch_count()
    ms_eager = r.timed(r.resident_step, steps, warmup)
    res["gpu_launches_per_step"] = (_lib.launch_count() - l0) / float(steps + warmup)
    launch_mode = "eager"
    sampler = None
    step_fn = r.resident_step
    if not args.no_graph:
        launch_mode = r.capture()
        if r.graph is not None:
            step_fn = r.replay
    if full and rank == 0:
        sampler = ClockSampler(dev.index or 0)
        sampler.start()
        sampler.wait_first(2.0)
    ms_step = r.timed(step_fn, steps, warmup)
    if full and rank == 0 and args.dump_outputs:
        dump_outputs(r, args.dump_outputs)
    if full:
        # the timed region is a few tens of milliseconds, shorter than nvidia-smi's sampling period: every rank keeps
        # the SAME step running (untimed, same count everywhere) for ~0.7 s so the clocks line describes this load
        for _ in range(int(min(0.7 / (ms_step * 1e-3), 5000))):
            step_fn()
        torch.cuda.synchronize()
        if sampler is not None:
            res["clocks"] = sampler.stop()
            res["clocks"]["note"] = ("sampled every 100 ms from just before the timed region to the end of ~0.7 s of "
                                     "the same step replayed back to back right after it")
    step_fn = None
    r.release()
    res.update({"value": world * r.B / (ms_step * 1e-3), "unit": "graphs/s", "ms_per_step": ms_step,
                "ms_per_step_eager": ms_eager, "launch": launch_mode})
    # ---- e2e from the pinned wire-layout host buffers
    e2e_steps = max(50, steps)    # (the pipeline fill / drain of a run is one un-overlapped staging: amortise it)
    ms_e2e = r.timed_e2e(e2e_steps, 3, "zero_copy")
    res["e2e"] = {"value": world * r.B / (ms_e2e * 1e-3), "unit": "graphs/s", "ms_per_step": ms_e2e,
                  "steps_timed": e2e_steps, "h2d_bytes_per_step": r.h2d_bytes(True), "host_layout_bytes": r.h2d_bytes(False), "d2h_bytes_per_step": 4,
                  "pipeline": "pinned host buffers in the reference's padded wire layout; per step: topology plan, pack "
                              "kernels reading the host arrays in place over PCIe (only the real rows move) on a side "
                              "stream under the previous step, one agcn_stack_loss_grad call + all-reduce + Adam "
                              "(eager launches), loss read back"}
    if world == 1 or os.environ.get("AGCN_BENCH_GRAPH_COLLECTIVES"):
        r.model.graph_collectives = world > 1     # opt-in: the NCCL all-reduce joins the capture (tools/e2e_multi.py)
        # the same loop with the step as ONE graph launch: re-captured for every batch (a new plan, new buffers and grid
        # sizes every step), the executable graph of the previous step updated in place (SimpleAGCNStep.step_graphed);
        # the next batch is staged by a feeder thread.  Bulk PCIe traffic delays eager launch commands, not a graph launch.
        upd0 = r.model.step_graph_updates
        # (8 untimed steps: the first process on a fresh box showed a one-off ~30 ms stall a few steps into the first
        # graph-launched run, tools/e2e_quick.py)
        try:
            ms_g = r.timed_e2e(e2e_steps, 8, "graph")
        except Exception as exc:      # the eager-launch loop above stands; say why the graph-launched one did not run
            ms_g = float("inf")
            res["e2e_graph_launch_error"] = str(exc)[:300]
            try:
                torch.cuda.synchronize()
            except Exception:
                pass
        graphed = dict(res["e2e"], value=world * r.B / (ms_g * 1e-3), ms_per_step=ms_g,
                       graph_updates_in_place=r.model.step_graph_updates - upd0, steps_run=e2e_steps + 8,
                       pipeline="pinned host buffers in the reference's padded wire layout; a feeder thread stages batch "
                                "i+1 (topology plan, pack kernels reading the host arrays in place over PCIe on a side "
                                "stream, labels) while the main thread captures step i (agcn_stack_loss_grad + Adam) for "
                                "ITS batch, updates the executable graph kept from step i-1 in place "
                                "(agcn_capture_end_launch) and launches it once; loss read back")
        if ms_g < ms_e2e:
            res["e2e_eager_launches"], res["e2e"], ms_e2e = res["e2e"], graphed, ms_g
        elif ms_g != float("inf"):
            res["e2e_graph_launch"] = graphed
    if "adj_rule" in cfg:
        ms_pt = r.timed_e2e(e2e_steps, 3, "points")
        res["e2e_points_in"] = {"value": world * r.B / (ms_pt * 1e-3), "unit": "graphs/s", "ms_per_step": ms_pt,
                                "h2d_bytes_per_step": int(r.batch.total_nodes * cfg["F"] * 4 + r.label_bytes() +
                                                          r.n_nodes.nbytes * 8),
                                "d2h_bytes_per_step": 4,
                                "pipeline": "the host hands over the point coordinates only (pinned, read in place); "
                                            "threshold adjacency + normalised Laplacian built on the device "
                                            "(agcn_point_laplacian) inside every timed step, then the same train step"}
    if full:
        ms_ce = r.timed_e2e(e2e_steps, 3, "copy_engine")
        res["e2e_copy_engine"] = {"value": world * r.B / (ms_ce * 1e-3), "unit": "graphs/s", "ms_per_step": ms_ce,
                                  "h2d_bytes_per_step": r.h2d_bytes(False), "d2h_bytes_per_step": 4,
                                  "pipeline": "the padded arrays staged through the copy engine, then packed on the device"}
        ms_se = r.timed_e2e(e2e_steps, 3, "serial")
        res["e2e_serial"] = {"value": world * r.B / (ms_se * 1e-3), "unit": "graphs/s", "ms_per_step": ms_se,
                             "h2d_bytes_per_step": r.h2d_bytes(True), "d2h_bytes_per_step": 4,
                             "pipeline": "zero-copy pack, step and loss read strictly one after the other"}
    # ---- per-kernel table of one eager step and the roofline of the dominant kernel (rank 0; no collectives inside)
    if rank == 0 and world == 1:
        table, ms_prof = r.kernel_table()
        res["kernels"] = {"note": "one eager step with every main kernel bracketed by CUDA events on its stream "
                                  "(side streams overlap: the sum can exceed the step)",
                          "ms_step_under_profile": ms_prof, "table": table}
        res["roofline"] = layer3_roofline(r, peaks, tf32_peak)
        flops, bytes_ = step_algorithmic(r.n_nodes, cfg["F"], FILTERS, K_ORDER, False)
        res["step_roofline"] = {"algorithmic_gflop": flops / 1e9, "algorithmic_mb": bytes_ / 1e6,
                                "achieved_tflops": flops / (ms_step * 1e-3) / 1e12,
                                "achieved_gbs": bytes_ / (ms_step * 1e-3) / 1e9,
                                "tensor_frac": flops / (ms_step * 1e-3) / 1e12 / tf32_peak,
                                "hbm_frac": bytes_ / (ms_step * 1e-3) / 1e9 / peaks["hbm_gbs"],
                                "note": "SGC_LL layers only (SURVEY.md section 8d formulas, real n), whole fwd+bwd step"}
    # ---- the same step with the paper's semantics (normalised Laplacian + differentiable metric): every kernel of
    # the metric / Laplacian block runs, forward and backward -- under CUDA-graph replay like the headline
    if full and not args.no_paper:
        del r
        gc.collect()
        rp = Runner(cfg, dev, rank, world, laplacian="paper", metric_grad="full")
        ms_pe = rp.timed(rp.resident_step, max(3, steps // 2), 3)
        mode = "eager" if args.no_graph else rp.capture()
        fn = rp.replay if rp.graph is not None else rp.resident_step
        ms_p = rp.timed(fn, max(3, steps // 2), 3)
        fn = None
        rp.release()
        res["paper_full_semantics"] = {"value": world * rp.B / (ms_p * 1e-3), "unit": "graphs/s", "ms_per_step": ms_p,
                                       "ms_per_step_eager": ms_pe, "semantics": "laplacian=paper, metric_grad=full",
                                       "launch": mode}
        if rank == 0 and world == 1:
            table, _ = rp.kernel_table()
            res["paper_full_semantics"]["kernels"] = table
        del rp
    gc.collect()
    torch.cuda.synchronize()
    return res


def run_ours(args):
    import torch
    import torch.distributed as dist
    import agcn_b200  # noqa: F401  (fails loudly when the library is missing)
    from agcn_b200 import _lib

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))

    def mark(what):   # progress markers on stderr (AGCN_BENCH_VERBOSE=1): where a multi-rank run is
        if os.environ.get("AGCN_BENCH_VERBOSE"):
            sys.stderr.write("[bench rank %d] %s\n" % (rank, what))
            sys.stderr.flush()

    if not torch.cuda.is_available():
        raise RuntimeError("bench.py needs a CUDA device; there is no CPU path")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    peaks = load_peaks()
    measured = measure_peaks(dev) if rank == 0 else {}
    tf32_peak = measured.get("tf32_tflops") or peaks["bf16_tflops"] / 2.0

    cfg = WORKLOADS[args.workload]
    mark("headline workload")
    main = measure_workload(cfg, dev, rank, world, args, peaks, tf32_peak, full=True)
    mark("headline done: %.3f ms" % main["ms_per_step"])
    others = {}
    keys = [] if args.no_configs else (["C1", "C3", "C4"] if world == 1 else ["C3"])
    for k in keys:
        if k == cfg["key"]:
            continue
        mark("config " + k)
        try:
            others[k] = measure_workload(WORKLOADS[k], dev, rank, world, args, peaks, tf32_peak, full=False)
        except Exception as exc:     # a secondary line must not take the headline down (all ranks fail alike)
            others[k] = {"workload": WORKLOADS[k]["name"], "error": str(exc)[:300]}
            torch.cuda.synchronize()

    if rank == 0:
        if args.skip_cpu:    # quick experiments only: the driver's runs always carry the CPU leg
            cpu_main = {"value": None, "unit": "graphs/s", "cores": 0, "kind": "port", "sample": "skipped (--skip-cpu)"}
            cpu_vec = None
        else:
            cpu_main = cpu_leg(cfg, "literal", 2, 1)
            cpu_vec = cpu_leg(cfg, "vectorised", 5, 2)
            if "paper_full_semantics" in main:
                main["paper_full_semantics"]["cpu_vectorised"] = cpu_leg(cfg, "vectorised", 3, 1, paper=True)
            for k, res in others.items():
                if "error" not in res:
                    res["cpu_baseline"] = cpu_leg(WORKLOADS[k], "vectorised", 3, 1)
                    if k == "C1":
                        res["cpu_literal"] = cpu_leg(WORKLOADS[k], "literal", 2, 1)
        config = bench_config(cfg, world)
        line = {"metric": "sgc_ll_train_graphs_per_s", "value": main["value"], "unit": "graphs/s", "n_gpus": world,
                "steps": args.steps, "warmup": args.warmup, "ms_per_step": main["ms_per_step"],
                "ms_per_step_eager": main["ms_per_step_eager"], "higher_is_better": True, "scaling": "weak",
                "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": config,
                "launch": main["launch"], "mean_nodes": main["mean_nodes"], "parameters": main["parameters"],
                "clocks": main.get("clocks"), "e2e": main["e2e"], "e2e_eager_launches": main.get("e2e_eager_launches"),
                "e2e_graph_launch": main.get("e2e_graph_launch"),
                "e2e_graph_launch_error": main.get("e2e_graph_launch_error"), "e2e_copy_engine": main.get("e2e_copy_engine"),
                "e2e_serial": main.get("e2e_serial"), "paper_full_semantics": main.get("paper_full_semantics"),
                "gpu_launches": int(round(main["gpu_launches_per_step"] * args.steps)),
                "gpu_launches_per_step": main["gpu_launches_per_step"],
                "roofline": main.get("roofline"), "step_roofline": main.get("step_roofline"),
                "kernels": main.get("kernels"), "peaks": dict(peaks, **measured),
                "cpu_baseline": {k: cpu_main.get(k) for k in ("value", "unit", "cores", "kind", "sample")},
                "cpu_vectorised": cpu_vec, "configs": others}
        print(json.dumps(result_line(line)))
        sys.stdout.flush()
        sys.stderr.write(json.dumps(line) + "\n")
        sys.stderr.flush()
    mark("done")
    if world > 1:
        # every CUDA graph that captured a collective is released (Runner.release) before the process group goes;
        # the watchdog only exists so a stuck teardown can never hold the driver's run
        watchdog = threading.Timer(60.0, lambda: os._exit(0))
        watchdog.daemon = True
        watchdog.start()
        gc.collect()
        torch.cuda.synchronize()
        dist.barrier()
        dist.destroy_process_group()
        watchdog.cancel()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="C2", choices=sorted(WORKLOADS))
    ap.add_argument("--cpu-kind", default="literal", choices=["literal", "vectorised"],
                    help="--impl reference: the reference-as-written port (default) or the batched torch restatement")
    ap.add_argument("--paper", action="store_true", help="--impl reference --cpu-kind vectorised: paper/full semantics")
    ap.add_argument("--no-graph", action="store_true", help="time eager launches only")
    ap.add_argument("--no-paper", action="store_true", help="skip the paper-semantics co-headline")
    ap.add_argument("--no-configs", action="store_true", help="skip the C1/C3/C4 block")
    ap.add_argument("--skip-cpu", action="store_true", help="skip the CPU legs (quick experiments)")
    ap.add_argument("--no-overlap", action="store_true", help="N > 1: one all-reduce after backward instead of buckets")
    ap.add_argument("--ref-graphs", type=int, default=0, help="graphs per step of the reference arm (default: the batch)")
    ap.add_argument("--dump-outputs", metavar="DIR", default="",
                    help="write the loss, gradients and parameters of the last timed step as DIR/*.npy")
    args = ap.parse_args()
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
