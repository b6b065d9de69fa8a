"""Prediction rate of the SimpleAGCN stack against its training step, on bench.py's workloads.

    python tools/predict_rate.py --out DIR [--configs C1,C2,C3] [--warmup 20] [--iters 100] [--regression C1:1,C2:617]

For every workload, with the batch resident in HBM (bench.py's inputs, one GPU):
  predict_eager     SimpleAGCNStep.predict_proba (one agcn_stack_predict call), eager launches
  predict_replay    the same call captured in a CUDA graph and replayed
  train_eager       loss_and_grads + apply_adam (one agcn_stack_loss_grad call + agcn_adam_step), eager launches
  train_replay      the same step captured and replayed
Each is the median over `iters` calls timed with CUDA events after `warmup` untimed ones; L2 is flushed (a 256 MB fill,
not timed) before every timed call, as bench.py does.  graphs/s = B / median.  The per-kernel table of one eager
prediction comes from the library's own launch profiler (agcn_profile_enable / agcn_profile_read).  The card's name and
power limit are read with a read-only nvidia-smi query in the same run.  Writes DIR/predict_rate.json and prints it.

--regression KEY:T,... (opt-in) times the same four calls for the regression head (loss="weighted_l2", T outputs) on the
inputs of workload KEY, with synthetic N(0, 1) targets and 0/1 weights; predict_* is SimpleAGCNStep.predict (the values).
The results go to "regression" in the record, beside the classifiers of "configs".

--residual KEY,... (opt-in) times the same four calls for ResAGCNStep (agcn_b200.residual_agcn: the default residual
body of SGC_LL_Reslap layers and BlockEnd blocks, then workload KEY's head) on workload KEY's inputs, and also counts the
launches of one training step.  The results go to "residual" in the record.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench  # noqa: E402


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                             stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True, timeout=30).stdout.strip()
        name, power = [p.strip() for p in out.split(",")[:2]]
        return {"name": name, "power_limit": power}
    except Exception as exc:
        return {"name": torch.cuda.get_device_name(0), "power_limit": "unread (%s)" % type(exc).__name__}


def median_ms(fn, warmup, iters, flush):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    times = []
    for _ in range(iters):
        flush.fill_(1.0)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        e1.synchronize()
        times.append(e0.elapsed_time(e1))
    return statistics.median(times)


def captured(fn):
    """fn captured in a CUDA graph (warmed up on a side stream first); returns the graph's replay."""
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        for _ in range(3):
            fn()
    torch.cuda.current_stream().wait_stream(side)
    torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        fn()
    return graph


def run_config(key, warmup, iters, flush, regression_tasks=None, residual=False):
    """regression_tasks = T: the weighted-L2 regressor with T outputs on workload `key`'s inputs instead of its
    classifier.  residual: ResAGCNStep's body instead of SimpleAGCN's."""
    import agcn_b200
    from agcn_b200 import _lib
    from agcn_b200.residual_agcn import ResAGCNStep
    from agcn_b200.simple_agcn import SimpleAGCNStep, synthetic_labels
    cfg = bench.WORKLOADS[key]
    dev = torch.device("cuda:0")
    X, L, n, tg, w = bench.make_inputs(cfg, 0)
    B = cfg["B"]
    loss, n_tasks = cfg["loss"], cfg["n_tasks"]
    if regression_tasks is not None:
        loss, n_tasks = "weighted_l2", regression_tasks
    if residual:
        model = ResAGCNStep(cfg["F"], final_feature_n=bench.FINAL, n_tasks=n_tasks, K=bench.K_ORDER, batch_size=B,
                            device=dev, loss=loss)
    else:
        model = SimpleAGCNStep(cfg["F"], bench.FILTERS, bench.FINAL, n_tasks, bench.K_ORDER, B, device=dev, loss=loss)
    batch = agcn_b200.GraphBatch(n, cfg["Nmax"], device=dev)
    Xd, Ld = batch.pack_nodes(torch.from_numpy(X).to(dev)), batch.pack_lap(torch.from_numpy(L).to(dev))
    if regression_tasks is None:
        tg_d, w_d = torch.from_numpy(tg).to(dev), torch.from_numpy(w).to(dev)
    else:
        tg_d, w_d = synthetic_labels(B, n_tasks, cfg["seed"], dev, loss)

    def predict():
        if regression_tasks is None:
            model.predict_proba(Xd, Ld, batch)
        else:
            model.predict(Xd, Ld, batch)

    def train():
        model.loss_and_grads(Xd, Ld, batch, tg_d, w_d)
        model.apply_adam()

    res = {"workload": cfg["name"], "B": B}
    if regression_tasks is not None:
        res.update(loss=loss, n_tasks=n_tasks)
    ms = {"predict_eager": median_ms(predict, warmup, iters, flush)}
    g = captured(predict)
    ms["predict_replay"] = median_ms(g.replay, warmup, iters, flush)
    del g
    ms["train_eager"] = median_ms(train, warmup, iters, flush)
    g = captured(train)
    ms["train_replay"] = median_ms(g.replay, warmup, iters, flush)
    del g
    for k, v in ms.items():
        res[k] = {"ms": v, "graphs_per_s": B / (v * 1e-3)}
    # the per-kernel table of one eager prediction
    predict()
    torch.cuda.synchronize()
    _lib.profile_enable(True)
    c0 = _lib.launch_count()
    predict()
    c1 = _lib.launch_count()
    table = _lib.profile_read()
    _lib.profile_enable(False)
    res["predict_launches"] = c1 - c0
    if residual:
        res["layout"] = [type(l).__name__ for l in model.layers]
        c0 = _lib.launch_count()
        train()
        res["train_launches"] = _lib.launch_count() - c0
        torch.cuda.synchronize()
    res["predict_kernels_ms"] = {k: {"launches": v[0], "ms": v[1]} for k, v in sorted(table.items(),
                                                                                    key=lambda kv: -kv[1][1])}
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True, help="directory for predict_rate.json (the only file written)")
    ap.add_argument("--configs", default="C1,C2,C3")
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--iters", type=int, default=100)
    ap.add_argument("--regression", default="",
                    help="opt-in: KEY:T,... times the weighted-L2 regressor with T outputs on workload KEY's inputs")
    ap.add_argument("--residual", default="",
                    help="opt-in: KEY,... times ResAGCNStep (the residual body) on workload KEY's inputs")
    args = ap.parse_args()
    regression = [(k, int(t)) for k, t in (item.split(":") for item in args.regression.split(",") if item)]
    for k, t in regression:
        if k not in bench.WORKLOADS or t < 1:
            raise SystemExit("--regression: KEY:T with KEY one of %s and T >= 1" % sorted(bench.WORKLOADS))
    residual = [k for k in args.residual.split(",") if k]
    for k in residual:
        if k not in bench.WORKLOADS:
            raise SystemExit("--residual: KEY,... with KEY one of %s" % sorted(bench.WORKLOADS))
    if not torch.cuda.is_available():
        raise SystemExit("predict_rate.py measures on the GPU; no CUDA device found")
    flush = torch.empty(256 * 1024 * 1024 // 4, dtype=torch.float32, device="cuda:0")
    out = {"gpu": gpu_info(), "warmup": args.warmup, "iters": args.iters, "statistic": "median, CUDA events",
           "configs": {}}
    for key in args.configs.split(","):
        out["configs"][key] = run_config(key, args.warmup, args.iters, flush)
        r = out["configs"][key]
        print("%s: predict %.0f graphs/s eager, %.0f replay; train step %.0f eager, %.0f replay; %d launches per predict"
              % (key, r["predict_eager"]["graphs_per_s"], r["predict_replay"]["graphs_per_s"],
                 r["train_eager"]["graphs_per_s"], r["train_replay"]["graphs_per_s"], r["predict_launches"]),
              flush=True)
    if regression:
        out["regression"] = {}
    for key, t in regression:
        name = "%s_T%d" % (key, t)
        out["regression"][name] = r = run_config(key, args.warmup, args.iters, flush, regression_tasks=t)
        print("%s weighted_l2: predict %.0f graphs/s eager, %.0f replay; train step %.0f eager, %.0f replay; "
              "%d launches per predict"
              % (name, r["predict_eager"]["graphs_per_s"], r["predict_replay"]["graphs_per_s"],
                 r["train_eager"]["graphs_per_s"], r["train_replay"]["graphs_per_s"], r["predict_launches"]),
              flush=True)
    if residual:
        out["residual"] = {}
    for key in residual:
        out["residual"][key] = r = run_config(key, args.warmup, args.iters, flush, residual=True)
        print("%s residual: predict %.0f graphs/s eager, %.0f replay; train step %.0f eager, %.0f replay; "
              "%d launches per predict, %d per training step"
              % (key, r["predict_eager"]["graphs_per_s"], r["predict_replay"]["graphs_per_s"],
                 r["train_eager"]["graphs_per_s"], r["train_replay"]["graphs_per_s"], r["predict_launches"],
                 r["train_launches"]), flush=True)
    os.makedirs(args.out, exist_ok=True)
    with open(os.path.join(args.out, "predict_rate.json"), "w") as f:
        json.dump(out, f, indent=1)
    print(json.dumps(out))


if __name__ == "__main__":
    main()
