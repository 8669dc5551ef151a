#!/usr/bin/env python
"""Validation and inference throughput: the captured GraphedEvaluator against the eager drop-in path it replaces, in one process.

One JSON line per network (skippfn, gat, gine) on the Oberrhein feeder (ober_sub, N=70, E=69) at B=4096 scenarios per batch:
  evaluate  = pack -> eval-mode forward -> dss2_eval_metrics_acc (no host sync), one CUDA graph replay per batch
  infer     = pack -> eval-mode forward -> dss2_pflow_est, one CUDA graph replay per batch
  eager_*   = the drop-in path a user of the networks / data modules runs: batching.pack_batch (host-side sizes), the module in eval()
              under no_grad, then metrics.evaluate_batch (one host sync per batch) or the estimate built with torch ops + data.get_pflow
              (bench.py's inference step)
The four arms alternate round by round; each time is the median over rounds of (CUDA-event time of `calls` back-to-back calls) / calls.
Launches per call count the project's kernels (`_lib.launch_count`; for the captured arms the kernels inside the graph, which one replay
issues); the eager arms also run torch ops that are not counted.
The working set (store + activations at B=4096, > 1 GB) exceeds the 126 MB L2; no flush between calls.

    python tools/eval_bench.py [--batch 4096] [--scenarios 16384] [--rounds 7] [--calls 20] [--out FILE]
"""
import argparse
import json
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "deep-statistical-solver-for-distribution-system-state-estimation_b200"))


def card():
    import torch
    info = {"device": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"], capture_output=True,
                           text=True, timeout=30).stdout.strip()
        info["power_limit"], info["sm_max_clock"] = [s.strip() for s in q.split(",")]
    except Exception as exc:   # no nvidia-smi: say so instead of inventing a number
        info["power_limit"] = f"unavailable:{type(exc).__name__}"
    return info


def module(network):
    import networks
    if network == "skippfn":
        return networks.SkipPFN(dim_featn=8, dim_feate=6, dim_out=2, dim_hid=32, n_gnn_layers=8, K=2, dropout_rate=0.3, L=5)
    if network == "gat":
        return networks.GAT_DSSE(dim_feat=8, dim_dense=32, dim_out=2, heads=1, num_layers=8, edge_dim=6)
    return networks.GINE_DSSE(dim_feat=8, dim_dense=32, dim_out=2, num_layers=8, edge_dim=6)


def run(network, store, args, dev):
    import torch
    import data
    from dss2 import _lib, batching, metrics
    from dss2.evaluator import GraphedEvaluator
    B = args.batch
    torch.manual_seed(0)
    model = module(network).to(dev).eval()
    sd = {k: v.detach() for k, v in model.state_dict().items()}
    ev = GraphedEvaluator(store, B, network=network, state_dict=sd)
    xs, xm = store.x_std.to(dev), store.x_mean.to(dev)
    nb = store.num_scenarios // B
    sels = [torch.arange(i * B, (i + 1) * B, device=dev) for i in range(nb)]
    k = {"i": 0}

    def next_ids():
        k["i"] += 1
        return sels[k["i"] % nb]

    def eager_evaluate():
        sel = next_ids()
        pb = batching.pack_batch(store, sel)
        with torch.no_grad():
            out = model(pb.x[:, :8], pb.edge_index, pb.edge_attr[:, :6])
        metrics.evaluate_batch(out, pb.y, pb.x, pb.edge_index, pb.edge_attr, store.x_mean, store.x_std)

    def eager_infer():
        sel = next_ids()
        pb = batching.pack_batch(store, sel)
        with torch.no_grad():
            out = model(pb.x[:, :8], pb.edge_index, pb.edge_attr[:, :6])
            est = torch.cat([out[:, 0:1] * xs[:1] + xm[:1], out[:, 1:] * (1. - pb.x[:, 9:10])], 1)
            data.get_pflow(est, pb.edge_index, node_param=pb.x[:, 8:], edge_param=pb.edge_attr[:, 6:])

    arms = {"evaluate": lambda: ev.evaluate(next_ids()), "infer": lambda: ev.infer(next_ids()), "eager_evaluate": eager_evaluate,
            "eager_infer": eager_infer}
    launches = {}
    for name, fn in arms.items():        # warm-up (captures the graphs), then one counted call
        for _ in range(3):
            fn()
        torch.cuda.synchronize()
        n0 = _lib.launch_count()
        fn()
        torch.cuda.synchronize()
        launches[name] = _lib.launch_count() - n0
    for name in ("evaluate", "infer"):   # a replay issues no launches of its own: the kernels inside the graph, counted at its warm-up
        launches[name] = ev.launches_per_call[name]
    times = {name: [] for name in arms}
    for _ in range(args.rounds):
        for name, fn in arms.items():
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            torch.cuda.synchronize()
            a.record()
            for _ in range(args.calls):
                fn()
            b.record()
            b.synchronize()
            times[name].append(a.elapsed_time(b) / args.calls)
    ev.metrics(reset=True)
    res = {"network": network, "grid": "ober_sub (N=70,E=69)", "batch": B, "resident_scenarios": store.num_scenarios, "rounds": args.rounds,
           "calls_per_round": args.calls}
    for name, ts in times.items():
        ms = statistics.median(ts)
        res[name] = {"ms_per_call": round(ms, 4), "ms_min": round(min(ts), 4), "ms_max": round(max(ts), 4),
                     "scenarios_per_s": round(B / ms * 1e3, 1), "launches_per_call": launches[name],
                     "graph_replays_per_call": 0 if name.startswith("eager") else 1}
    res["speedup_evaluate"] = round(res["eager_evaluate"]["ms_per_call"] / res["evaluate"]["ms_per_call"], 3)
    res["speedup_infer"] = round(res["eager_infer"]["ms_per_call"] / res["infer"]["ms_per_call"], 3)
    res["evaluator_memory_MB"] = round(ev.memory_bytes() / 2 ** 20, 2)
    res.update(card())
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=4096)
    ap.add_argument("--scenarios", type=int, default=16384)
    ap.add_argument("--rounds", type=int, default=7)
    ap.add_argument("--calls", type=int, default=20)
    ap.add_argument("--networks", default="skippfn,gat,gine")
    ap.add_argument("--out", default=None, help="also write the JSON lines to this file")
    args = ap.parse_args()
    import torch
    from dss2 import synth
    if not torch.cuda.is_available():
        raise SystemExit("eval_bench.py measures on a CUDA device; none found")
    dev = torch.device("cuda:0")
    store = synth.synthetic_store(synth.load_grid("ober_sub"), args.scenarios, seed=1234, device=dev)
    lines = []
    for network in args.networks.split(","):
        line = json.dumps(run(network, store, args, dev))
        print(line, flush=True)
        lines.append(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
