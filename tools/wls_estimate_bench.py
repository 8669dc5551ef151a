#!/usr/bin/env python
"""WLS state estimation (dss2.estimation.wls_estimate, csrc/estimate.cu) on the device beside the trained-model path it is compared
with, and a host baseline, in one process.

Workloads:
  ober      Oberrhein synthetic stores (synth.synthetic_store(ober_sub, S, seed=1234): N=70, 69 closed edges) at S = 10^5 and 10^6,
            estimated in batches of B=4096 scenarios (contiguous scenario ranges, PyG order) with the default chunk.  The iteration
            histogram, the objective, convergence and the evaluate_batch metrics of the estimate against the labels (mean over batches).
  chunk     the same 10^5 store in batches of 32 768 scenarios, with the 1 GiB-budget chunk (the whole batch) against an L2-sized chunk
            (at most 100 MB of workspace), alternating.  At B = 4096 the budget chunk is the whole batch and below 100 MB as well.
  infer     GraphedEvaluator.infer (SkipPFN, 8 layers x 5 sub-nets, random weights) on the same B = 4096 batches of the 10^5 store.
  feeder10k 100 scenarios of synth.replicate_feeder(ober_sub, 143) (N = 9 868) in one call.
Times: CUDA events around a whole pass over the store (every batch), the window ending in a synchronise; median of `rounds` passes after
a warm-up pass.  Each wls_estimate call includes its one host synchronisation (the topology check).  The bytes one Gauss-Newton
iteration touches per scenario are counted from shapes (every workspace double the kernel reads or writes, once per access in its
loops): an analytical count, not a measured traffic.
Host baseline: tests/wls_estimate_reference.py (fp64 Gauss-Newton with an autograd Jacobian and dense least squares; the test oracle,
not an optimised host solver) over the first scenarios of the 10^5 store in a process pool with one worker per host core.

    python tools/wls_estimate_bench.py [--rounds 3] [--host-scenarios 1000] [--out FILE]
"""
import os

for _v in ("OMP_NUM_THREADS", "OPENBLAS_NUM_THREADS", "MKL_NUM_THREADS"):   # one BLAS thread per host worker
    os.environ.setdefault(_v, "1")

import argparse
import json
import multiprocessing
import statistics
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for _p in ("deep-statistical-solver-for-distribution-system-state-estimation_b200", "tests", "oracle", "tools"):
    sys.path.insert(0, os.path.join(ROOT, _p))

B = 4096
L2_BYTES = 100 * 10 ** 6


def batches(store, b):
    import torch
    N, E = store.max_nodes, store.max_edges
    dev = store.x.device
    out = []
    for s0 in range(0, store.num_scenarios, b):
        n = min(b, store.num_scenarios - s0)
        off = torch.arange(n, device=dev).repeat_interleave(E) * N
        out.append({"x": store.x[s0 * N:(s0 + n) * N], "edge_attr": store.edge_attr[s0 * E:(s0 + n) * E], "y": store.y[s0 * N:(s0 + n) * N],
                    "edge_index": store.edge_index[:, s0 * E:(s0 + n) * E] + off, "ptr": torch.arange(n + 1, device=dev) * N})
    return out


def timed(fn, rounds):
    import torch
    fn()
    torch.cuda.synchronize()
    ms = []
    for _ in range(rounds):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        torch.cuda.synchronize()
        ms.append(a.elapsed_time(b))
    return statistics.median(ms), ms


def per_iteration_bytes(sym):
    """Workspace doubles one Gauss-Newton iteration reads + writes per scenario, counted from the kernel's loops (not a measurement)."""
    N, E, nb, nu = sym["num_buses"], sym["num_edges"], int(sym["blk_col"].size), int(sym["upd"].shape[0])
    m = (sym["sup_ptr"][1:] - sym["sup_ptr"][:-1]).astype("int64")
    inc = int(sym["inc_ptr"][-1])
    edge_pass = 28 * E                                    # V, th of both ends and 4 parameters in, flows and partials out
    zero = 4 * nb + 2 * N
    buses = 12 * N + 26 * inc + int((4 * m + 8 * m + 12 * m * m).sum())   # measurements, state, F; incident flows into H; H^T W H
    edges = 54 * E                                        # measurements, flows, partials, F and 4 blocks read-modify-write
    lu = 12 * nb + 12 * nu + 8 * N + 8 * nb + 4 * N       # factor (lower blocks, updates, pivots), both substitutions
    update = 6 * N
    return 8 * (edge_pass + zero + buses + edges + lu + update)


def _host(args):
    import wls_estimate_reference as ref
    out = []
    for x, ea, ei, st in args:
        out.append(ref.estimate(x, ea, ei, st)[2])
    return out


def host_baseline(parts):
    cores = os.cpu_count()
    chunks = [parts[i::cores] for i in range(cores) if parts[i::cores]]
    ctx = multiprocessing.get_context("spawn")
    with ctx.Pool(len(chunks)) as pool:
        pool.map(_host, [c[:1] for c in chunks])     # warm-up: imports in every worker
        t0 = time.perf_counter()
        its = [i for r in pool.map(_host, chunks) for i in r]
        dt = time.perf_counter() - t0
    return {"scenarios": len(parts), "host_cores": cores, "seconds": dt, "scenarios_per_s": len(parts) / dt,
            "iteration_histogram": {int(k): its.count(k) for k in sorted(set(its))}}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--sizes", default="100000,1000000")
    ap.add_argument("--feeder-scenarios", type=int, default=100)
    ap.add_argument("--host-scenarios", type=int, default=1000)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    from powerflow_bench import card
    from dss2 import estimation, metrics, synth
    from dss2.evaluator import GraphedEvaluator
    from eval_bench import module
    if not torch.cuda.is_available():
        raise SystemExit("wls_estimate_bench: no CUDA device")
    out = {"card": card(), "batch": B}
    ober = synth.load_grid("ober_sub")
    host_parts = None
    for S in [int(s) for s in args.sizes.split(",")]:
        store = synth.synthetic_store(ober, S, seed=1234, device="cuda")
        bs = batches(store, B)
        stats = [store.x_mean, store.x_std, store.edge_mean, store.edge_std]
        ep = ober["edge_param"]
        sym = estimation.symbolic(ep[ep[:, 6] == 1.0, :2].astype("int64"), ober["bus_param"][:, 1])
        med, ms = timed(lambda: [estimation.wls_estimate(b["x"], b["edge_index"], b["edge_attr"], b["ptr"], *stats) for b in bs], args.rounds)
        its, conv, obj, acc = [], 0, [], {}
        for b in bs:
            r = estimation.wls_estimate(b["x"], b["edge_index"], b["edge_attr"], b["ptr"], *stats)
            its.append(r["iterations"].long())
            conv += int(r["converged"].sum())
            obj.append(r["objective"])
            m = metrics.evaluate_batch(r["output"], b["y"], b["x"], b["edge_index"], b["edge_attr"], store.x_mean, store.x_std)
            for k, v in m.items():
                acc[k] = acc.get(k, 0.0) + v / len(bs)
        its = torch.cat(its)
        res = {"scenarios": S, "buses": sym["num_buses"], "closed_edges": sym["num_edges"], "blocks": int(sym["blk_col"].size),
               "fill": int(sym["fill"]), "pass_ms_median": med, "pass_ms_all": ms, "scenarios_per_s": S / (med / 1e3),
               "converged": conv, "iteration_histogram": {int(k): int(v) for k, v in enumerate(torch.bincount(its).tolist()) if v},
               "objective_median": float(torch.cat(obj).median()), "metrics_vs_labels_mean_over_batches": acc,
               "workspace_bytes_per_scenario": estimation.workspace_bytes(sym, 1),
               "bytes_per_iteration_per_scenario_from_shapes": per_iteration_bytes(sym)}
        it_mean = float(its.double().mean())
        res["analytical_workspace_bandwidth_GBps"] = res["bytes_per_iteration_per_scenario_from_shapes"] * it_mean * S / (med / 1e3) / 1e9
        out[f"ober_{S}"] = res
        print(json.dumps({f"ober_{S}": res}), flush=True)
        if host_parts is None:
            import test_wls_estimate as T
            hb, _ = T.store_batch(store, min(args.host_scenarios, S))
            host_parts = [T.scenario(hb, stats, s) for s in range(min(args.host_scenarios, S))]
            # chunk: 1 GiB budget (the whole batch) against an L2-sized chunk, alternating, on batches of 32 768
            big = batches(store, 32768)
            per = estimation.workspace_bytes(sym, 1)
            arms = {"budget_1GiB": min(32768, (1 << 30) // per), "l2_100MB": L2_BYTES // per}
            times = {k: [] for k in arms}
            for _ in range(args.rounds):
                for k, c in arms.items():
                    times[k].append(timed(lambda: [estimation.wls_estimate(b["x"], b["edge_index"], b["edge_attr"], b["ptr"], *stats, chunk=c)
                                                   for b in big], 1)[0])
            out["chunk"] = {"batch": 32768, "scenarios": S, **{k: {"chunk": int(arms[k]), "pass_ms": v, "scenarios_per_s": S / (statistics.median(v) / 1e3)}
                                                               for k, v in times.items()}}
            print(json.dumps({"chunk": out["chunk"]}), flush=True)
            # the trained-model path on the same batches
            torch.manual_seed(0)
            sd = {k: v.detach() for k, v in module("skippfn").cuda().eval().state_dict().items()}
            ev = GraphedEvaluator(store, B, network="skippfn", state_dict=sd)
            sels = [torch.arange(i * B, min((i + 1) * B, S), device="cuda") for i in range(len(bs))]
            med_i, ms_i = timed(lambda: [ev.infer(s) for s in sels], args.rounds)
            out["infer_skippfn"] = {"scenarios": S, "pass_ms_median": med_i, "pass_ms_all": ms_i, "scenarios_per_s": S / (med_i / 1e3),
                                    "wls_over_infer_time": med / med_i}
            print(json.dumps({"infer_skippfn": out["infer_skippfn"]}), flush=True)
            del ev
        del store, bs
        torch.cuda.empty_cache()
    feeder = synth.replicate_feeder(ober, 143)
    fs = synth.synthetic_store(feeder, args.feeder_scenarios, seed=1234, device="cuda")
    fb = batches(fs, args.feeder_scenarios)[0]
    fstats = [fs.x_mean, fs.x_std, fs.edge_mean, fs.edge_std]
    med, ms = timed(lambda: estimation.wls_estimate(fb["x"], fb["edge_index"], fb["edge_attr"], fb["ptr"], *fstats), max(1, args.rounds - 1))
    r = estimation.wls_estimate(fb["x"], fb["edge_index"], fb["edge_attr"], fb["ptr"], *fstats)
    ep = feeder["edge_param"]
    fsym = estimation.symbolic(ep[ep[:, 6] == 1.0, :2].astype("int64"), feeder["bus_param"][:, 1])
    out["feeder10k"] = {"scenarios": args.feeder_scenarios, "buses": fsym["num_buses"], "blocks": int(fsym["blk_col"].size),
                        "lu_updates": int(fsym["upd"].shape[0]), "call_ms_median": med, "call_ms_all": ms,
                        "scenarios_per_s": args.feeder_scenarios / (med / 1e3), "converged": int(r["converged"].sum()),
                        "iteration_histogram": {int(k): int(v) for k, v in enumerate(torch.bincount(r["iterations"].long()).tolist()) if v},
                        "workspace_bytes_per_scenario": estimation.workspace_bytes(fsym, 1),
                        "max_abs_err_vm_pu_vs_labels": float((r["vm_pu"] - fb["y"][:, 0].double()).abs().max())}
    print(json.dumps({"feeder10k": out["feeder10k"]}), flush=True)
    out["host_baseline_ober"] = host_baseline(host_parts)
    print(json.dumps({"host_baseline_ober": out["host_baseline_ober"]}), flush=True)
    out["gpu_speedup_over_host_ober"] = out[f"ober_{args.sizes.split(',')[0]}"]["scenarios_per_s"] / out["host_baseline_ober"]["scenarios_per_s"]
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(out, f, indent=1)
    print(json.dumps(out))


if __name__ == "__main__":
    main()
