#!/usr/bin/env python
"""Batched AC power flow (dss2.powerflow.solve, csrc/powerflow.cu) on the device, and a host baseline, in one process.

Workloads:
  ober      10^6 Oberrhein scenarios (ober_sub, N=70, 69 closed edges).  Injections: the pi-model's injections at the states of
            synth.sample_scenarios(ober_sub, 10**6, seed=1234) (dss2.powerflow.injections: the scenarios' own p/q columns, with the model's
            value at the declared zero-injection buses, which sample_scenarios reports as zero), so every solution has a known answer.
  feeder10k 1 000 scenarios of synth.replicate_feeder(ober_sub, 143) (N=10 010), same recipe.
Reported per workload: solve time (median over rounds of CUDA-event time around one solve; the window ends in a synchronise) and
scenarios/s; the iteration histogram; max |V - V_true| and |theta - theta_true|; the workspace; the bytes one Newton iteration touches
per scenario, counted from shapes (every workspace double read and written once, the injections read once: a count, not a measured
traffic).  For ober also solve + build_scenario_store (solved_scenarios, noise draws, the CUDA dataset builder).
Host baseline: powerflow_nr of tests/powerflow_reference.py (dense fp64 Newton-Raphson, numpy) over the first 1 000 ober scenarios in a
process pool with one worker and one BLAS thread per host core; the core count is printed.  The working sets exceed the 126 MB L2; no flush between rounds.

    python tools/powerflow_bench.py [--scenarios 1000000] [--feeder-scenarios 1000] [--rounds 3] [--host-scenarios 1000] [--out FILE]
"""
import os

for _v in ("OMP_NUM_THREADS", "OPENBLAS_NUM_THREADS", "MKL_NUM_THREADS"):   # one BLAS thread per host worker
    os.environ.setdefault(_v, "1")

import argparse
import json
import multiprocessing
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "deep-statistical-solver-for-distribution-system-state-estimation_b200"))
sys.path.insert(0, os.path.join(ROOT, "tests"))


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


def timed(fn, rounds):
    import torch
    fn()                                      # warm-up: module load, symbolic analysis and its upload, allocator
    torch.cuda.synchronize()
    ms = []
    for _ in range(rounds):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        out = fn()
        b.record()
        torch.cuda.synchronize()
        ms.append(a.elapsed_time(b))
    return statistics.median(ms), ms, out


def workload(grid, S, rounds, seed=1234):
    import torch
    from dss2 import _lib, powerflow, synth
    _, _, labels = synth.sample_scenarios(grid, S, seed=seed, device="cuda")
    p, q = powerflow.injections(grid, labels[..., 0], labels[..., 1])
    torch.cuda.synchronize()
    med, ms, r = timed(lambda: powerflow.solve(grid, p, q), rounds)
    sym = powerflow.symbolic(grid)
    N, n, blocks = sym["num_buses"], sym["num_buses"] - 1, sym["blk_col"].size
    per = powerflow.workspace_bytes(grid, 1)
    chunk = max(1, min(S, powerflow.WORKSPACE_BUDGET // per))
    its = r["iterations"].long()
    res = {"scenarios": S, "buses": N, "closed_edges": int(sym["edge_ft"].shape[0]), "blocks": int(blocks), "fill": int(sym["fill"]),
           "solve_ms_median": med, "solve_ms_all": ms, "scenarios_per_s": S / (med / 1e3),
           "converged": int(r["converged"].sum()), "iteration_histogram": {int(k): int(v) for k, v in enumerate(torch.bincount(its).tolist()) if v},
           "max_abs_err_vm_pu": float((r["vm_pu"] - labels[..., 0]).abs().max()), "max_abs_err_va_rad": float((r["va_rad"] - labels[..., 1]).abs().max()),
           "max_mismatch_mva": float(r["max_mismatch_mva"].max()), "chunk_scenarios": int(chunk), "workspace_bytes": int(powerflow.workspace_bytes(grid, chunk)),
           "workspace_bytes_per_scenario": int(per),
           "bytes_per_iteration_per_scenario_from_shapes": 8 * (2 * (4 * N + 2 * n + 4 * blocks) + 2 * n),
           "kernel_launches_per_solve": None}
    before = _lib.launch_count()
    powerflow.solve(grid, p, q)
    res["kernel_launches_per_solve"] = _lib.launch_count() - before
    return res, p, q, labels


def _host_chunk(args):
    import powerflow_reference as ref
    bus, edge, p, q = args
    return ref.powerflow_nr(bus, edge, p, q, 1.03)[2]


def host_baseline(grid, p, q):
    import numpy as np
    cores = os.cpu_count()
    parts = [(grid["bus_param"], grid["edge_param"], pp, qq) for pp, qq in zip(np.array_split(p, cores), np.array_split(q, cores)) if len(pp)]
    ctx = multiprocessing.get_context("spawn")
    with ctx.Pool(cores) as pool:
        pool.map(_host_chunk, parts[:cores])  # warm-up: imports in every worker
        t0 = time.perf_counter()
        its = np.concatenate(pool.map(_host_chunk, parts))
        dt = time.perf_counter() - t0
    return {"scenarios": int(p.shape[0]), "host_cores": cores, "seconds": dt, "scenarios_per_s": p.shape[0] / dt,
            "iteration_histogram": {int(k): int(v) for k, v in enumerate(np.bincount(its)) if v}}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--scenarios", type=int, default=10 ** 6)
    ap.add_argument("--feeder-scenarios", type=int, default=1000)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--host-scenarios", type=int, default=1000)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    from dss2 import dataset, powerflow, synth
    if not torch.cuda.is_available():
        raise SystemExit("powerflow_bench: no CUDA device")
    out = {"card": card()}
    ober = synth.load_grid("ober_sub")
    res, p, q, _ = workload(ober, args.scenarios, args.rounds)
    S, N = p.shape
    E = res["closed_edges"]

    def solve_and_store():
        nodes, edges, labels = powerflow.solved_scenarios(ober, p, q)
        gen = torch.Generator(device="cuda").manual_seed(7)
        zn = torch.randn(S, N, 4, generator=gen, dtype=torch.float64, device="cuda")
        ze = torch.randn(S, E, 2, generator=gen, dtype=torch.float64, device="cuda")
        return dataset.build_scenario_store(nodes, edges, labels, ober["noise_param"], ober["meas_v"], ober["meas_pflow"], zn, ze, device="cuda")

    med, ms, _ = timed(solve_and_store, args.rounds)
    res["solve_plus_build_store_ms_median"], res["solve_plus_build_store_ms_all"] = med, ms
    out["ober"] = res
    print(json.dumps({"ober": res}), flush=True)
    host_p, host_q = p[:args.host_scenarios].cpu().numpy(), q[:args.host_scenarios].cpu().numpy()
    del p, q
    torch.cuda.empty_cache()
    feeder = synth.replicate_feeder(ober, 143)
    out["feeder10k"], *_ = workload(feeder, args.feeder_scenarios, max(1, args.rounds - 1))
    print(json.dumps({"feeder10k": out["feeder10k"]}), flush=True)
    out["host_baseline_ober"] = host_baseline(ober, host_p, host_q)
    print(json.dumps({"host_baseline_ober": out["host_baseline_ober"]}), flush=True)
    out["gpu_speedup_over_host_ober"] = out["ober"]["scenarios_per_s"] / out["host_baseline_ober"]["scenarios_per_s"]
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(out, f, indent=1)
    print(json.dumps(out))


if __name__ == "__main__":
    main()
