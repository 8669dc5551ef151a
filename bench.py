#!/usr/bin/env python
"""bench.py - the driver's measurement contract for the DSS2 hot path on B200.

Metric (BASELINE.json): train scenarios/s = scenarios pushed through one full training step
(batch packer -> SkipPFN(8,6,2,32,8,2,0.3,5) forward with in-kernel dropout -> fused branch-flow/WLS loss forward+backward ->
GNN backward (recompute) -> gradient reduction [-> NCCL all-reduce] -> flat Adamax) per second, whole job.
Workload: BASELINE config 3, Oberrhein feeder (N=70 buses, E=69 closed branches), B=4096 scenarios per GPU per step,
synthetic scenarios from the deterministic generator (dss2.synth; the reference's Oberrhein scenario pickles are missing
from its repository), random-init weights.  Weak scaling: every rank owns its own shard and batch.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]

Prints ONE JSON line on rank 0 (see the task's contract): value = device-resident throughput, e2e = through the host-buffer
API (pinned host scenarios -> H2D -> step -> D2H loss) inside the timed region, roofline = the dominant kernel (TAG-layer
backward) timed live with CUDA events against MEASURED_PEAKS.json, cpu_baseline = the oracle port of the reference path on
the host cores (bounded sample), clocks = SM clocks / throttle reasons sampled during the timed region.
"""
import argparse
import ctypes
import json
import os
import statistics
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
PKG = os.path.join(ROOT, "deep-statistical-solver-for-distribution-system-state-estimation_b200")
sys.path.insert(0, PKG)

REG = {"mu_v": 1e-1, "mu_theta": 1e-1, "lam_v": 1e-4, "lam_p": 1e-8, "lam_pf": 1e-6, "lam_reg": 1e2}
# BASELINE.json configs: name -> (grid loader key, default batch per GPU, default resident scenarios, description)
CONFIGS = {
    "ober": ("ober_sub", 4096, 16384, "ober_sub (N=70,E=69)"),                              # configs[2] / [3], the headline
    "cigre14": ("cigre14", 4096, 16384, "cigre14 (N=15,E=14)"),                             # configs[0]
    "reswitched": ("cigre14_reswitched", 4096, 16384, "cigre14_reswitched (N=15,E=15)"),    # configs[1]
    "feeder10k": ("ober_sub_x143", 32, 64, "10k-bus radial feeder (ober_sub x143 under one slack; N=9868,E=9867)"),   # configs[4]
}
NETWORKS = {"skippfn": "SkipPFN(8,6,2,32,8,2,0.3,5)", "gat": "GAT_DSSE(8,32,2,heads=1,num_layers=8,edge_dim=6)",
            "gine": "GINE_DSSE(8,32,2,num_layers=8,edge_dim=6)"}


def workload_string(args):
    what = ("train step: pack+fwd+WLS loss+bwd+Adamax" if args.mode == "train" else "inference: fwd+get_pflow")
    return f"{CONFIGS[args.config][3]} B={args.batch}/GPU {NETWORKS[args.network]} {what}"


def config_dict(args, n, e):
    """The workload description: identical in the `ours` and `reference` arms (nothing implementation specific in here)."""
    return {"workload": workload_string(args), "grid": CONFIGS[args.config][0], "network": NETWORKS[args.network], "mode": args.mode,
            "batch_per_gpu": args.batch, "nodes_per_step_per_gpu": args.batch * n, "edges_per_step_per_gpu": args.batch * e,
            "resident_scenarios_per_gpu": args.scenarios, "scenario_seed": 1234,
            "parallelism": f"dp{args.gpus}" if args.gpus > 1 else "single",
            "l2": "inputs larger than L2: the per-step working set (saved activations + scenario store, > 1 GB at the headline size) exceeds the 126 MB L2, no flush"}


def load_grid(config):
    from dss2 import synth
    key = CONFIGS[config][0]
    if key.startswith("ober_sub_x"):
        return synth.replicate_feeder(synth.load_grid("ober_sub"), int(key.split("x")[-1]))
    return synth.load_grid(key)


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", default="ober", choices=sorted(CONFIGS), help="BASELINE.json config (default: the headline, Oberrhein B=4096)")
    ap.add_argument("--exact-global-batch", action="store_true",
                    help="N > 1: train on ONE batch of N*B scenarios exactly (loss sums all-reduced between the loss passes, gradients summed) "
                         "instead of the default DDP mean of per-shard gradients")
    ap.add_argument("--network", "--model", dest="network", default="skippfn", choices=sorted(NETWORKS))
    ap.add_argument("--mode", default="train", choices=["train", "infer"])
    ap.add_argument("--batch", type=int, default=None)
    ap.add_argument("--scenarios", type=int, default=None, help="synthetic scenarios resident per GPU")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-graph", action="store_true", help="launch eagerly instead of replaying a CUDA graph")
    ap.add_argument("--same-shards", action="store_true", help="every rank uses rank 0's scenarios and ids (multi-GPU == single-GPU check)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last timed step computed as DIR/<name>.npy (rank 0), so that two builds "
                         "can be compared output for output on the same seeded inputs")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the outputs of --impl ours")
    if args.batch is None:
        args.batch = CONFIGS[args.config][1]
    if args.scenarios is None:
        args.scenarios = max(CONFIGS[args.config][2], args.batch)
    return args


# ---------------------------------------------------------------------------------------------------------------------
# CPU arm: the reference's own networks.py / data.py (verbatim copies in the git-ignored oracle/_ref, see
# tools/make_oracle_ref.sh) executed over oracle/pyg_shim on the host cores; the oracle port only when oracle/_ref is absent
# ---------------------------------------------------------------------------------------------------------------------
class CpuArm:
    """One step = the SAME workload as the GPU arm's step (same grid, network, mode and batch size) on the host cores."""

    def __init__(self, args, batch_graphs=None):
        import torch
        sys.path.insert(0, os.path.join(ROOT, "oracle"))
        import dss2_oracle as orc
        import ref_runner
        from dss2 import synth
        self.torch, self.orc, self.args = torch, orc, args
        self.cores = os.cpu_count() or 1
        torch.set_num_threads(self.cores)
        self.B = batch_graphs or args.batch
        store = synth.synthetic_store(load_grid(args.config), self.B, seed=1234)
        self.batch = orc.collate([store.graph(i) for i in range(self.B)])
        self.stats = (store.x_mean, store.x_std, store.edge_mean, store.edge_std)
        self.kind = "reference" if ref_runner.available() else "port"
        if self.kind == "reference":
            net, dat = ref_runner.load_reference(stub_laplacian=True)
            torch.manual_seed(0)
            if args.network == "skippfn":
                self.model = net.SkipPFN(8, 6, 2, 32, 8, 2, 0.3, 5)
            elif args.network == "gat":
                self.model = net.GAT_DSSE(dim_feat=8, dim_dense=32, dim_out=2, heads=1, num_layers=8, edge_dim=6)
            else:
                self.model = net.GINE_DSSE(dim_feat=8, dim_dense=32, dim_out=2, num_layers=8, edge_dim=6)
            self.dat = dat
            self.opt = torch.optim.Adamax(self.model.parameters(), lr=3e-3)     # dss2_run.py:91-92
        else:
            if args.network != "skippfn" or args.mode != "train":
                raise SystemExit("the oracle-port fallback of the CPU arm covers SkipPFN training only; run tools/make_oracle_ref.sh")
            self.sd = {k: v.requires_grad_(True) for k, v in orc.init_state_dict("SkipPFN", seed=0).items()}
            self.opt_state = {}

    def describe(self):
        if self.kind == "reference":
            return ("the reference's own networks.py + data.py (verbatim copies, oracle/_ref) over the torch_geometric stand-in oracle/pyg_shim, "
                    "eager torch on the host cores; data.get_laplacian stubbed (its dense O(Nt^2) result is discarded by the loss: 329 GB at this size)")
        return "oracle port of the reference's networks.py/data.py semantics (oracle/_ref absent), eager torch on the host cores"

    def step(self):
        torch, b, st = self.torch, self.batch, self.stats
        if self.kind != "reference":
            return self.orc.train_step(self.sd, b, {"x_mean": st[0], "x_std": st[1], "edge_mean": st[2], "edge_std": st[3]}, REG, 0.3, self.opt_state)
        x, ei, ea = b["x"], b["edge_index"], b["edge_attr"]
        if self.args.mode == "infer":                                    # dss2_run.py:177-194 (forward + get_pflow)
            self.model.eval()
            with torch.no_grad():
                out = self.model(x[:, :8], ei, ea[:, :6])
                est = torch.cat([out[:, 0:1] * st[1][:1] + st[0][:1], out[:, 1:] * (1. - x[:, 9:10])], 1)
                return self.dat.get_pflow(est, ei, node_param=x[:, 8:], edge_param=ea[:, 6:])[0]
        self.model.train()                                               # dss2_run.py:133-143
        self.opt.zero_grad()
        out = self.model(x[:, :8], ei, ea[:, :6])
        loss = self.dat.gsp_wls_edge(input=x[:, :8], edge_input=ea[:, :6], output=out, x_mean=st[0], x_std=st[1], edge_mean=st[2],
                                     edge_std=st[3], edge_index=ei, reg_coefs=REG, num_samples=None, node_param=x[:, 8:],
                                     edge_param=ea[:, 6:])
        loss.backward()
        self.opt.step()
        return loss

    def time_steps(self, steps, warmup):
        times = []
        for i in range(warmup + steps):
            t0 = time.perf_counter()
            self.step()
            if i >= warmup:
                times.append(time.perf_counter() - t0)
        total = sum(times)
        return self.B * len(times) / total, 1000.0 * total / len(times)


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    arm = CpuArm(args)
    n = arm.batch["x"].shape[0] // arm.B
    e = arm.batch["edge_attr"].shape[0] // arm.B
    # a full-size step is seconds of CPU work: one untimed step, then exactly --steps timed ones
    rate, ms = arm.time_steps(args.steps, 1)
    sample = f"{args.steps} timed steps of the full workload ({arm.B} scenarios per step) after 1 warm-up step; {arm.describe()}"
    line = {
        "impl": "reference", "metric": "train scenarios/s" if args.mode == "train" else "inference scenarios/s", "value": rate,
        "unit": "scenarios/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": 1, "ms_per_step": ms, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": config_dict(args, n, e),
        "cpu_baseline": {"value": rate, "unit": "scenarios/s", "cores": arm.cores, "kind": arm.kind, "sample": sample},
        "e2e": {"value": rate, "unit": "scenarios/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line))


# ---------------------------------------------------------------------------------------------------------------------
# --dump-outputs
# ---------------------------------------------------------------------------------------------------------------------
DUMP_BUDGET = 60 << 20   # bytes of array data in all: with the .npy headers the dump stays under 64 MB


def dump_outputs(out_dir, arrays):
    """Writes every tensor of `arrays` as out_dir/<name>.npy, float64 tensors as float64 and all others as float32.  Should the arrays
    exceed DUMP_BUDGET together, each one larger than an even share of it keeps a seeded random sample of its rows in their original
    order (of its entries, flattened, when one row alone exceeds the share): the same rows in every run with the same shapes, so dumps
    of two builds still compare entry for entry."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    host = {}
    for name, t in arrays.items():
        a = t.detach().cpu().numpy()
        host[name] = a if a.dtype == np.float64 else a.astype(np.float32)
    share = DUMP_BUDGET // len(host)
    sample = sum(a.nbytes for a in host.values()) > DUMP_BUDGET
    for name, a in host.items():
        if sample and a.nbytes > share:
            if a.nbytes // a.shape[0] > share:
                a = a.reshape(-1)
            rows = share // (a.nbytes // a.shape[0])
            a = a[np.sort(np.random.default_rng(0).choice(a.shape[0], rows, replace=False))]
        np.save(os.path.join(out_dir, f"{name}.npy"), a)


def named_parameters_flat(params):
    """{name: tensor} -> one vector, concatenated in the order of the sorted names: independent of how a build lays the parameters
    out in its flat buffer."""
    import torch
    return torch.cat([params[k].detach().reshape(-1) for k in sorted(params)])


# ---------------------------------------------------------------------------------------------------------------------
# clocks
# ---------------------------------------------------------------------------------------------------------------------
class ClockSampler(threading.Thread):
    """Samples SM clock and throttle reasons of one GPU through NVML while the timed region runs."""
    BAD = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown"}
    NOTE = {0x4: "sw_power_cap", 0x80: "hw_power_brake", 0x2: "applications_clocks_setting", 0x100: "display_clock_setting"}

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.stop_flag, self.samples, self.reasons, self.max_mhz = index, threading.Event(), [], set(), None

    def run(self):
        try:
            import pynvml
            pynvml.nvmlInit()
            h = pynvml.nvmlDeviceGetHandleByIndex(self.index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(h, pynvml.NVML_CLOCK_SM)
            while not self.stop_flag.is_set():
                self.samples.append(pynvml.nvmlDeviceGetClockInfo(h, pynvml.NVML_CLOCK_SM))
                mask = pynvml.nvmlDeviceGetCurrentClocksThrottleReasons(h)
                for bit, name in {**self.BAD, **self.NOTE}.items():
                    if mask & bit:
                        self.reasons.add(name)
                time.sleep(0.005)
        except Exception as exc:   # NVML missing: report that instead of inventing numbers
            self.reasons.add(f"nvml_unavailable:{type(exc).__name__}")

    def result(self):
        return {"sm_mhz": statistics.median(self.samples) if self.samples else None, "sm_max_mhz": self.max_mhz,
                "reasons": sorted(self.reasons), "samples": len(self.samples)}


# ---------------------------------------------------------------------------------------------------------------------
# GPU arm, secondary workloads: GAT_DSSE / GINE_DSSE training and inference through the drop-in modules (eager launches)
# ---------------------------------------------------------------------------------------------------------------------
def run_eager(args, dev, rank, world, local, K, W):
    import torch
    import data as d3
    import networks
    from dss2 import _lib, batching, synth
    if world > 1:
        raise SystemExit("--network gat/gine and --mode infer are single-GPU measurements (replicas only)")
    B = args.batch
    store = synth.synthetic_store(load_grid(args.config), args.scenarios, seed=1234, device=dev)
    n, e = store.max_nodes, store.max_edges
    batch = batching.pack_batch(store, torch.arange(B, device=dev))
    if args.network == "skippfn":
        model = networks.SkipPFN(dim_featn=8, dim_feate=6, dim_out=2, dim_hid=32, n_gnn_layers=8, K=2, dropout_rate=0.3, L=5)
    elif args.network == "gat":
        model = networks.GAT_DSSE(dim_feat=8, dim_dense=32, dim_out=2, heads=1, num_layers=8, edge_dim=6)
    else:
        model = networks.GINE_DSSE(dim_feat=8, dim_dense=32, dim_out=2, num_layers=8, edge_dim=6)
    model = model.to(dev)
    opt = torch.optim.Adamax(model.parameters(), lr=3e-3)
    stats = [t.to(dev) for t in (store.x_mean, store.x_std, store.edge_mean, store.edge_std)]
    x, ea, ei = batch.x, batch.edge_attr, batch.edge_index
    last = {}      # what the latest step handed its caller (for --dump-outputs)

    def step():
        if args.mode == "infer":                                   # dss2_run.py:177-194
            with torch.no_grad():
                out = model(x[:, :8], ei, ea[:, :6])
                est = torch.cat([out[:, 0:1] * stats[1][:1] + stats[0][:1], out[:, 1:] * (1. - x[:, 9:10])], 1)
                pflow = d3.get_pflow(est, ei, node_param=x[:, 8:], edge_param=ea[:, 6:])
                last.update(output=out, pflow=pflow)
                return pflow[0].sum()
        opt.zero_grad(set_to_none=True)                            # dss2_run.py:137-143
        out = model(x[:, :8], ei, ea[:, :6])
        loss = d3.gsp_wls_edge(input=x[:, :8], edge_input=ea[:, :6], output=out, x_mean=stats[0], x_std=stats[1], edge_mean=stats[2],
                               edge_std=stats[3], edge_index=ei, reg_coefs=REG, num_samples=None, node_param=x[:, 8:], edge_param=ea[:, 6:])
        loss.backward()
        opt.step()
        return loss

    if args.mode == "infer":
        model.eval()
    for _ in range(W):
        step()
    torch.cuda.synchronize()
    sampler = ClockSampler(local)
    sampler.start()
    n0 = _lib.launch_count()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(K):
        res = step()
    b.record()
    b.synchronize()
    sampler.stop_flag.set()
    sampler.join()
    ms = a.elapsed_time(b)
    launches = _lib.launch_count() - n0
    if args.dump_outputs:   # inference (training runs through GraphedTrainer in main); pflow columns: loading_lines, loading_trafo,
        # P_from, Q_from, P_to, Q_to, I_from, I_to
        dump_outputs(args.dump_outputs, {"output": last["output"], "pflow": torch.stack(last["pflow"], dim=1)})
    # end to end: the batch's features come from pinned host memory every step, the scalar result goes back
    hx, hea = x.cpu().pin_memory(), ea.cpu().pin_memory()
    hres = torch.zeros(1).pin_memory()
    a2, b2 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    a2.record()
    for _ in range(K):
        x.copy_(hx, non_blocking=True)
        ea.copy_(hea, non_blocking=True)
        hres.copy_(step().reshape(1).float(), non_blocking=True)
    b2.record()
    b2.synchronize()
    ms2 = a2.elapsed_time(b2)
    cpu = None
    if not args.no_cpu_baseline:
        CpuArm(args, batch_graphs=min(256, B)).time_steps(1, 0)
        arm = CpuArm(args)
        rate, cms = arm.time_steps(2, 0)
        cpu = {"value": rate, "unit": "scenarios/s", "cores": arm.cores, "kind": arm.kind, "ms_per_step": cms,
               "sample": f"2 timed steps of the full workload ({B} scenarios per step) after a 256-scenario warm-up step; " + arm.describe()}
    line = {
        "metric": "train scenarios/s" if args.mode == "train" else "inference scenarios/s", "value": B * K / (ms / 1e3), "unit": "scenarios/s",
        "n_gpus": 1, "steps": K, "warmup": W, "ms_per_step": ms / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic", "config": config_dict(args, n, e),
        "impl_detail": {"cuda_graph": False, "path": "drop-in modules (networks / data), eager launches, torch.optim.Adamax"},
        "e2e": {"value": B * K / (ms2 / 1e3), "unit": "scenarios/s", "h2d_bytes_per_step": (hx.numel() + hea.numel()) * 4, "d2h_bytes_per_step": 4,
                "ms_per_step": ms2 / K, "api": "model(...) / gsp_wls_edge / get_pflow of the drop-in modules on a batch refreshed from pinned host memory"},
        "gpu_launches": int(launches), "launches_per_step": launches / K, "roofline": None, "cpu_baseline": cpu, "clocks": sampler.result(),
        "final_loss": float(res),
    }
    print(json.dumps(line), flush=True)


# ---------------------------------------------------------------------------------------------------------------------
# GPU arm
# ---------------------------------------------------------------------------------------------------------------------
def main():
    args = parse()
    if args.impl == "reference":
        return run_reference(args)

    import torch
    import torch.distributed as dist
    from dss2 import _lib, synth
    from dss2.dataset import ScenarioStore
    from dss2.trainer import GraphedTrainer, default_spec

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the hot path has no CPU fallback (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    pg = None
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)
        pg = dist.group.WORLD
    K, W, B = args.steps, max(args.warmup, 3), args.batch

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    def max_over_ranks(v):
        t = torch.tensor([v], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    if args.mode != "train":
        return run_eager(args, dev, rank, world, local, K, W)
    grid = load_grid(args.config)
    shard = 0 if args.same_shards else rank
    store = synth.synthetic_store(grid, args.scenarios, seed=1234 + shard, device=dev)
    n, e = store.max_nodes, store.max_edges
    spec = default_spec() if args.network == "skippfn" else None      # gat / gine: the constructor arguments of dss2_run.py:73-86
    trainer = GraphedTrainer(store, B, spec=spec, reg_coefs=REG, seed=0, process_group=pg, world_size=world, network=args.network,
                             use_cuda_graph=not args.no_graph, dropout_stream=0 if args.same_shards else None,
                             exact_global_batch=args.exact_global_batch).capture()
    gen = torch.Generator().manual_seed(99 + shard)
    ids_host = torch.randint(0, args.scenarios, (W + K, B), generator=gen).pin_memory()

    # ---- device-resident throughput: scenarios already in HBM, ids copied per step (32 KB) ----
    for i in range(W):
        trainer.step(ids_host[i])
    barrier()
    sampler = ClockSampler(local)
    sampler.start()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.profiler.start()      # lets `ncu --profile-from-start off` see exactly the timed steps
    loss_hist = torch.zeros(K, dtype=torch.float32, device=dev)
    ev0.record()
    for i in range(K):
        trainer.step(ids_host[W + i])
        loss_hist[i:i + 1].copy_(trainer.loss.reshape(1), non_blocking=True)     # 4-byte device copy: the loss trajectory, for the hash below
    ev1.record()
    barrier()
    torch.cuda.profiler.stop()
    sampler.stop_flag.set()
    sampler.join()
    ms_total = max_over_ranks(ev0.elapsed_time(ev1))
    loss_end = float(trainer.loss.item())
    if args.dump_outputs and rank == 0:   # before the kernel timings below reuse the trainer's buffers
        dump_outputs(args.dump_outputs, {"loss": trainer.loss, "loss_per_step": loss_hist,
                                         "parameters": named_parameters_flat(trainer.state_dict())})
    value = world * B * K / (ms_total / 1e3)
    # data-parallel sanity, outside the timed region: every replica must hold bit-identical parameters after the K steps (same
    # all-reduced gradient, same update), and with --same-shards the loss trajectory must be the one a single GPU produces
    import hashlib
    loss_sha = hashlib.sha256(loss_hist.cpu().numpy().tobytes()).hexdigest()[:16]
    sync = None
    if world > 1:
        ref_flat = trainer.flat.clone()
        dist.broadcast(ref_flat, src=0)
        sync = {"replicas_in_sync": max_over_ranks(float((trainer.flat - ref_flat).abs().max().item())) == 0.0,
                "max_abs_param_diff_vs_rank0": max_over_ranks(float((trainer.flat - ref_flat).abs().max().item()))}

    roofline, tiled = None, trainer.graph.c.num_tiles > 0
    from dss2 import ops as _ops
    if args.network == "skippfn":   # per-kernel roofline of the SkipPFN step (GAT / GINE: thread-per-bus kernels, whole-step figure only)
        # ---- layer kernels timed live on the launching stream (hidden layer 32 -> 32, K = 2, the shapes of 35 of the 40 TAG layers) ----
        lib, P = _lib.load(), _lib.ptr
        from dss2 import ops as _ops
        sp, run, bufs = trainer.spec, trainer.runner, trainer.bufs
        nt, et = trainer.nt, trainer.et
        name_w, name_b = "mpns.0.convs.3.lins.0.weight", "mpns.0.convs.3.bias"
        w_off, b_off = run.table[name_w][0], run.table[name_b][0]
        part_w = ctypes.c_void_p(bufs["partials"].data_ptr() + 4 * w_off)
        gref, st_ = trainer.graph.ref, _lib.stream
        x_l, y_l, bits_l = bufs["acts"][0, 3], bufs["acts"][0, 4], bufs["bits"][0, 3]
        gy_l, gx_l, lvl = bufs["g32"][0], bufs["g32"][1], bufs["lvl"]
        wp, bp = run._p(trainer.flat, name_w), run._p(trainer.flat, name_b)
        tiled = trainer.graph.c.num_tiles > 0
        tc2 = tiled and _ops.TAG_IMPL == "tc2" and bool(lib.dss2_tag_tc2_supported(gref, sp.K))
        kernels = {}
        if tc2:
            kernels["k_tag_tc3<BGX> (TAG backward-to-input, tcgen05, TMA-fed)"] = (lambda: _lib.check(lib.dss2_tag_bwd_tc2_gx(
                gref, wp, 32, sp.K, 1, sp.p_drop, P(bits_l), P(gy_l), P(gx_l), P(lvl), lvl.numel() * 4, st_()), "gx"),
                nt * (128 + 128 + 4 + 24), "grad_y + sign word + ELL topology in, grad_x out; excludes the 256 B/node hop-level spill it writes for k_tag_gw")
            kernels["k_tag_tc3<FWD> (TAG forward, tcgen05, TMA-fed)"] = (lambda: _lib.check(lib.dss2_tag_fwd_tc2(
                gref, P(x_l), wp, bp, 32, sp.K, 1, sp.p_drop, 1, P(trainer.step_state), 3, None, None, 0, P(y_l), P(bits_l), st_()), "fwd"),
                nt * (128 + 128 + 4 + 24), "x + ELL topology in, y + sign word out")
            in_step = " [in the step]"
            kernels["k_tag_gw (TAG weight gradients, tcgen05 MN-major, TMA ring)" + (in_step if _ops.GW_IMPL == "tc" else " [alternative]")] = (
                lambda: _lib.check(lib.dss2_tag_bwd_tc2_gw(
                    nt, P(x_l), 32, sp.K, 1, sp.p_drop, P(bits_l), P(gy_l), part_w, run.flat_size, b_off - w_off, P(lvl), lvl.numel() * 4, st_()), "gw"),
                nt * (128 + 128 + 4), "x + grad_y + sign word in; excludes the 256 B/node hop levels it re-reads")
            kernels["k_tag_gw_ffma (TAG weight gradients, exact fp32 FFMA, TMA ring)" + (in_step if _ops.GW_IMPL != "tc" else " [alternative]")] = (
                lambda: _lib.check(lib.dss2_tag_gw_ffma(
                    nt, P(x_l), 32, sp.K, 1, sp.p_drop, P(bits_l), P(gy_l), part_w, run.flat_size, b_off - w_off, P(lvl), lvl.numel() * 4, st_()), "gwf"),
                nt * (128 + 128 + 4), "x + grad_y + sign word in; excludes the 256 B/node hop levels it re-reads")
        elif tiled:
            kernels["k_tag_bwd<2,32> (TAG backward, CUDA cores)"] = (lambda: _lib.check(lib.dss2_tag_bwd(
                gref, P(x_l), wp, 32, sp.K, 1, sp.p_drop, P(bits_l), P(gy_l), P(gx_l), part_w, run.flat_size, b_off - w_off, st_()), "bwd"),
                nt * (3 * 128 + 4) + 4 * (nt + 1) + 16 * et, "x, grad_y in, grad_x out, sign word, CSR")
            kernels["k_tag_fwd<2> (TAG forward, CUDA cores)"] = (lambda: _lib.check(lib.dss2_tag_fwd(
                gref, P(x_l), wp, bp, 32, sp.K, 1, sp.p_drop, 1, P(trainer.step_state), 3, None, None, 0, P(y_l), P(bits_l), st_()), "fwd"),
                nt * (2 * 128 + 4) + 4 * (nt + 1) + 16 * et, "x in, y out, sign word, CSR")

        # EdgeAggregation of sub-net 1 (input = the previous sub-net's 8-wide output, gradient to the input and skip path needed)
        pre1 = "mpns.1.edge_aggr.edge_aggr."
        ea_w = [run._p(trainer.flat, pre1 + n_) for n_ in ("0.weight", "0.bias", "2.weight", "2.bias")]
        ea_part = ctypes.c_void_p(bufs["partials"].data_ptr() + 4 * run.table[pre1 + "0.weight"][0])
        x_in, eattr = bufs["outs"][0], trainer.batch["edge_attr"]
        ea_fwd_bytes = 32 * nt + 52 * et + 16 * et + 128 * nt
        if run.ea_slots(trainer.graph, 11, 13):   # the step's path: weights prepared once per step, thread-per-row kernels read slot 1
            run.ea_upload(trainer.flat)
            kernels["k_ea_row_fwd (EdgeAggregation forward, thread per bus, FFMA2)"] = (lambda: _lib.check(lib.dss2_edgeagg_fwd_slot(
                gref, P(x_in), sp.fn, sp.fn, P(eattr), 13, sp.fe, 1, P(bufs["acts"][1, 0]), st_()), "ea_fwd"),
                ea_fwd_bytes, "SURVEY 8(d): x row 32 + out row 128 per bus, edge_attr row 52 + edge_index 16 per branch")
            kernels["k_ea_row_bwd (EdgeAggregation backward: grad_x + parameter gradients)"] = (lambda: _lib.check(lib.dss2_edgeagg_bwd_slot(
                gref, P(x_in), sp.fn, sp.fn, P(eattr), 13, sp.fe, 1, P(gy_l), P(bufs["gsub"][0]), sp.fn, P(bufs["gsub"][1]), ea_part,
                run.flat_size, st_()), "ea_bwd"),
                ea_fwd_bytes + 32 * nt, "SURVEY 8(d): forward bytes with grad_out in place of out, + grad_x row 32 per bus")
        else:
            kernels["k_edgeagg_fwd (EdgeAggregation forward)"] = (lambda: _lib.check(lib.dss2_edgeagg_fwd(
                gref, P(x_in), sp.fn, sp.fn, P(eattr), 13, sp.fe, *ea_w, P(bufs["acts"][1, 0]), st_()), "ea_fwd"),
                ea_fwd_bytes, "SURVEY 8(d): x row 32 + out row 128 per bus, edge_attr row 52 + edge_index 16 per branch")
            kernels["k_edgeagg_bwd (EdgeAggregation backward: grad_x + parameter gradients)"] = (lambda: _lib.check(lib.dss2_edgeagg_bwd(
                gref, P(x_in), sp.fn, sp.fn, P(eattr), 13, sp.fe, *ea_w, P(gy_l), P(bufs["gsub"][0]), sp.fn, P(bufs["gsub"][1]), ea_part,
                run.flat_size, st_()), "ea_bwd"),
                ea_fwd_bytes + 32 * nt, "SURVEY 8(d): forward bytes with grad_out in place of out, + grad_x row 32 per bus")

        # the fused loss (2 kernels: reduction pass + gradient pass), on the trainer's own buffers
        kernels["k_wls<false>+k_wls<true> (branch flows + WLS loss, forward and backward)"] = (lambda: _lib.check(lib.dss2_wls_fwd_bwd(
            gref, P(trainer.batch["x"]), 11, P(trainer.batch["edge_attr"]), 13, P(bufs["outs"][-1]), P(trainer.stats), REG["lam_v"], REG["lam_p"],
            REG["lam_pf"], REG["lam_reg"], P(trainer.batch["vminmax"]), 1, P(trainer.loss), None, P(trainer.grad_out), P(trainer.wls_ws),
            trainer.wls_ws.numel(), st_()), "wls"), 60 * nt + 68 * et,
            "SURVEY 8(d), fused forward+backward: x row 44 + out 8 + grad_out 8 per bus, edge_attr row 52 + edge_index 16 per branch, counted ONCE "
            "(the two passes of the kernel pair re-read them; the second read mostly hits L2)")
        # the batch packer (PyG collate): reads the selected scenarios, writes the batch
        from dss2.batching import launch_pack as _launch_pack
        kernels["k_pack_scan+k_pack_copy (batch packer = PyG collate)"] = (
            lambda: _launch_pack(trainer.store, trainer.ids, trainer.batch, nt, et), 2 * (44 * nt + 52 * et + 8 * nt) + 16 * et + 8 * nt,
            "x 44 + y 8 per bus and edge_attr 52 per branch read and written, edge_index 16 per branch and batch vector 8 per bus written")

        def time_kernel(fn, reps=30):
            flush = torch.empty(256 * 1024 * 1024 // 4, dtype=torch.float32, device=dev)   # 256 MB > 126 MB L2
            durs = []
            for _ in range(3):
                fn()
            for _ in range(reps):
                flush.zero_()
                a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                a.record()
                fn()
                b.record()
                b.synchronize()
                durs.append(a.elapsed_time(b))
            return statistics.mean(durs) * 1e-3

        peaks_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
        if os.path.exists(peaks_path):
            peak, peak_src = float(json.load(open(peaks_path))["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
        else:
            peak, peak_src = 6650.0, "fallback (B200_PROFILING.md)"
        traffic_tab = {}
        tpath = os.path.join(ROOT, "profiles", "dominant_kernel_traffic.json")
        if os.path.exists(tpath):
            traffic_tab = json.load(open(tpath))
        n_tag = sp.L * sp.n_layers

        def launches_per_step(kname):   # how often the step launches this kernel (shape of the timed launch: hidden layer / sub-net 1)
            if kname.startswith("k_tag_"):
                return n_tag
            return sp.L if kname.startswith(("k_edgeagg", "k_ea_row")) else 1

        timed = []
        for kname, (fn, nbytes, what) in kernels.items():
            t = time_kernel(fn)
            timed.append({"kernel": kname, "us_per_launch": t * 1e6, "launches_per_step": launches_per_step(kname),
                          "algorithmic_bytes_per_launch": nbytes, "bytes_counted": what,
                          "achieved": nbytes / t / 1e9, "frac": nbytes / t / 1e9 / peak, "traffic": traffic_tab.get(kname.split(" ")[0])})
        # dominant = largest share of the step (duration x launches per step)
        dom = max((r for r in timed if "[alternative]" not in r["kernel"]), key=lambda r: r["us_per_launch"] * r["launches_per_step"])
        roofline = {"bound": "hbm", "kernel": dom["kernel"], "achieved": dom["achieved"], "peak": peak, "unit": "GB/s", "frac": dom["frac"],
                    "traffic": dom["traffic"], "peak_source": peak_src, "us_per_launch": dom["us_per_launch"],
                    "algorithmic_bytes_per_launch": dom["algorithmic_bytes_per_launch"], "bytes_counted": dom["bytes_counted"],
                    "note": "layer kernels are bound by the per-tile dependency chain (shared-memory gathers, barriers, tcgen05 issue), not by HBM: "
                            "see DESIGN.md section 4 and profiles/",
                    "all_layer_kernels": timed}
        # whole-step view with SURVEY.md 8(d)'s per-layer algorithmic bytes (topology counted as 0: per-topology template)
        hid, fn = 32, sp.fn
        step_bytes = 60 * nt + 68 * et                                           # fused loss (SURVEY 8d)
        for s_ in range(sp.L):
            cin0 = 44 if s_ == 0 else 4 * fn                                     # EdgeAggregation reads the 11-wide x rows in sub-net 0
            step_bytes += (cin0 * nt + 52 * et + 16 * et + 4 * hid * nt) + (cin0 * nt + 52 * et + 16 * et + 4 * hid * nt + (4 * fn * nt if s_ else 0))
            for l_ in range(sp.n_layers):
                cout_ = (sp.dim_out if s_ == sp.L - 1 else fn) if l_ == sp.n_layers - 1 else hid
                step_bytes += 4 * nt * (hid + cout_) + 4 * nt * (2 * hid + cout_)  # TAG forward + recompute-style backward
        roofline["step"] = {"algorithmic_bytes_per_step": step_bytes, "achieved": step_bytes / (ms_total / K / 1e3) / 1e9, "unit": "GB/s",
                            "frac": step_bytes / (ms_total / K / 1e3) / 1e9 / peak,
                            "definition": "SURVEY.md 8(d): loss 60 Nt + 68 Et; EdgeAggregation fwd+bwd; TAG 4 Nt (Cin+Cout) fwd + 4 Nt (2 Cin+Cout) bwd per layer"}

    # ---- end to end through the host-buffer API: pinned host scenarios -> H2D -> step -> D2H loss, all inside the timed region ----
    e2e = None
    if not args.no_e2e:
        # Two slots of B scenarios in ONE staging store: step i trains on slot i % 2 (selected by the scenario ids the packer gathers)
        # while a copy stream lands step i+1's scenarios in the other slot - the input pipeline a user of the API would write.
        slots = 2 if args.scenarios >= 2 * B else 1
        SB = slots * B
        stage = ScenarioStore(x=torch.empty(SB * n, 11, device=dev), edge_attr=torch.empty(SB * e, 13, device=dev),
                              y=torch.zeros(SB * n, 2, device=dev), edge_index=store.edge_index[:, :SB * e].contiguous(),
                              node_off=store.node_off[:SB + 1].contiguous(), edge_off=store.edge_off[:SB + 1].contiguous(),
                              x_mean=store.x_mean, x_std=store.x_std, edge_mean=store.edge_mean, edge_std=store.edge_std,
                              max_nodes=n, max_edges=e)
        stage.x.copy_(store.x[:SB * n])
        stage.edge_attr.copy_(store.edge_attr[:SB * e])
        t2 = GraphedTrainer(stage, B, spec=spec, reg_coefs=REG, seed=0, process_group=pg, world_size=world, network=args.network,
                            use_cuda_graph=not args.no_graph, exact_global_batch=args.exact_global_batch).capture()
        nbuf = max(1, min(4, args.scenarios // B))
        host_x = [store.x[i * B * n:(i + 1) * B * n].cpu().pin_memory() for i in range(nbuf)]
        host_ea = [store.edge_attr[i * B * e:(i + 1) * B * e].cpu().pin_memory() for i in range(nbuf)]
        host_loss = torch.zeros(K + W, dtype=torch.float32).pin_memory()
        slot_ids = [torch.arange(B, device=dev) + sl * B for sl in range(slots)]
        copy_stream = torch.cuda.Stream(device=dev)
        slot_free = [torch.cuda.Event() for _ in range(slots)]     # the last step that read the slot has finished
        slot_ready = [torch.cuda.Event() for _ in range(slots)]    # the slot's H2D copies have landed

        def feed(i):   # host -> device copy of step i's scenarios
            sl = i % slots
            with torch.cuda.stream(copy_stream):
                copy_stream.wait_event(slot_free[sl])
                stage.x[sl * B * n:(sl + 1) * B * n].copy_(host_x[i % nbuf], non_blocking=True)
                stage.edge_attr[sl * B * e:(sl + 1) * B * e].copy_(host_ea[i % nbuf], non_blocking=True)
                slot_ready[sl].record(copy_stream)

        def e2e_step(i):
            sl = i % slots
            if slots == 1:
                feed(i)
            else:
                feed(i + 1)                                  # overlaps this step's compute
            torch.cuda.current_stream().wait_event(slot_ready[sl])
            t2.step(slot_ids[sl])
            slot_free[sl].record()
            host_loss[i:i + 1].copy_(t2.loss.reshape(1), non_blocking=True)

        if slots == 2:
            feed(0)
        for i in range(W):
            e2e_step(i)
        barrier()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for i in range(K):
            e2e_step(W + i)
        b.record()
        barrier()
        ms_e2e = max_over_ranks(a.elapsed_time(b))
        e2e = {"value": world * B * K / (ms_e2e / 1e3), "unit": "scenarios/s", "h2d_bytes_per_step": (B * n * 11 + B * e * 13) * 4,
               "d2h_bytes_per_step": 4, "ms_per_step": ms_e2e / K, "api": "GraphedTrainer.step on a staging store fed from pinned host memory; " +
               ("two slots, the H2D copy of step i+1 runs on a copy stream while step i computes" if slots == 2 else "one slot, copies serialised"),
               "h2d_copies_in_timed_region": K}

    # ---- CPU baseline (rank 0, N = 1 only): bounded sample = 1 small warm-up step + 2 full-size steps of the same workload ----
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        CpuArm(args, batch_graphs=min(256, B)).time_steps(1, 0)          # warms the torch CPU kernels up
        arm = CpuArm(args)
        rate, ms = arm.time_steps(2, 0)
        cpu = {"value": rate, "unit": "scenarios/s", "cores": arm.cores, "kind": arm.kind, "ms_per_step": ms,
               "sample": f"2 timed steps of the full workload ({B} scenarios per step: fwd+loss+bwd+Adamax) after a 256-scenario warm-up step; " + arm.describe()}

    if rank == 0:
        line = {
            "metric": "train scenarios/s", "value": value, "unit": "scenarios/s", "n_gpus": world, "steps": K, "warmup": W,
            "ms_per_step": ms_total / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": config_dict(args, n, e),
            "impl_detail": {"cuda_graph": not args.no_graph, "tag_impl": _ops.TAG_IMPL, "tiled": bool(tiled),
                            "tc3": os.environ.get("DSS2_TC3", "1") != "0"},
            "loss_trajectory_sha256_16": loss_sha, "data_parallel_check": sync,
            "data_parallel_mode": ("exact global batch (loss sums all-reduced between the loss passes, gradients summed)" if args.exact_global_batch
                                   else "mean of per-shard gradients (DDP semantics)") if world > 1 else None,
            "e2e": e2e, "gpu_launches": int(trainer.launches_per_step) * K, "launches_per_step": int(trainer.launches_per_step),
            "roofline": roofline, "cpu_baseline": cpu, "clocks": sampler.result(), "final_loss": loss_end,
        }
        print(json.dumps(line), flush=True)
    if world > 1:
        # a process group that has collectives captured in live CUDA graphs can hang in destroy_process_group(): leave together, hard
        torch.cuda.synchronize()
        dist.barrier()
        sys.stdout.flush()
        sys.stderr.flush()
        os._exit(0)


if __name__ == "__main__":
    main()
