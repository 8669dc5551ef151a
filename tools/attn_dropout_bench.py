"""Cost of the attention dropout of GAT_DSSE and gnn_dsse(model='fagcn') on the device, at the workload bench.py uses (ober_sub,
B = 4096 scenarios): the captured GraphedTrainer(network='gat') step and the eager drop-in gnn_dsse(model='fagcn') training step
(forward, gsp_wls_edge, backward, torch.optim.Adamax), each at dropout 0 and 0.1.  The two settings of a model alternate over the
repeats, every repeat is timed with CUDA events around `steps` steps, and the median is reported.

usage (GPU box): python tools/attn_dropout_bench.py out_dir [B] [steps] [repeats]   -> out_dir/attn_dropout.json"""
import json
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "deep-statistical-solver-for-distribution-system-state-estimation_b200"))
import torch

import data as d3
import networks
from dss2 import batching, synth
from dss2.gat import GATSpec
from dss2.trainer import GraphedTrainer

REG = {"mu_v": 1e-1, "mu_theta": 1e-1, "lam_v": 1e-4, "lam_p": 1e-8, "lam_pf": 1e-6, "lam_reg": 1e2}
if len(sys.argv) < 2:
    raise SystemExit(__doc__)
OUT = sys.argv[1]
B = int(sys.argv[2]) if len(sys.argv) > 2 else 4096
STEPS = int(sys.argv[3]) if len(sys.argv) > 3 else 50
REPEATS = int(sys.argv[4]) if len(sys.argv) > 4 else 7
P_VALUES = (0.0, 0.1)


def timed(step, n):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(n):
        step()
    b.record()
    b.synchronize()
    return a.elapsed_time(b) / n


def measure(steps_by_p):
    for step in steps_by_p.values():      # warm-up of every shape the timed window uses
        for _ in range(3):
            step()
    torch.cuda.synchronize()
    ms = {p: [] for p in steps_by_p}
    for _ in range(REPEATS):
        for p, step in steps_by_p.items():
            ms[p].append(timed(step, STEPS))
    return {f"dropout={p}": {"ms_per_step_median": statistics.median(v), "ms_per_step_all": v} for p, v in ms.items()}


store = synth.synthetic_store(synth.load_grid("ober_sub"), B, seed=3, device="cuda")
ids = torch.arange(B, device="cuda")

trainers = {}
for p in P_VALUES:
    spec = GATSpec(dim_feat=8, dim_dense=32, dim_out=2, num_layers=8, edge_dim=6, dropout=p)
    trainers[p] = GraphedTrainer(store, B, spec=spec, reg_coefs=REG, seed=0, network="gat").capture()
gat = measure({p: (lambda t=t: t.step(ids)) for p, t in trainers.items()})
del trainers

batch = batching.pack_batch(store, ids)
stats = [t.cuda() for t in (store.x_mean, store.x_std, store.edge_mean, store.edge_std)]


def fagcn_step(p):
    torch.manual_seed(0)
    model = networks.gnn_dsse(dim_feat=8, dim_dense=32, dim_out=2, num_layers=8, model="fagcn", dropout=p).cuda().train()
    opt = torch.optim.Adamax(model.parameters(), lr=3e-3)

    def step():
        opt.zero_grad(set_to_none=True)
        out = model(batch.x[:, :8], batch.edge_index)
        loss = d3.gsp_wls_edge(input=batch.x[:, :8], edge_input=batch.edge_attr[:, :6], output=out, x_mean=stats[0], x_std=stats[1],
                               edge_mean=stats[2], edge_std=stats[3], edge_index=batch.edge_index, reg_coefs=REG, num_samples=None,
                               node_param=batch.x[:, 8:], edge_param=batch.edge_attr[:, 6:])
        loss.backward()
        opt.step()
    return step


fagcn = measure({p: fagcn_step(p) for p in P_VALUES})
smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True).stdout
res = {"device": torch.cuda.get_device_name(0), "nvidia_smi_name_power_limit_max_sm_clock": smi.strip(), "workload": f"ober_sub B={B}",
       "steps_per_repeat": STEPS, "repeats": REPEATS, "timing": "CUDA events around each repeat, the two dropout settings alternating",
       "GraphedTrainer(network='gat') captured step": gat,
       "gnn_dsse(model='fagcn', num_layers=8) eager drop-in step (forward, gsp_wls_edge, backward, Adamax)": fagcn}
os.makedirs(OUT, exist_ok=True)
with open(os.path.join(OUT, "attn_dropout.json"), "w") as f:
    json.dump(res, f, indent=1)
print(json.dumps(res))
