"""Device-resident training step: packer -> SkipPFN forward -> fused WLS loss fwd+bwd -> backward -> (all-reduce) ->
flat Adamax, launched straight through the C ABI over static buffers and replayed as ONE CUDA graph.

This is the throughput path (what `bench.py` measures); it issues exactly the same kernels as the drop-in
`networks` / `data` modules but skips autograd and per-step allocation.  It mirrors one iteration of the
reference's training loop (dss2_run.py:134-144): `optimizer.zero_grad(); out = model(...); loss = gsp_wls_edge(...);
loss.backward(); optimizer.step()` with Adamax(lr=3e-3) (dss2_run.py:91-92) and the always-on dropout
(networks.py:268) drawn in-kernel from a counter-based generator keyed by (seed, step).

Data parallelism (SURVEY.md 8e): every rank owns a shard of the scenarios and packs its own batch; the only
exchange is one sum all-reduce of the flat fp32 gradient (~484 KB for the default SkipPFN) per step, followed by
the identical Adamax update on every rank with the gradient scaled by 1/world_size ("mean of per-shard
gradients", i.e. DDP semantics - the loss's squared batch means make sharding inexact w.r.t. one large batch).
"""
import os

import torch

from . import _lib
from .batching import launch_pack
from .graph import BatchGraph
from .ops import ParamPack, PFNRunner, PFNSpec


def default_spec(p_drop=0.3, L=5, n_layers=8, K=2, dim_out=2, fn=8, fe=6):
    """SkipPFN(8, 6, 2, 32, 8, 2, 0.3, 5): dss2_run.py:72-82,88."""
    return PFNSpec(fn=fn, fe=fe, dim_out=dim_out, n_layers=n_layers, K=K, L=L, p_drop=p_drop,
                   skip=tuple(s < L - 1 for s in range(L)), prefix_fmt="mpns.{s}.")


def make_runner(network, spec=None):
    """(runner, spec, torch module factory) of a model family: 'skippfn' (any PFNSpec: MPN / SkipMPN / PFN / SkipPFN), 'gat' = GAT_DSSE
    (the script's as-shipped model, dss2_run.py:86), 'gine' = GINE_DSSE.  All three runners share forward / backward over static buffers
    and a flat parameter buffer whose first `flat_size` floats are the parameters."""
    if network == "skippfn":
        spec = spec or default_spec()
        return PFNRunner(spec), spec
    if network == "gat":
        from .gat import GATRunner, GATSpec
        spec = spec or GATSpec(dim_feat=8, dim_dense=32, dim_out=2, num_layers=8, edge_dim=6)
        return GATRunner(spec), spec
    if network == "gine":
        from .gine import GINERunner, GINESpec
        spec = spec or GINESpec(dim_feat=8, dim_dense=32, dim_out=2, num_layers=8, edge_dim=6)
        return GINERunner(spec), spec
    raise ValueError(f"GraphedTrainer: unknown network {network!r}")


# N > 1: DSS2_BUCKETED_ALLREDUCE=1 all-reduces the gradient per sub-net under the backward of the next one instead of once after the
# backward (measured at N = 2: 6.133 vs 6.084 ms per step - the five NCCL kernels displace CTAs of the chained backward; off by default)
BUCKETED_ALLREDUCE = os.environ.get("DSS2_BUCKETED_ALLREDUCE", "0") != "0"

class GraphedTrainer:
    def __init__(self, store, batch_graphs, spec=None, reg_coefs=None, lr=3e-3, seed=0, init_state_dict=None,
                 process_group=None, world_size=1, use_cuda_graph=True, dropout_stream=None, network="skippfn", exact_global_batch=False):
        """seed: parameter initialisation (all ranks must agree; rank 0's parameters are broadcast anyway).
        dropout_stream: index of this replica's dropout stream (default: its rank, so that every shard draws its own masks;
        pass the same value on all ranks to reproduce a single-GPU run on identical shards).
        network: 'skippfn' (default, any PFNSpec), 'gat', 'gine' - see make_runner.
        exact_global_batch (world_size > 1): the R ranks train on ONE batch of R*B scenarios exactly - the loss's batch sums and counts are
        all-reduced between the two loss passes (7 doubles) and the parameter gradients are summed; default (False) = DDP semantics, the mean
        of the ranks' per-shard gradients (the loss squares batch means, data.py:453-455, so the two differ)."""
        self.lib = _lib.load()
        self.network = network
        self.runner, self.spec = make_runner(network, spec)
        self.store = store
        self.B = int(batch_graphs)
        self.dev = store.x.device
        if self.dev.type != "cuda":
            raise _lib.Dss2Error("GraphedTrainer needs a CUDA-resident ScenarioStore")
        if store.x.size(0) != store.num_scenarios * store.max_nodes:
            raise _lib.Dss2Error("GraphedTrainer needs a uniform-topology store (static batch shapes)")
        self.pg, self.world = process_group, int(world_size)
        self.exact = bool(exact_global_batch) and self.world > 1
        self.lr = float(lr)
        rc = reg_coefs or {"lam_v": 1e-4, "lam_p": 1e-8, "lam_pf": 1e-6, "lam_reg": 1e2}   # dss2_run.py:104-112
        self.coefs = (float(rc["lam_v"]), float(rc["lam_p"]), float(rc["lam_pf"]), float(rc["lam_reg"]))
        n, e = store.max_nodes, store.max_edges
        self.nt, self.et = self.B * n, self.B * e
        f32 = dict(dtype=torch.float32, device=self.dev)
        i64 = dict(dtype=torch.long, device=self.dev)
        with torch.cuda.device(self.dev):
            # parameters: same init distribution as the reference modules, one flat buffer
            self.flat = torch.zeros(self.runner.flat_size, **f32)
            self._init_params(seed, init_state_dict)
            # gradient buffer: the parameters' gradients first; GINE keeps per-layer shares of its shared Linear behind them
            self.flat_grad = torch.zeros(getattr(self.runner, "grad_size", self.runner.flat_size), **f32)
            self.exp_avg = torch.zeros_like(self.flat)
            self.exp_inf = torch.zeros_like(self.flat)
            rank = torch.distributed.get_rank(process_group) if (self.world > 1 and torch.distributed.is_initialized()) else 0
            stream_id = rank if dropout_stream is None else int(dropout_stream)
            philox_seed = (seed * 2654435761 + stream_id * 0x9E3779B97F4A7C15) % (2 ** 62) + 12345
            self.step_state = torch.tensor([philox_seed, 0], **i64)   # {philox seed, step}
            if self.world > 1 and torch.distributed.is_initialized():
                torch.distributed.broadcast(self.flat, src=torch.distributed.get_global_rank(process_group, 0) if process_group is not None else 0,
                                            group=process_group)
            # static batch buffers
            self.ids = torch.zeros(self.B, **i64)
            self.batch = {
                "x": torch.empty(self.nt, 11, **f32), "edge_attr": torch.empty(self.et, 13, **f32), "y": torch.empty(self.nt, 2, **f32),
                "edge_index": torch.empty(2, self.et, **i64), "batch": torch.empty(self.nt, **i64),
                "ptr": torch.empty(self.B + 1, **i64), "eptr": torch.empty(self.B + 1, **i64), "vminmax": torch.empty(2, **f32),
            }
            self.stats = torch.cat([store.x_mean, store.x_std, store.edge_mean, store.edge_std]).to(**f32).contiguous()
            self.loss = torch.zeros((), **f32)
            self.grad_out = torch.empty(self.nt, 2, **f32)
            self.bufs = self.runner.alloc(self.nt, self.dev, need_grad=True, **({'pipelined': True} if self.network == 'skippfn' else {}))
            # structure: one eager pack, then build once (uniform topology: identical for every batch)
            self.ids.copy_(torch.arange(self.B, device=self.dev) % store.num_scenarios)
            launch_pack(store, self.ids, self.batch, self.nt, self.et)
            from .ops import tile_cap
            self.graph = BatchGraph(self.batch["edge_index"], self.nt, ptr=self.batch["ptr"], undirect=1, tile_cap=tile_cap())
            self.wls_ws = self.graph.wls_workspace()
            # the seven doubles the reduction pass of the loss leaves in its workspace (5 batch sums, bus count, branch count)
            self.wls_sums = self.wls_ws.view(torch.uint8)[256:256 + 56].view(torch.float64)
            if self.exact and self.graph.c.num_tiles == 0:
                raise _lib.Dss2Error("GraphedTrainer(exact_global_batch=True) serves tiled batches (graphs of up to 256 buses)")
        self.cuda_graph = None
        self.launches_per_step = None
        self.use_cuda_graph = use_cuda_graph

    # ---- parameters ----
    def _init_params(self, seed, sd):
        table = self.runner.table
        if sd is None and self.network != "skippfn":   # the drop-in module's own initialisation (PyG's glorot / zeros, torch's Linear)
            import sys, os
            pkg = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
            if pkg not in sys.path:
                sys.path.insert(0, pkg)
            import networks
            sp = self.spec
            torch.manual_seed(seed)
            if self.network == "gat":
                m = networks.GAT_DSSE(dim_feat=sp.dim_feat, dim_dense=sp.dim_dense, dim_out=sp.dim_out, heads=1, num_layers=sp.num_layers,
                                      edge_dim=sp.edge_dim, slope=sp.att_slope, self_loops=sp.self_loops, nonlin=sp.act)
            else:
                m = networks.GINE_DSSE(dim_feat=sp.dim_feat, dim_dense=sp.dim_dense, dim_out=sp.dim_out, num_layers=sp.num_layers,
                                       edge_dim=sp.edge_dim, eps=sp.eps, train_eps=sp.train_eps)
            sd = {k: v.detach() for k, v in m.named_parameters()}
        if sd is None:
            import math
            g = torch.Generator().manual_seed(seed)
            sd = {}
            for name, shape in self.spec.param_names():
                if "convs." in name and name.endswith(".bias"):
                    sd[name] = torch.zeros(shape)                      # PyG TAGConv bias: zeros
                else:
                    bound = 1.0 / math.sqrt(shape[-1] if len(shape) > 1 else self._fan_in(name))
                    sd[name] = (torch.rand(shape, generator=g) * 2 - 1) * bound
        for name, (off, n) in table.items():
            self.flat[off:off + n].copy_(sd[name].reshape(-1).to(self.flat))

    def _fan_in(self, name):
        return 2 * self.spec.fn + self.spec.fe if "edge_aggr.0" in name else self.spec.hid

    def state_dict(self):
        if self.network != "skippfn":
            return {name: self.flat[off:off + n].clone() for name, (off, n) in self.runner.table.items()}
        return {name: self.flat[off:off + n].view(shape).clone()
                for (name, shape), (off, n) in zip(self.spec.param_names(), self.runner.table.values())}

    # ---- one step ----
    def _enqueue(self, with_optimizer=True):
        lib, st = self.lib, _lib.stream()
        b = self.batch
        if not with_optimizer:   # the step counter (= the sequence number of the tile marks of the chained layers) will not advance
            for k in ("marks", "marks_b"):
                if k in self.bufs:
                    self.bufs[k].zero_()
        pre = self.network == "skippfn" and self.runner.ea_slots(self.graph, 11, 13)
        if pre:      # the EdgeAggregation weights go to their constant-memory slots on a second stream, beside the batch packer
            main = torch.cuda.current_stream()
            if getattr(self, "_prep_stream", None) is None:
                self._prep_stream = torch.cuda.Stream(device=self.dev)
            self._prep_stream.wait_stream(main)
            with torch.cuda.stream(self._prep_stream):
                self.runner.ea_upload(self.flat)
        launch_pack(self.store, self.ids, b, self.nt, self.et)
        if pre:
            main.wait_stream(self._prep_stream)
        if self.network == "skippfn":
            out = self.runner.forward(self.graph, b["x"], 11, b["edge_attr"], 13, self.flat, self.bufs,
                                      drop_mode=1 if self.spec.p_drop > 0 else 0, rng_state=self.step_state, ea_uploaded=bool(pre))
        else:
            # GAT: the attention dropout of GATSpec.dropout (training mode) draws from the same device {seed, step} as the TAG dropout
            kw = {"rng_state": self.step_state} if self.network == "gat" else {}
            out = self.runner.forward(self.graph, b["x"], 11, b["edge_attr"], 13, self.flat, self.bufs, **kw)
        wls_args = (self.graph.ref, _lib.ptr(b["x"]), 11, _lib.ptr(b["edge_attr"]), 13, _lib.ptr(out), _lib.ptr(self.stats), *self.coefs,
                    _lib.ptr(b["vminmax"]), 1, _lib.ptr(self.loss), None, _lib.ptr(self.grad_out), _lib.ptr(self.wls_ws),
                    self.wls_ws.numel() * self.wls_ws.element_size(), st)
        if self.exact:   # reduction pass -> all-reduce of the batch sums and counts -> gradient pass on the global means
            _lib.check(lib.dss2_wls_pass(1, *wls_args), "dss2_wls_pass(1)")
            torch.distributed.all_reduce(self.wls_sums, group=self.pg)
            _lib.check(lib.dss2_wls_pass(2, *wls_args), "dss2_wls_pass(2)")
        else:
            _lib.check(lib.dss2_wls_fwd_bwd(*wls_args), "dss2_wls_fwd_bwd")
        if self.network == "skippfn":
            # N > 1: each sub-net's slice of the gradient is all-reduced on the backward's second stream while the next sub-net runs
            hook = None
            if self.world > 1 and BUCKETED_ALLREDUCE:
                def hook(lo, hi):
                    torch.distributed.all_reduce(self.flat_grad[lo:hi], group=self.pg)
            self.runner.backward(self.graph, b["x"], 11, b["edge_attr"], 13, self.flat, self.bufs, self.grad_out, self.flat_grad, ea_uploaded=True,
                                 rng_state=self.step_state, bucket_hook=hook)
            reduced = self.runner.bucketed
        else:
            # GAT: the forward's constant-memory weight slots are still valid, and the backward re-draws the forward's dropout masks
            kw = {"uploaded": True, "rng_state": self.step_state} if self.network == "gat" else {}
            self.runner.backward(self.graph, b["x"], 11, b["edge_attr"], 13, self.flat, self.bufs, self.grad_out, self.flat_grad, **kw)
            reduced = False
        if self.world > 1 and not reduced:
            torch.distributed.all_reduce(self.flat_grad[:self.flat.numel()], group=self.pg)
        if with_optimizer:
            _lib.check(lib.dss2_adamax_step(_lib.ptr(self.flat), _lib.ptr(self.flat_grad), _lib.ptr(self.exp_avg), _lib.ptr(self.exp_inf),
                                            self.flat.numel(), self.lr, 0.9, 0.999, 1e-8, 1.0 if self.exact else 1.0 / self.world, _lib.ptr(self.step_state), 1,
                                            st), "dss2_adamax_step")

    def capture(self):
        """Warm up eagerly (also counts the launches of one step), then capture the step into a CUDA graph."""
        with torch.cuda.device(self.dev):
            # the warm-up steps are real steps: put the trainable state back afterwards so that the user's first step() is step 1
            keep = [t.clone() for t in (self.flat, self.exp_avg, self.exp_inf, self.step_state)]
            side = torch.cuda.Stream()
            side.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(side):
                for _ in range(2):
                    before = _lib.launch_count()
                    self._enqueue()
                    self.launches_per_step = _lib.launch_count() - before + (1 if self.world > 1 else 0) + (1 if self.exact else 0)
            torch.cuda.current_stream().wait_stream(side)
            torch.cuda.synchronize()
            for t, k in zip((self.flat, self.exp_avg, self.exp_inf, self.step_state), keep):
                t.copy_(k)
            if self.use_cuda_graph:
                g = torch.cuda.CUDAGraph()
                with torch.cuda.graph(g):
                    self._enqueue()
                self.cuda_graph = g
        return self

    def step(self, ids=None):
        """Enqueue one training step for scenario ids (device or pinned-host int64 [B]); returns the device loss scalar."""
        if ids is not None:
            self.ids.copy_(ids, non_blocking=True)
        if self.cuda_graph is not None:
            self.cuda_graph.replay()
        else:
            self._enqueue()
        return self.loss
