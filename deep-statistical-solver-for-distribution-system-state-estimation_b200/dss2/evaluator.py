"""Device-resident validation and inference: packer -> eval-mode forward -> (epoch metrics | branch flows of the estimate), launched
straight through the C ABI over static buffers and replayed as ONE CUDA graph per batch length.

The other half of the reference's loop beside `GraphedTrainer`: the per-epoch validation pass (dss2_run.py:165-236) and the inference
workload (forward + get_pflow).  Each batch's ten metrics are finalised on the device and added into an fp64 epoch accumulator
(`dss2_eval_metrics_acc`), so an epoch costs one device-to-host copy in `metrics()` instead of one synchronisation per batch.

Eval-mode semantics follow the drop-in modules: SkipPFN keeps its dropout on in eval() (networks.py:268), drawn from the evaluator's own
Philox stream; GAT_DSSE and GINE_DSSE run without dropout.  The evaluator never writes the trainer's parameters, optimizer state or step
counter, nor any buffer its captured step reads: it has its own batch buffers, activations, tile marks and {seed, step} clock
(and, for GAT_DSSE with heads > 1, whose forward rewrites constant blocks of its parameter buffer, its own copy of the parameters).
"""
import ctypes

import torch

from . import _lib
from .batching import launch_pack
from .graph import BatchGraph
from .metrics import epoch_means
from .trainer import make_runner


class GraphedEvaluator:
    def __init__(self, store, batch_graphs, trainer=None, network="skippfn", spec=None, state_dict=None, seed=0, use_cuda_graph=True):
        """store: CUDA-resident uniform-topology ScenarioStore (may differ from the trainer's).  batch_graphs: the largest batch.
        trainer: a GraphedTrainer whose parameters (`flat`) are evaluated in place (GAT with heads > 1: copied on the device
        at the start of every call), or None with network / spec / state_dict (the
        reference's parameter names, e.g. a checkpoint) - the evaluator then keeps its own copy.  seed: the evaluator's dropout stream
        (SkipPFN's eval-mode dropout); its Philox seeds lie outside the range the training streams use."""
        self.lib = _lib.load()
        self.store = store
        self.B = int(batch_graphs)
        self.dev = store.x.device
        if self.dev.type != "cuda":
            raise _lib.Dss2Error("GraphedEvaluator needs a CUDA-resident ScenarioStore")
        if store.x.size(0) != store.num_scenarios * store.max_nodes or store.edge_index.size(1) != store.num_scenarios * store.max_edges:
            raise _lib.Dss2Error("GraphedEvaluator needs a uniform-topology store (static batch shapes)")
        if self.B < 1:
            raise _lib.Dss2Error("GraphedEvaluator: batch_graphs must be >= 1")
        if trainer is not None:
            network, spec = trainer.network, trainer.spec
        self.network = network
        self.runner, self.spec = make_runner(network, spec)
        self.use_cuda_graph = use_cuda_graph
        n, e = store.max_nodes, store.max_edges
        self.nt, self.et = self.B * n, self.B * e
        f32 = dict(dtype=torch.float32, device=self.dev)
        i64 = dict(dtype=torch.long, device=self.dev)
        # GAT with heads > 1: the runner's forward rewrites the constant tail of the buffer it reads (GATRunner.prepare), so the evaluator
        # reads a private copy of the trainer's parameters, refreshed by one device-to-device copy at the start of every call
        self._src = trainer.flat if (trainer is not None and network == "gat" and self.spec.heads > 1) else None
        self.owns_flat = trainer is None or self._src is not None
        with torch.cuda.device(self.dev):
            if self._src is not None:
                self.flat = self._src.clone()
            elif trainer is not None:
                self.flat = trainer.flat          # read in place: the next epoch sees the parameters of the latest step
            else:
                if state_dict is None:
                    raise _lib.Dss2Error("GraphedEvaluator needs a trainer or a state_dict")
                self.flat = torch.zeros(self.runner.flat_size, **f32)
                for name, (off, cnt) in self.runner.table.items():
                    if name.startswith("_"):      # GAT's constant blocks (heads > 1): written by the runner itself
                        continue
                    self.flat[off:off + cnt].copy_(torch.as_tensor(state_dict[name]).reshape(-1).to(self.flat))
            # {philox seed, step}: the training streams' seeds lie in [12345, 2^62 + 12345), these above
            self.rng = torch.tensor([2 ** 62 + 12345 + (int(seed) * 2654435761) % 2 ** 61, 0], **i64)
            self.x_mean0, self.x_std0 = float(store.x_mean[0]), float(store.x_std[0])
            self.ids = torch.zeros(self.B, **i64)
            self.batch = {"x": torch.empty(self.nt, 11, **f32), "edge_attr": torch.empty(self.et, 13, **f32), "y": torch.empty(self.nt, 2, **f32),
                          "batch": torch.empty(self.nt, **i64), "ptr": torch.empty(self.B + 1, **i64), "eptr": torch.empty(self.B + 1, **i64),
                          "vminmax": torch.empty(2, **f32)}
            self.bufs = self.runner.alloc(self.nt, self.dev, need_grad=False)
            self.pflow = torch.empty(8 * self.et, **f32)
            self.acc = torch.zeros(11, dtype=torch.float64, device=self.dev)
            self.ws = torch.zeros(self.lib.dss2_eval_workspace_bytes(), dtype=torch.uint8, device=self.dev)
        self._lens = {}                 # batch length -> {"edge_index", "graph", "evaluate" / "infer": CUDA graph}
        self.launches_per_call = {}

    # ---- per-length structure ----
    def _length(self, n):
        ent = self._lens.get(n)
        if ent is None:
            from .ops import tile_cap
            nt, et = n * self.store.max_nodes, n * self.store.max_edges
            ei = torch.empty(2, et, dtype=torch.long, device=self.dev)     # contiguous [2, Et]: the metric and flow kernels need it
            self.ids[:n].copy_(torch.arange(n, device=self.dev) % self.store.num_scenarios)
            launch_pack(self.store, self.ids[:n], dict(self.batch, edge_index=ei), nt, et)
            graph = BatchGraph(ei, nt, ptr=self.batch["ptr"][:n + 1].clone(), undirect=1, tile_cap=tile_cap())
            ent = self._lens[n] = {"edge_index": ei, "graph": graph, "nt": nt, "et": et}
        return ent

    def _enqueue(self, n, mode):
        lib, st = self.lib, _lib.stream()
        ent = self._lens[n]
        b, graph, nt, et, ei = self.batch, ent["graph"], ent["nt"], ent["et"], ent["edge_index"]
        if self._src is not None:
            self.flat.copy_(self._src)
        launch_pack(self.store, self.ids[:n], dict(b, edge_index=ei), nt, et)
        if self.network == "skippfn":   # eval() keeps SkipPFN's dropout on (networks.py:268); the clock also numbers the tile marks
            out = self.runner.forward(graph, b["x"], 11, b["edge_attr"], 13, self.flat, self.bufs, drop_mode=1 if self.spec.p_drop > 0 else 0,
                                      rng_state=self.rng)
        else:                           # GAT_DSSE / GINE_DSSE: no dropout in eval()
            out = self.runner.forward(graph, b["x"], 11, b["edge_attr"], 13, self.flat, self.bufs)
        _lib.check(lib.dss2_step_advance(_lib.ptr(self.rng), st), "dss2_step_advance")
        os_ = out.stride(0)
        if mode == "evaluate":
            _lib.check(lib.dss2_eval_metrics_acc(_lib.ptr(ei), nt, et, _lib.ptr(b["x"]), 11, _lib.ptr(b["edge_attr"]), 13, _lib.ptr(out), os_,
                                                 _lib.ptr(b["y"]), 2, self.x_mean0, self.x_std0, _lib.ptr(b["vminmax"]), _lib.ptr(self.acc),
                                                 _lib.ptr(self.ws), self.ws.numel(), st), "dss2_eval_metrics_acc")
        else:
            ep = ctypes.c_void_p(b["edge_attr"].data_ptr() + 6 * 4)
            _lib.check(lib.dss2_pflow_est(_lib.ptr(ei), et, _lib.ptr(out), os_, _lib.ptr(b["x"]), 11, self.x_mean0, self.x_std0, ep, 13,
                                          _lib.ptr(b["vminmax"]), _lib.ptr(self.pflow), st), "dss2_pflow_est")
        return out

    def _run(self, ids, mode):
        if not torch.is_tensor(ids) or ids.dtype != torch.long or ids.dim() != 1:
            raise _lib.Dss2Error("GraphedEvaluator: ids must be a 1-D int64 tensor")
        n = ids.numel()
        if not 1 <= n <= self.B:
            raise _lib.Dss2Error(f"GraphedEvaluator: batch of {n} scenarios; 1 <= len(ids) <= batch_graphs = {self.B}")
        with torch.cuda.device(self.dev):
            ent = self._length(n)
            self.ids[:n].copy_(ids, non_blocking=True)
            if not self.use_cuda_graph:
                self._enqueue(n, mode)
            else:
                g = ent.get(mode)
                if g is None:
                    g = ent[mode] = self._capture(n, mode)
                g.replay()
        return n

    def _capture(self, n, mode):
        """Warm up eagerly (counts the launches of one call; the accumulator is put back afterwards), then capture."""
        keep = self.acc.clone()
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            before = _lib.launch_count()
            self._enqueue(n, mode)
            self.launches_per_call[mode] = _lib.launch_count() - before
        torch.cuda.current_stream().wait_stream(side)
        torch.cuda.synchronize()
        self.acc.copy_(keep)
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            self._enqueue(n, mode)
        return g

    # ---- public ----
    def evaluate(self, ids):
        """Enqueue one validation batch (int64 scenario ids, device or pinned host, 1 <= len <= batch_graphs): its ten metrics are added
        to the epoch accumulator on the device.  No host synchronisation once the graph of this length exists."""
        self._run(ids, "evaluate")

    def infer(self, ids):
        """(out [n*N, dim_out], pflow): the model output and get_pflow's eight [n*E] outputs of the de-normalised estimate, as views of
        static buffers that the next call overwrites."""
        n = self._run(ids, "infer")
        nt, et = n * self.store.max_nodes, n * self.store.max_edges
        out = self.bufs["outs"][-1] if self.network == "skippfn" else self.bufs["out"]
        pf = self.pflow[:8 * et].view(8, et)
        return out[:nt], tuple(pf[i] for i in range(8))

    def metrics(self, reset=True):
        """Epoch means of the batches evaluated since the last reset: evaluate_batch's ten keys + "batches".  One device-to-host copy."""
        with torch.cuda.device(self.dev):
            res = epoch_means(self.acc)
            if reset:
                self.acc.zero_()
        return res

    def memory_bytes(self):
        """Device memory the evaluator owns (buffers, per-length structures; the parameters only when it holds its own copy)."""
        seen, total = set(), 0

        def add(t):
            nonlocal total
            if torch.is_tensor(t) and t.data_ptr() not in seen:
                seen.add(t.data_ptr())
                total += t.numel() * t.element_size()
            elif isinstance(t, (list, tuple)):
                for u in t:
                    add(u)
            elif isinstance(t, dict):
                for u in t.values():
                    add(u)
        add([self.ids, self.batch, self.bufs, self.pflow, self.acc, self.ws, self.rng])
        for ent in self._lens.values():
            g = ent["graph"]
            add([ent["edge_index"], g.ptr, g.ws, g.scratch])
        if self.owns_flat:
            add(self.flat)
        return total
