"""Drop-in for the reference's `networks` module (reference networks.py), B200-native underneath.

Same class names, constructor keywords, `forward(x, edge_index, edge_attr)` signature and parameter names /
shapes (so reference checkpoints load both ways, dss2_run.py:95-101,240-247) - but a forward / backward is a
sequence of hand-written sm_100a kernels (libdss2_b200.so): one fused kernel per EdgeAggregation and per
TAGConv(+Dropout+ReLU) layer over a batch structure that is built once per batch instead of once per layer.

Hot path (BASELINE.json north_star): EdgeAggregation, MPN, SkipMPN, PFN, SkipPFN.
Reference behaviours kept on purpose (SURVEY.md appendix A): dropout is active in eval() too
(networks.py:268 builds a fresh nn.Dropout inside forward); the degree norm computed in
EdgeAggregation.forward (networks.py:196-200) never reaches `message` and is not applied; all sub-nets of a
PFN receive the same raw edge attributes; reversed edges negate attribute columns 0 and 2 (networks.py:252).
There is no CPU fallback: without a CUDA device or the built library, forward raises.
GAT_DSSE (networks.py:113-156, the as-shipped default of dss2_run.py:86; SURVEY.md 8f-1) runs on its own fused GATv2 kernels
(csrc/gat.cu), and so do GINE_DSSE (networks.py:71-111) and gnn_dsse (networks.py:11-69; model='gcn2', 'fagcn' and 'tagcn').
"""
import math

import torch
import torch.nn as nn

from dss2 import ops
from dss2.ops import PFNSpec


class _LazyMachinery:
    """The launch machinery (runner with the ctypes library handle, flat parameter pack) is a per-object cache in `__dict__`; it must
    not travel with copy.deepcopy / pickle / torch.save(model) - ctypes function pointers cannot be pickled - and is rebuilt on the
    next forward."""

    def __getstate__(self):
        state = self.__dict__.copy()
        state.pop("_dss2_machinery", None)
        state.pop("_dss2_param_slots", None)
        return state

    def _named_params(self):
        """dict(self.named_parameters()) without walking the module tree on every forward (181 parameters for the default SkipPFN: 0.85 ms of
        a 8 ms script-scale step): the (name, owning module, attribute) triples are cached, the Parameter objects are looked up fresh, so
        .to() / load_state_dict / parameter replacement keep working."""
        slots = self.__dict__.get("_dss2_param_slots")
        if slots is None:
            slots = []
            seen = set()
            for prefix, mod in self.named_modules():
                for attr, p in mod._parameters.items():
                    if p is not None and id(p) not in seen:          # shared parameters once, under their first name (named_parameters' rule)
                        seen.add(id(p))
                        slots.append((prefix + "." + attr if prefix else attr, mod, attr))
            self.__dict__["_dss2_param_slots"] = slots
        return {name: mod._parameters[attr] for name, mod, attr in slots}


class TAGConv(nn.Module):
    """Parameter container with PyG TAGConv's names: lins.{0..K}.weight [out, in] (no bias), bias [out]
    (zero-initialised).  Inside MPN the fused layer kernel consumes the parameters directly; called on its
    own it evaluates sum_k (A_hat^k x) W_k^T + b on the un-directed version of `edge_index`."""

    def __init__(self, in_channels, out_channels, K=3, bias=True):
        super().__init__()
        self.in_channels, self.out_channels, self.K = in_channels, out_channels, K
        self.lins = nn.ModuleList([nn.Linear(in_channels, out_channels, bias=False) for _ in range(K + 1)])
        self.bias = nn.Parameter(torch.zeros(out_channels))

    def forward(self, x, edge_index):
        return ops.tag_conv(x, edge_index, [lin.weight for lin in self.lins], self.bias)


class EdgeAggregation(nn.Module):
    """networks.py:159-209: out[i] = sum over edges (j -> i) of MLP([x_i | x_j | a_ji]), aggr='add'.
    Takes the ONE-WAY edge list of the reference's data and applies MPN's un-directing (reversed edges with
    attribute columns 0 and 2 negated) inside the kernel."""

    def __init__(self, dim_featn, dim_feate, dim_hid, dim_out):
        super().__init__()
        self.dim_featn, self.dim_feate, self.dim_out = dim_featn, dim_feate, dim_out
        self.edge_aggr = nn.Sequential(nn.Linear(dim_featn * 2 + dim_feate, dim_hid), nn.ReLU(), nn.Linear(dim_hid, dim_out))

    def forward(self, x, edge_index, edge_attr):
        return ops.edge_aggregation(x, edge_index, edge_attr, self.edge_aggr[0].weight, self.edge_aggr[0].bias,
                                    self.edge_aggr[2].weight, self.edge_aggr[2].bias)


class _Stack(_LazyMachinery, nn.Module):
    """Shared machinery of MPN / SkipMPN / PFN / SkipPFN: spec, flat parameter pack, fused launch sequence."""
    _dss2_masks = None        # test hook: [sub-net][layer] 0/1 masks consumed by the next forward (exact torch parity)
    _dss2_rng_state = None    # optional device int64 {seed, step} for the in-kernel Philox dropout

    def _spec(self):
        raise NotImplementedError

    def _machinery(self):
        m = self.__dict__.get("_dss2_machinery")
        if m is None:
            spec = self._spec()
            m = (ops.PFNRunner(spec), ops.ParamPack(spec))
            self.__dict__["_dss2_machinery"] = m
        return m

    def forward(self, x, edge_index, edge_attr):
        runner, pack = self._machinery()
        masks, self._dss2_masks = self._dss2_masks, None
        return ops.pfn_apply(runner, pack, self._named_params(), x, edge_index, edge_attr, masks=masks,
                             rng_state=self._dss2_rng_state)


def _build_mpn(self, dim_featn, dim_feate, dim_out, dim_hid, n_gnn_layers, K, dropout_rate):
    self.dim_featn, self.dim_feate, self.dim_out, self.dim_hid = dim_featn, dim_feate, dim_out, dim_hid
    self.n_gnn_layers, self.K, self.dropout_rate = n_gnn_layers, K, dropout_rate
    self.edge_aggr = EdgeAggregation(dim_featn, dim_feate, dim_hid, dim_hid)
    self.convs = nn.ModuleList()
    for l in range(n_gnn_layers):
        self.convs.append(TAGConv(dim_hid, dim_out if l == n_gnn_layers - 1 else dim_hid, K=K))


class MPN(_Stack):
    """networks.py:212-273: EdgeAggregation, then n_gnn_layers TAGConv(K) with Dropout+ReLU between them."""
    _skip = False

    def __init__(self, dim_featn, dim_feate, dim_out, dim_hid, n_gnn_layers, K, dropout_rate):
        super().__init__()
        _build_mpn(self, dim_featn, dim_feate, dim_out, dim_hid, n_gnn_layers, K, dropout_rate)

    def _spec(self):
        return PFNSpec(fn=self.dim_featn, fe=self.dim_feate, dim_out=self.dim_out, n_layers=self.n_gnn_layers, K=self.K, L=1,
                       p_drop=float(self.dropout_rate), skip=(self._skip,), prefix_fmt="", hid=self.dim_hid)


class SkipMPN(MPN):
    """networks.py:275-338: MPN whose input is added to its output (needs dim_out == dim_featn)."""
    _skip = True


def _build_pfn(self, sub_cls, dim_featn, dim_feate, dim_out, dim_hid, n_gnn_layers, K, dropout_rate, L):
    self.dim_featn, self.dim_feate, self.dim_out, self.dim_hid = dim_featn, dim_feate, dim_out, dim_hid
    self.n_gnn_layers, self.K, self.dropout_rate, self.L = n_gnn_layers, K, dropout_rate, L
    self.mpns = nn.ModuleList()
    for l in range(L):
        if l == L - 1:   # the last sub-net is always a plain MPN onto dim_out (networks.py:355,380)
            self.mpns.append(MPN(dim_featn, dim_feate, dim_out, dim_hid, n_gnn_layers, K, dropout_rate))
        else:
            self.mpns.append(sub_cls(dim_featn, dim_feate, dim_featn, dim_hid, n_gnn_layers, K, dropout_rate))


class PFN(_Stack):
    """networks.py:340-363: L stacked MPNs, every one fed the same raw edge attributes."""
    _sub = MPN

    def __init__(self, dim_featn, dim_feate, dim_out, dim_hid, n_gnn_layers, K, dropout_rate, L):
        super().__init__()
        _build_pfn(self, self._sub, dim_featn, dim_feate, dim_out, dim_hid, n_gnn_layers, K, dropout_rate, L)

    def _spec(self):
        skip = tuple((self._sub is SkipMPN) and s < self.L - 1 for s in range(self.L))
        return PFNSpec(fn=self.dim_featn, fe=self.dim_feate, dim_out=self.dim_out, n_layers=self.n_gnn_layers, K=self.K, L=self.L,
                       p_drop=float(self.dropout_rate), skip=skip, prefix_fmt="mpns.{s}.", hid=self.dim_hid)


class SkipPFN(PFN):
    """networks.py:365-388: PFN whose first L-1 sub-nets are SkipMPNs."""
    _sub = SkipMPN


def _check_attn_dropout(p, who):
    """Attention dropout probability as F.dropout accepts it (ValueError outside [0, 1]); p == 1 (every coefficient dropped) is not built.
    p > 0 exists only as CUDA kernels (the masks are drawn inside them): without a CUDA device it is refused when the model is built."""
    if p < 0. or p > 1.:
        raise ValueError(f"dropout probability has to be between 0 and 1, but got {p}")
    if p == 1.:
        raise NotImplementedError(f"{who}: attention dropout p == 1 (every attention coefficient dropped) is not supported")
    if p > 0. and not torch.cuda.is_available():
        raise NotImplementedError(f"{who}: attention dropout runs in the CUDA kernels only and no CUDA device is available "
                                  "(there is no CPU implementation)")


class _GCN2Params(nn.Module):
    """Parameter holder with PyG GCN2Conv's name / shape / initialisation: `weight1` [channels, channels], glorot (shared_weights=True:
    no `weight2`).  The arithmetic is in the fused kernels (csrc/gat.cu)."""

    def __init__(self, channels):
        super().__init__()
        self.weight1 = nn.Parameter(torch.empty(channels, channels))
        nn.init.xavier_uniform_(self.weight1)


class _FAParams(nn.Module):
    """Parameter holder with PyG FAConv's names / shapes / initialisation: `att_l`, `att_r` = Linear(channels, 1, bias=False)."""

    def __init__(self, channels):
        super().__init__()
        self.att_l = nn.Linear(channels, 1, bias=False)
        self.att_r = nn.Linear(channels, 1, bias=False)


class gnn_dsse(_LazyMachinery, nn.Module):
    """networks.py:11-69: (num_layers - 1) x [conv + nonlin], Linear(dim_feat, dim_dense), Linear(dim_dense, dim_out) in a PyG `Sequential`
    (children `module_{i}`), `forward(x, edge_index)` with x_0 = x.  conv = GCN2Conv(channels, alpha=main_param, theta, shared_weights,
    cached, normalize, add_self_loops) for model='gcn2' (the default), FAConv(channels, eps=main_param, dropout, cached, normalize,
    add_self_loops) for model='fagcn', or TAGConv(channels, channels, K, bias, normalize) for model='tagcn'.  Built for what the
    reference's defaults select (theta=None, shared_weights=True, normalize=True); the other settings raise.  `dropout` is FAConv's
    attention dropout (0 <= p < 1), active in train() only like PyG's; gcn2 and tagcn ignore it, as the reference does.
    `cached=True` is accepted and ignored: the normalisation is recomputed per batch."""
    _dss2_attn_masks = None   # test hook (fagcn): per layer uint8 [1, Et + Nt] keep masks in the kernels' edge-key layout, consumed by the next forward

    def __init__(self, dim_feat, dim_dense, dim_out, num_layers, nonlin='leaky_relu', main_param=0.1, K=3, bias=True, dropout=0., theta=None,
                 shared_weights=True, cached=True, add_self_loops=True, normalize=True, model='gcn2'):
        super().__init__()
        if nonlin not in ('relu', 'tanh', 'leaky_relu'):
            raise Exception('invalid activation type')
        if model not in ('gcn2', 'fagcn', 'tagcn'):
            raise Exception('invalid model type')
        if model == 'fagcn':
            _check_attn_dropout(dropout, "gnn_dsse(model='fagcn')")
        if theta is not None or not shared_weights or not normalize:
            raise NotImplementedError("gnn_dsse kernels cover theta=None, shared_weights=True, normalize=True (the reference's defaults)")
        self.channels, self.main_param, self.dim_out, self.K, self.dropout, self.bias = dim_feat, main_param, dim_out, K, dropout, bias
        self.theta, self.num_layers, self.shared_weights, self.cached = theta, num_layers, shared_weights, cached
        self.normalize, self.add_self_loops, self.dim_dense, self.kind, self.nonlin_name = normalize, add_self_loops, dim_dense, model, nonlin
        self.nonlin = {'relu': nn.ReLU, 'tanh': nn.Tanh, 'leaky_relu': nn.LeakyReLU}[nonlin]()
        self.model = nn.Module()
        i = 0
        for _ in range(num_layers - 1):
            conv = _GCN2Params(dim_feat) if model == 'gcn2' else _FAParams(dim_feat) if model == 'fagcn' else TAGConv(dim_feat, dim_feat, K=K, bias=bias)
            self.model.add_module(f"module_{i}", conv)
            self.model.add_module(f"module_{i + 1}", self.nonlin)
            i += 2
        self.model.add_module(f"module_{i}", nn.Linear(dim_feat, dim_dense))
        self.model.add_module(f"module_{i + 1}", nn.Linear(dim_dense, dim_out))

    def _machinery(self):
        m = self.__dict__.get("_dss2_machinery")
        if m is None:
            from dss2 import gnn
            spec = gnn.GNNSpec(model=self.kind, dim_feat=self.channels, dim_dense=self.dim_dense, dim_out=self.dim_out,
                               num_layers=self.num_layers, alpha=float(self.main_param), K=self.K, bias=bool(self.bias),
                               self_loops=bool(self.add_self_loops), normalize=bool(self.normalize), act=self.nonlin_name,
                               act_slope=float(getattr(self.nonlin, "negative_slope", 0.0)),
                               dropout=float(self.dropout) if self.kind == 'fagcn' else 0.0)
            m = gnn.make_machinery(spec)
            self.__dict__["_dss2_machinery"] = m
        return m

    def forward(self, x, edge_index):
        from dss2 import gnn
        runner, pack = self._machinery()
        masks, self._dss2_attn_masks = self._dss2_attn_masks, None
        drop = self.training and runner.spec.dropout > 0.      # FAConv: F.dropout(..., training=self.training)
        return gnn.gnn_apply(runner, pack, self._named_params(), x, edge_index, drop=drop, masks=masks)


class _GINEParams(nn.Module):
    """Parameter holder with PyG GINEConv's names: `nn` (the Linear handed in, shared by every layer of the model), `lin`
    (Linear(edge_dim, in_channels)), buffer `eps`.  The arithmetic is in the fused kernel (csrc/gat.cu)."""

    def __init__(self, shared_nn, eps, edge_dim, train_eps=False):
        super().__init__()
        self.nn = shared_nn
        if train_eps:
            self.eps = nn.Parameter(torch.full((1,), float(eps)))
        else:
            self.register_buffer("eps", torch.full((1,), float(eps)))
        self.lin = nn.Linear(edge_dim, shared_nn.in_features)


class GINE_DSSE(_LazyMachinery, nn.Module):
    """networks.py:71-111: (num_layers - 1) x [GINEConv(nn, eps, train_eps, edge_dim) + LeakyReLU()], Linear(dim_feat, dim_dense),
    Linear(dim_dense, dim_out) inside a PyG `Sequential` (children `module_{i}`).  As in the reference, `nn` is ONE
    Linear(dim_feat, dim_feat) shared by all layers (it also appears as `model.module_{2l}.nn.*` in the state_dict)."""

    def __init__(self, dim_feat, dim_dense, dim_out, num_layers, edge_dim, nn='mlp', nonlin='leaky_relu', eps=0., train_eps=False,
                 model='gine'):
        super().__init__()
        import torch.nn as tnn        # the reference's `nn` argument shadows torch.nn (networks.py:72): only leaky_relu can work there
        if nn != 'mlp':
            raise Exception('invalid nn type')
        if nonlin != 'leaky_relu':
            raise NotImplementedError("GINE_DSSE: the reference itself only works with nonlin='leaky_relu' (its `nn` argument shadows "
                                      "torch.nn, networks.py:72,88-91)")
        if model != 'gine':
            raise Exception('invalid model type')
        self.dim_out, self.num_layers, self.dim_feat, self.dim_dense = dim_out, num_layers, dim_feat, dim_dense
        self.eps, self.train_eps, self.edge_dim, self.dim_hidden = eps, train_eps, edge_dim, dim_feat
        self.nn = tnn.Linear(dim_feat, dim_feat)
        self.nonlin = tnn.LeakyReLU()
        self.model = tnn.Module()
        i = 0
        for _ in range(num_layers - 1):
            self.model.add_module(f"module_{i}", _GINEParams(self.nn, eps, edge_dim, train_eps))
            self.model.add_module(f"module_{i + 1}", self.nonlin)
            i += 2
        self.model.add_module(f"module_{i}", tnn.Linear(dim_feat, dim_dense))
        self.model.add_module(f"module_{i + 1}", tnn.Linear(dim_dense, dim_out))

    def _machinery(self):
        m = self.__dict__.get("_dss2_machinery")
        if m is None:
            from dss2 import gine
            spec = gine.GINESpec(dim_feat=self.dim_feat, dim_dense=self.dim_dense, dim_out=self.dim_out, num_layers=self.num_layers,
                                 edge_dim=self.edge_dim, eps=float(self.eps), act_slope=float(self.nonlin.negative_slope),
                                 train_eps=bool(self.train_eps))
            m = gine.make_machinery(spec)
            self.__dict__["_dss2_machinery"] = m
        return m

    def forward(self, x, edge_index, edge_attr):
        from dss2 import gine
        runner, pack = self._machinery()
        return gine.gine_apply(runner, pack, self._named_params(), x, edge_index, edge_attr)


class _GATv2Params(nn.Module):
    """Parameter holder with PyG GATv2Conv's names / shapes / initialisation (glorot weights, zero biases); the arithmetic is in the
    fused kernel (csrc/gat.cu), so this module has no forward of its own."""

    def __init__(self, channels, edge_dim, heads=1):
        super().__init__()
        self.att = nn.Parameter(torch.empty(1, heads, channels))
        self.bias = nn.Parameter(torch.zeros(channels))          # concat=False (or one head): [channels]
        self.lin_l = nn.Linear(channels, heads * channels, bias=True)
        self.lin_r = nn.Linear(channels, heads * channels, bias=True)
        self.lin_edge = nn.Linear(edge_dim, heads * channels, bias=False)
        for lin in (self.lin_l, self.lin_r, self.lin_edge):
            nn.init.xavier_uniform_(lin.weight)
            if lin.bias is not None:
                nn.init.zeros_(lin.bias)
        nn.init.xavier_uniform_(self.att)


class GAT_DSSE(_LazyMachinery, nn.Module):
    """networks.py:113-156, the as-shipped default model of dss2_run.py:86: (num_layers - 1) x [GATv2Conv(dim_feat, dim_feat, heads,
    edge_dim, add_self_loops, fill 'mean') + LeakyReLU()], Linear(dim_feat, dim_dense), Linear(dim_dense, dim_out), wrapped in a PyG
    `Sequential` whose children are called `module_{i}` - kept, so that reference checkpoints (`model.module_0.att`, ...) load.
    heads=1 (with either `concat`: one head concatenated = one head averaged) or heads 2..4 with concat=False (averaged heads);
    `self_loops`, `slope` and the three `nonlin` choices are free.  `dropout` (0 <= p < 1) is GATv2Conv's attention dropout, active in
    train() only like PyG's (unlike the MPN family's always-on nn.Dropout); each forward draws a fresh Philox seed from torch's global
    generator.  heads > 1 with concat=True raises (the reference's own stack cannot run it: channel mismatch)."""
    _dss2_attn_masks = None   # test hook: per layer uint8 [heads, Et + Nt] keep masks in the kernels' edge-key layout, consumed by the next forward

    def __init__(self, dim_feat, dim_dense, dim_out, num_layers, edge_dim, heads=1, concat=True, slope=0.2, self_loops=True, dropout=0.,
                 nonlin='leaky_relu', model='gat'):
        super().__init__()
        if model != 'gat':
            raise Exception('invalid model type')
        if nonlin not in ('relu', 'tanh', 'leaky_relu'):
            raise Exception('invalid activation type')
        if heads != 1 and concat:
            raise NotImplementedError("GAT_DSSE(heads > 1, concat=True): the reference's own stack cannot run this - every GATv2Conv maps "
                                      "dim_feat -> heads * dim_feat channels while the next layer expects dim_feat (networks.py:144-147)")
        if not 1 <= heads <= 4:
            raise NotImplementedError("GAT_DSSE kernels support heads in 1..4 (dss2_run.py:79 uses 1)")
        _check_attn_dropout(dropout, "GAT_DSSE")
        self.dim_out, self.num_layers, self.dim_feat, self.dim_dense, self.edge_dim = dim_out, num_layers, dim_feat, dim_dense, edge_dim
        self.dim_hidden = self.channels = dim_feat
        self.heads, self.concat, self.slope, self.dropout, self.loop = heads, concat, slope, dropout, self_loops
        self.nonlin_name = nonlin
        self.nonlin = {'relu': nn.ReLU, 'tanh': nn.Tanh, 'leaky_relu': nn.LeakyReLU}[nonlin]()
        self.model = nn.Module()
        i = 0
        for _ in range(num_layers - 1):
            self.model.add_module(f"module_{i}", _GATv2Params(dim_feat, edge_dim, heads))
            self.model.add_module(f"module_{i + 1}", self.nonlin)
            i += 2
        self.model.add_module(f"module_{i}", nn.Linear(dim_feat, dim_dense))
        self.model.add_module(f"module_{i + 1}", nn.Linear(dim_dense, dim_out))

    def _machinery(self):
        m = self.__dict__.get("_dss2_machinery")
        if m is None:
            from dss2 import gat
            spec = gat.GATSpec(dim_feat=self.dim_feat, dim_dense=self.dim_dense, dim_out=self.dim_out, num_layers=self.num_layers,
                               edge_dim=self.edge_dim, att_slope=float(self.slope), act_slope=float(getattr(self.nonlin, "negative_slope", 0.0)),
                               act=self.nonlin_name, self_loops=bool(self.loop), heads=int(self.heads), dropout=float(self.dropout))
            m = gat.make_machinery(spec)
            self.__dict__["_dss2_machinery"] = m
        return m

    def forward(self, x, edge_index, edge_attr):
        from dss2 import gat
        runner, pack = self._machinery()
        masks, self._dss2_attn_masks = self._dss2_attn_masks, None
        drop = self.training and runner.spec.dropout > 0.      # GATv2Conv: F.dropout(alpha, training=self.training)
        return gat.gat_apply(runner, pack, self._named_params(), x, edge_index, edge_attr, drop=drop, masks=masks)
