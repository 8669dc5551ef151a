"""GAT_DSSE, GINE_DSSE and gnn_dsse (gcn2 / fagcn / tagcn) on graphs and settings where kernels go wrong.

Graph catalogue (buses and edge lists; features are seeded random numbers):
  loops    the 9-bus graph of the GAT / GINE self-loop tests plus a second (4, 4) loop, the edge 6 -> 7 given twice and a 10th bus
           without edges: input self loops, a duplicate loop, a multi-edge, buses without in-edges, an isolated bus
  hub      one graph of 256 buses: bus 0 has 200 in-edges and 50 out-edges, a chain hangs off it (long softmax segments, the out-edge
           gather of the backward kernels); edge order shuffled
  hub_big  one graph of 1003 buses, bus 0 with 1000 in-edges: larger than a tile, so the batch structure has no tiles
  ragged   ober_sub and cigre14 graphs collated, with a 3-bus graph without edges in the middle
  large    ober_sub graphs, as many as make Nt exceed the grid-stride cap of the thread-per-bus kernels (multi_processor_count * 8 CTAs
           of 128 threads) by 10 %: every forward thread handles at least two buses, the backward kernels (one CTA per SM) far more
  peaked   (case option) attention vectors scaled by 40: GATv2 scores of a segment span more than 100, exp underflows for all but one
           coefficient (the max shift and the 1e-16 term of the softmax); FAConv's tanh saturates
The first edge is never a loop and never has its reverse in the list, so the models take the lists as one-way (MPN.is_directed).

CPU: every layer of the oracle (GATv2 with and without self loops, GINE, GCN2Conv and FAConv with add_self_loops on and off, TAGConv
K = 1..3) against the PyG shim in fp64 on every graph.  GPU: the public modules, forward and backward with a seeded upstream gradient:
output, every parameter gradient and the gradient w.r.t. x against the fp64 oracle (the fp32 noise from the oracle's fp32 run and two
edge-permuted ones), and bit-identical results when the step is repeated."""
import math
import os
import sys

import pytest
import torch

from conftest import ROOT, assert_fp32_parity, permute_edges
import dss2_oracle as orc
import networks
from test_attention_dropout import P as P_DROP, fagcn_forward, random_masks

SHIM = os.path.join(ROOT, "oracle", "pyg_shim")
GRAPHS = ("loops", "hub", "hub_big", "ragged", "large")
PEAK = 40.0


# ------------------------------------------------------------------------------------------------ graph catalogue
def _grid_edges(case):
    from dss2 import synth
    g = synth.synthetic_store(synth.load_grid(case), 1, seed=1).graph(0)
    return g["edge_index"], g["x"].size(0)


def _collate(parts):
    """Disjoint union of (edge_index, num_nodes) parts, graph-major like PyG's Batch."""
    eis, off = [], 0
    for ei, n in parts:
        eis.append(ei + off)
        off += n
    return torch.cat(eis, 1), off


def _large_batch_nodes(num_sms):
    """Buses of the `large` batch: 10 % above the grid-stride cap num_sms * 8 CTAs * 128 threads."""
    return math.ceil(1.1 * num_sms * 8 * 128)


def build_graph(name, num_sms=148):
    """(edge_index [2, E] int64, num_nodes) of a catalogue graph."""
    if name == "loops":
        ei = torch.tensor([[0, 1, 2, 2, 3, 5, 6, 6, 4, 4, 6], [1, 2, 3, 2, 1, 1, 7, 8, 4, 4, 7]])
        return ei, 10
    if name == "hub":
        src = list(range(1, 201)) + [0] * 50 + list(range(250, 255))
        dst = [0] * 200 + list(range(201, 251)) + list(range(251, 256))
        ei = torch.tensor([src, dst])
        perm = torch.randperm(ei.size(1) - 1, generator=torch.Generator().manual_seed(3)) + 1
        return torch.cat([ei[:, :1], ei[:, perm]], 1), 256
    if name == "hub_big":
        ei = torch.tensor([list(range(1, 1001)) + [0, 1001], [0] * 1000 + [1001, 1002]])
        return ei, 1003
    if name == "ragged":
        ober, cigre = _grid_edges("ober_sub"), _grid_edges("cigre14")
        return _collate([ober, cigre, (torch.zeros(2, 0, dtype=torch.long), 3), ober, cigre])
    if name == "large":
        ober = _grid_edges("ober_sub")
        return _collate([ober] * math.ceil(_large_batch_nodes(num_sms) / ober[1]))
    raise KeyError(name)


def features(n, e, fe, seed):
    g = torch.Generator().manual_seed(seed)
    return torch.randn(n, 8, generator=g, dtype=torch.float64), torch.randn(e, fe, generator=g, dtype=torch.float64)


# ------------------------------------------------------------------------------------------------ CPU: oracle layers against the PyG shim
def _shim_conv():
    if SHIM not in sys.path:
        sys.path.insert(0, SHIM)
    from torch_geometric.nn import conv
    return conv


def _head(sd, h, nl):
    i = 2 * (nl - 1)
    h = h @ sd[f"model.module_{i}.weight"].t() + sd[f"model.module_{i}.bias"]
    return h @ sd[f"model.module_{i + 1}.weight"].t() + sd[f"model.module_{i + 1}.bias"]


LAYERS = ["gatv2_loops", "gatv2_noloops", "gatv2_heads3", "gine", "gcn2_loops", "gcn2_noloops", "fagcn_loops", "fagcn_noloops",
          "tag_k1", "tag_k2", "tag_k3"]


ATTENTION_LAYERS = [l for l in LAYERS if l.startswith(("gatv2", "fagcn"))]


@pytest.mark.parametrize("graph,layer", [(g, l) for g in GRAPHS for l in LAYERS]
                         + [(g, l) for g in ("peaked_loops", "peaked_ragged") for l in ATTENTION_LAYERS])
def test_oracle_layer_matches_pyg_shim(graph, layer):
    """One conv layer + non-linearity + head of the oracle's model functions (num_layers = 2) against the shim's conv followed by the
    same non-linearity and head, fp64, on every catalogue graph."""
    conv = _shim_conv()
    peaked = graph.startswith("peaked_")
    ei, n = build_graph(graph.replace("peaked_", ""))
    x, ea = features(n, ei.size(1), 6, seed=7)
    f64 = torch.float64
    act = lambda t: torch.nn.functional.leaky_relu(t, 0.01)
    with torch.no_grad():
        if layer.startswith("gatv2"):
            heads, loops = (3 if layer == "gatv2_heads3" else 1), layer != "gatv2_noloops"
            sd = orc.init_gat_state_dict(num_layers=2, seed=4, heads=heads, dtype=f64)
            if peaked:
                sd["model.module_0.att"] *= PEAK
            m = conv.GATv2Conv(8, 8, heads=heads, concat=False, add_self_loops=loops, edge_dim=6).double()
            for k in ("att", "bias", "lin_l.weight", "lin_l.bias", "lin_r.weight", "lin_r.bias", "lin_edge.weight"):
                m.get_parameter(k).copy_(sd["model.module_0." + k])
            want = _head(sd, act(m(x, ei, ea)), 2)
            got = orc.gat_dsse_forward(sd, x, ei, ea, 2, self_loops=loops)
        elif layer == "gine":
            sd = orc.init_gine_state_dict(num_layers=2, seed=4, dtype=f64)
            sd["model.module_0.eps"] = torch.tensor([0.3], dtype=f64)
            lin = torch.nn.Linear(8, 8).double()
            lin.weight.copy_(sd["nn.weight"])
            lin.bias.copy_(sd["nn.bias"])
            m = conv.GINEConv(lin, eps=0.3, train_eps=True, edge_dim=6).double()
            m.lin.weight.copy_(sd["model.module_0.lin.weight"])
            m.lin.bias.copy_(sd["model.module_0.lin.bias"])
            m.eps.copy_(sd["model.module_0.eps"])         # (filled in fp32 before .double())
            want = _head(sd, act(m(x, ei, ea)), 2)
            got = orc.gine_dsse_forward(sd, x, ei, ea, 2)
        elif layer.startswith("gcn2") or layer.startswith("fagcn"):
            model, loops = layer.split("_")[0], layer.endswith("_loops")
            sd = orc.init_gnn_state_dict(model, num_layers=2, seed=4, dtype=f64)
            if model == "gcn2":
                m = conv.GCN2Conv(8, alpha=0.1, add_self_loops=loops).double()
                m.weight1.copy_(sd["model.module_0.weight1"])
            else:
                if peaked:
                    sd["model.module_0.att_l.weight"] *= PEAK
                    sd["model.module_0.att_r.weight"] *= PEAK
                m = conv.FAConv(8, eps=0.1, add_self_loops=loops).double()
                m.att_l.weight.copy_(sd["model.module_0.att_l.weight"])
                m.att_r.weight.copy_(sd["model.module_0.att_r.weight"])
            want = _head(sd, act(m(x, x, ei)), 2)
            got = orc.gnn_dsse_forward(sd, x, ei, 2, model=model, add_self_loops=loops)
        else:
            K = int(layer[-1])
            sd = orc.init_gnn_state_dict("tagcn", num_layers=2, K=K, seed=4, dtype=f64)
            m = conv.TAGConv(8, 8, K=K).double()
            m.bias.copy_(sd["model.module_0.bias"])
            for k in range(K + 1):
                m.lins[k].weight.copy_(sd[f"model.module_0.lins.{k}.weight"])
            want = _head(sd, act(m(x, ei)), 2)
            got = orc.gnn_dsse_forward(sd, x, ei, 2, model="tagcn", K=K)
    assert torch.allclose(got, want, rtol=1e-12, atol=1e-12), float((got - want).abs().max())


@pytest.mark.parametrize("nonlin", ["relu", "tanh", "leaky_relu"])
def test_oracle_gnn_nonlin(nonlin):
    """gnn_dsse_forward's `nonlin` is the module's activation after every conv (leaky_relu: PyTorch's default slope 0.01)."""
    ei, n = build_graph("loops")
    x, _ = features(n, ei.size(1), 1, seed=2)
    sd = orc.init_gnn_state_dict("gcn2", num_layers=3, seed=1, dtype=torch.float64)
    act = {"relu": torch.relu, "tanh": torch.tanh, "leaky_relu": lambda t: torch.nn.functional.leaky_relu(t, 0.01)}[nonlin]
    h = x
    for l in range(2):
        ei2, w = orc.gcn_norm_self_loops(ei, n, x.dtype)
        prop = orc.segment_sum(w.view(-1, 1) * h[ei2[0]], ei2[1], n)
        h = act((0.9 * prop + 0.1 * x) @ sd[f"model.module_{2 * l}.weight1"])
    got = orc.gnn_dsse_forward(sd, x, ei, 3, nonlin=nonlin)
    assert torch.allclose(got, _head(sd, h, 3), rtol=1e-12, atol=1e-12)


def test_catalogue_shapes():
    """The graphs are what the catalogue says they are."""
    ei, n = build_graph("loops")
    assert int((ei[0] == ei[1]).sum()) == 3 and n == 10 and not bool(((ei[0] == 9) | (ei[1] == 9)).any())
    ei, n = build_graph("hub")
    assert n == 256 and int((ei[1] == 0).sum()) == 200 and int((ei[0] == 0).sum()) == 50
    ei, n = build_graph("hub_big")
    assert n > 256 and int((ei[1] == 0).sum()) == 1000
    ei, n = build_graph("large", num_sms=148)
    assert n > 1.1 * 148 * 8 * 128
    for g in GRAPHS:
        ei, n = build_graph(g)
        assert orc.needs_reverse_edges(ei) and ei[0, 0] != ei[1, 0], g


# ------------------------------------------------------------------------------------------------ GPU: the modules against the fp64 oracle
# name -> (family, graph, constructor options, (dim_dense, dim_out), test options).  Pairwise coverage: every line reaches something the
# golden runs do not (edge_dim 1 / 3 / 8, heads 4, 9 convs > 8 weight slots, self_loops off, train_eps, add_self_loops on / off,
# TAGConv K = 1..3, relu / tanh, heads other than 8 -> 32 -> 2).  The `large` cases use tanh where the model allows it, so that the
# millions of activations hold no kink at which fp32 and fp64 may pick different sides.
CASES = {
    "gat_e1_loops": ("gat", "loops", dict(edge_dim=1), (32, 3), {}),
    "gat_e3_hub": ("gat", "hub", dict(edge_dim=3), (16, 2), {}),
    "gat_e8_ragged_relu": ("gat", "ragged", dict(edge_dim=8, nonlin="relu"), (24, 1), {}),
    "gat_heads4_hub_big": ("gat", "hub_big", dict(heads=4, concat=False), (20, 8), {}),
    "gat_heads4_loops_tanh": ("gat", "loops", dict(heads=4, concat=False, nonlin="tanh"), (8, 8), {}),
    "gat_l10_ragged": ("gat", "ragged", dict(num_layers=10), (32, 2), {}),
    "gat_noloops_loops": ("gat", "loops", dict(self_loops=False, edge_dim=3), (32, 2), {}),
    "gat_large": ("gat", "large", dict(num_layers=3, nonlin="tanh"), (32, 2), {}),
    "gat_peaked_loops": ("gat", "loops", {}, (32, 2), dict(peaked=True)),
    "gat_peaked_ragged_heads2": ("gat", "ragged", dict(heads=2, concat=False), (32, 2), dict(peaked=True)),
    "gine_e1_traineps_loops": ("gine", "loops", dict(edge_dim=1, train_eps=True), (32, 3), {}),
    "gine_e8_traineps_hub": ("gine", "hub", dict(edge_dim=8, train_eps=True), (16, 2), {}),
    "gine_hub_big": ("gine", "hub_big", {}, (24, 1), {}),
    "gine_e8_ragged": ("gine", "ragged", dict(edge_dim=8), (20, 8), {}),
    "gine_large": ("gine", "large", dict(num_layers=3), (8, 8), {}),
    "gcn2_loops": ("gnn", "loops", dict(model="gcn2"), (32, 3), {}),
    "gcn2_noloops_loops_tanh": ("gnn", "loops", dict(model="gcn2", add_self_loops=False, nonlin="tanh"), (32, 2), {}),
    "gcn2_hub_relu": ("gnn", "hub", dict(model="gcn2", nonlin="relu"), (16, 2), {}),
    "gcn2_noloops_hub_big": ("gnn", "hub_big", dict(model="gcn2", add_self_loops=False), (24, 1), {}),
    "gcn2_ragged": ("gnn", "ragged", dict(model="gcn2"), (8, 8), {}),
    "gcn2_large": ("gnn", "large", dict(model="gcn2", num_layers=3, nonlin="tanh"), (32, 2), {}),
    "fagcn_loops_tanh": ("gnn", "loops", dict(model="fagcn", nonlin="tanh"), (20, 8), {}),
    "fagcn_noloops_loops_relu": ("gnn", "loops", dict(model="fagcn", add_self_loops=False, nonlin="relu"), (8, 8), {}),
    "fagcn_hub_big": ("gnn", "hub_big", dict(model="fagcn"), (32, 2), {}),
    "fagcn_noloops_hub_tanh": ("gnn", "hub", dict(model="fagcn", add_self_loops=False, nonlin="tanh"), (16, 2), {}),
    "fagcn_peaked_loops": ("gnn", "loops", dict(model="fagcn"), (32, 2), dict(peaked=True)),
    "fagcn_peaked_ragged_relu": ("gnn", "ragged", dict(model="fagcn", nonlin="relu"), (32, 3), dict(peaked=True)),
    "fagcn_large": ("gnn", "large", dict(model="fagcn", num_layers=3, nonlin="tanh"), (32, 2), {}),
    "tagcn_k1_loops_relu": ("gnn", "loops", dict(model="tagcn", K=1, nonlin="relu"), (32, 2), {}),
    "tagcn_k2_hub_tanh": ("gnn", "hub", dict(model="tagcn", K=2, nonlin="tanh"), (24, 1), {}),
    "tagcn_k3_ragged": ("gnn", "ragged", dict(model="tagcn", K=3), (20, 8), {}),
    "tagcn_k2_hub_big": ("gnn", "hub_big", dict(model="tagcn", K=2), (32, 3), {}),
    "tagcn_k3_large": ("gnn", "large", dict(model="tagcn", K=3, num_layers=3, nonlin="tanh"), (32, 2), {}),
    "fagcn_dropout_loops": ("gnn", "loops", dict(model="fagcn", dropout=P_DROP), (32, 2), dict(masks=True)),
    "fagcn_dropout_noloops_loops": ("gnn", "loops", dict(model="fagcn", dropout=P_DROP, add_self_loops=False), (16, 2), dict(masks=True)),
}
DEFAULT_LAYERS = 5


def _num_sms():
    return torch.cuda.get_device_properties(0).multi_processor_count


def _setup(name, seed=9):
    """(module on the device in train(), reference-named fp32 state_dict, case options) of a case."""
    family, _, opts, (dd, do), extra = CASES[name]
    opts = dict(opts)
    nl = opts.pop("num_layers", DEFAULT_LAYERS)
    if family == "gat":
        sd = orc.init_gat_state_dict(dim_dense=dd, dim_out=do, num_layers=nl, edge_dim=opts.get("edge_dim", 6), heads=opts.get("heads", 1),
                                     seed=seed)
        if extra.get("peaked"):
            for l in range(nl - 1):
                sd[f"model.module_{2 * l}.att"] = sd[f"model.module_{2 * l}.att"] * PEAK
        opts.setdefault("edge_dim", 6)
        model = networks.GAT_DSSE(dim_feat=8, dim_dense=dd, dim_out=do, num_layers=nl, **opts)
        model.load_state_dict(sd, strict=True)
    elif family == "gine":
        sd = orc.init_gine_state_dict(dim_dense=dd, dim_out=do, num_layers=nl, edge_dim=opts.get("edge_dim", 6), seed=seed)
        if opts.get("train_eps"):
            for l in range(nl - 1):     # one trainable eps per layer, each its own value
                sd[f"model.module_{2 * l}.eps"] = torch.tensor([0.1 + 0.2 * l])
        opts.setdefault("edge_dim", 6)
        model = networks.GINE_DSSE(dim_feat=8, dim_dense=dd, dim_out=do, num_layers=nl, eps=0.1 if opts.get("train_eps") else 0., **opts)
        with torch.no_grad():
            for k, p in model.named_parameters():
                p.copy_(sd[k])
        assert set(dict(model.named_parameters())) == set(sd)
    else:
        sd = orc.init_gnn_state_dict(opts["model"], dim_dense=dd, dim_out=do, num_layers=nl, K=opts.get("K", 3), seed=seed)
        if extra.get("peaked"):
            for l in range(nl - 1):
                for k in ("att_l.weight", "att_r.weight"):
                    sd[f"model.module_{2 * l}.{k}"] = sd[f"model.module_{2 * l}.{k}"] * PEAK
        model = networks.gnn_dsse(dim_feat=8, dim_dense=dd, dim_out=do, num_layers=nl, **opts)
        model.load_state_dict(sd, strict=True)
    return model.cuda().train(), sd, dict(CASES[name][2], num_layers=nl)


def _oracle(name, sd, opts, x, ei, ea, go, dtype, masks=None):
    """Reference forward, then backward of sum(out * go): (out, parameter gradients, gradient w.r.t. x)."""
    family = CASES[name][0]
    nl = opts["num_layers"]
    p = {k: v.to(dtype).clone().requires_grad_(True) for k, v in sd.items()}
    xin = x.to(dtype).clone().requires_grad_(True)
    if family == "gat":
        out = orc.gat_dsse_forward(p, xin, ei, ea.to(dtype), nl, nonlin=opts.get("nonlin", "leaky_relu"), self_loops=opts.get("self_loops", True))
    elif family == "gine":
        out = orc.gine_dsse_forward(p, xin, ei, ea.to(dtype), nl)
    elif masks is not None:
        out = fagcn_forward(p, xin, ei, nl, self_loops=opts.get("add_self_loops", True), masks=masks, p=opts["dropout"])
    else:
        out = orc.gnn_dsse_forward(p, xin, ei, nl, model=opts["model"], K=opts.get("K", 3), add_self_loops=opts.get("add_self_loops", True),
                                   nonlin=opts.get("nonlin", "leaky_relu"))
    (out * go.to(dtype)).sum().backward()
    return out.detach(), {k: v.grad for k, v in p.items()}, xin.grad


def _step(name, model, x, ei, ea, go, masks):
    """Forward and backward of the module with upstream gradient go: (out, parameter gradients, gradient w.r.t. x)."""
    model.zero_grad()
    xin = x.clone().requires_grad_(True)
    if masks is not None:
        model._dss2_attn_masks = masks
    out = model(xin, ei, ea) if CASES[name][0] != "gnn" else model(xin, ei)
    out.backward(go)
    return out.detach().clone(), {k: p.grad.clone() for k, p in model.named_parameters()}, xin.grad.clone()


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(CASES))
def test_module_matches_oracle_on_edge_case_graphs(name):
    from dss2 import ops
    family, graph, _, (dd, do), extra = CASES[name]
    model, sd, opts = _setup(name)
    ei, n = build_graph(graph, num_sms=_num_sms())
    x, ea = features(n, ei.size(1), opts.get("edge_dim", 6), seed=21)
    x, ea = x.float(), ea.float()
    go = torch.randn(n, do, generator=torch.Generator().manual_seed(5))
    masks = random_masks(opts["num_layers"], 1, ei.size(1) + n, opts["dropout"], seed=23) if extra.get("masks") else None
    xg, eig, eag, gog = x.cuda(), ei.cuda(), ea.cuda(), go.cuda()
    # the batch structure is what the graph is meant to stress (`loops` has no tiles either: its edge list is not graph-major)
    bg = ops.resolve_graph(eig, n)
    assert bg.c.undirected == 1
    if graph in ("hub_big", "hub", "ragged", "large"):
        assert (bg.c.num_tiles == 0) == (graph == "hub_big")
    if graph == "large":
        assert n > _num_sms() * 8 * 128
    ours = _step(name, model, xg, eig, eag, gog, masks)
    # fixed-order reductions: the same step again gives the same bits
    again = _step(name, model, xg, eig, eag, gog, masks)
    assert torch.equal(ours[0], again[0]) and torch.equal(ours[2], again[2])
    for k in ours[1]:
        assert torch.equal(ours[1][k], again[1][k]), k
    r64 = _oracle(name, sd, opts, x, ei, ea, go, torch.float64, masks)
    runs = [_oracle(name, sd, opts, x, ei, ea, go, torch.float32, masks)]
    for s_ in (1, 2):     # the same graph with its edge list in another order: another valid fp32 summation order
        pb = permute_edges({"edge_index": ei, "edge_attr": ea}, s_)
        pm = None
        if masks is not None:
            perm = torch.randperm(ei.size(1), generator=torch.Generator().manual_seed(s_))
            assert torch.equal(pb["edge_index"], ei[:, perm])
            pm = [torch.cat([m[:, :ei.size(1)][:, perm], m[:, ei.size(1):]], 1) for m in masks]
        runs.append(_oracle(name, sd, opts, x, pb["edge_index"], pb["edge_attr"], go, torch.float32, pm))
    assert_fp32_parity(ours[0], [r[0] for r in runs], r64[0], "out")
    nl = opts["num_layers"]
    head_w2 = sd[f"model.module_{2 * (nl - 1) + 1}.weight"].double()
    # the head's bias gradients are column sums over the buses of go @ W2 and go: judged as sums (conftest)
    terms = {f"model.module_{2 * (nl - 1)}.bias": go.double() @ head_w2, f"model.module_{2 * (nl - 1) + 1}.bias": go}
    for k in sd:
        assert_fp32_parity(ours[1][k], [r[1][k] for r in runs], r64[1][k], k, sum_of=terms.get(k))
    assert_fp32_parity(ours[2], [r[2] for r in runs], r64[2], "grad_x")
