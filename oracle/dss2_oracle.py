"""CPU oracle for the DSS2 hot path - TEST INFRASTRUCTURE, NOT PRODUCT CODE.

A plain-PyTorch (CPU, fp32 or fp64) restatement of the reference algorithm on the north-star path:
PyG-style batching, the EdgeAggregation + TAGConv "PowerFlowNet" models and the physics-informed
WLS loss.  Only `tests/`, `__graft_entry__.smoke()` and the `cpu_baseline` / `--impl reference`
legs of `bench.py` may import this file; the product package never does.

Every function cites the reference lines it follows (paths relative to the reference root).  The
PyG pieces (`MessagePassing.propagate`, `TAGConv`, `gcn_norm`, `scatter`, `Batch.from_data_list`)
restate torch_geometric's published semantics, because torch_geometric is an un-vendored,
un-pinned dependency (reference README.md:31) that is not installable here.

How it is pinned (SURVEY.md 8c):
  * `get_pflow` / bus injections: against the pandapower-solved columns of the reference's own
    `data/cigre14` pickles (fixtures in tests/golden/, test_oracle_golden.py).
  * everything else: against outputs of the reference's own `networks.py` / `data.py` executed
    verbatim in the build container over `oracle/pyg_shim` (tests/golden/make_golden.py wrote them).
  * against real PyG: PARITY UNPINNED (no PyG available, the reference holds no tests).

Functional style on purpose: models are evaluated from a `state_dict` with the reference's
parameter names, so the same weights drive the reference, this oracle and the CUDA path.
"""
import math

import torch

# --------------------------------------------------------------------------------------------
# batching  (PyG Batch.from_data_list as used by dss2_run.py:68-69,134)
# --------------------------------------------------------------------------------------------


def collate(graphs):
    """Disjoint-union batch of `graphs` = list of dicts {x[N,11], edge_index[2,E] i64, edge_attr[E,13], y[N,2]}.

    PyG semantics: features concatenated graph-major on dim 0, `edge_index` concatenated on dim 1
    with the running node count added, per-graph edge order preserved; `batch[n]` = graph id of
    node n; `ptr` = exclusive prefix sum of node counts (length B+1)."""
    xs, eas, ys, eis, bvec, ptr = [], [], [], [], [], [0]
    for g, gr in enumerate(graphs):
        n = gr["x"].shape[0]
        xs.append(gr["x"])
        eas.append(gr["edge_attr"])
        ys.append(gr["y"])
        eis.append(gr["edge_index"] + ptr[-1])
        bvec.append(torch.full((n,), g, dtype=torch.long))
        ptr.append(ptr[-1] + n)
    return {
        "x": torch.cat(xs, 0), "edge_attr": torch.cat(eas, 0), "y": torch.cat(ys, 0),
        "edge_index": torch.cat(eis, 1), "batch": torch.cat(bvec, 0),
        "ptr": torch.tensor(ptr, dtype=torch.long),
    }


# --------------------------------------------------------------------------------------------
# graph helpers
# --------------------------------------------------------------------------------------------


def segment_sum(values, index, num_rows):
    """PyG `scatter(..., reduce='sum')`: zeros(num_rows, ...).scatter_add_ along dim 0."""
    shape = (num_rows,) + tuple(values.shape[1:])
    idx = index.view((-1,) + (1,) * (values.dim() - 1)).expand_as(values)
    return values.new_zeros(shape).scatter_add_(0, idx, values)


def needs_reverse_edges(edge_index):
    """networks.py:236-238 `is_directed`: looks only at edge 0 = (s0 -> t0) and reports "directed"
    when s0 does not occur among the targets of edges that leave t0."""
    s0, t0 = edge_index[0, 0], edge_index[1, 0]
    targets_of_t0 = edge_index[1, edge_index[0] == t0]
    return not bool((targets_of_t0 == s0).any())


def undirect(edge_index, edge_attr):
    """networks.py:240-258: append every edge reversed after all forward edges; the reversed copy
    of the attributes flips the sign of columns 0 and 2 (normalised P and Q flow) only (:252)."""
    if not needs_reverse_edges(edge_index):
        return edge_index, edge_attr
    both = torch.cat([edge_index, edge_index.flip(0)], dim=1)
    sign = edge_attr.new_ones(edge_attr.shape[1])
    sign[0] = -1.0
    sign[2] = -1.0
    # multiplying by -1/+1 is exact and gives -0.0 for masked zeros exactly like unary minus
    return both, torch.cat([edge_attr, edge_attr * sign], dim=0)


def gcn_weights(edge_index, num_nodes, dtype):
    """PyG gcn_norm(add_self_loops=False) as TAGConv calls it: in-degree by target,
    w_e = deg[src]^-1/2 * deg[dst]^-1/2, infinities zeroed."""
    src, dst = edge_index[0], edge_index[1]
    deg = segment_sum(torch.ones(src.numel(), dtype=dtype), dst, num_nodes)
    dis = deg.pow(-0.5)
    dis = torch.where(torch.isinf(dis), torch.zeros_like(dis), dis)
    return dis[src] * dis[dst]


# --------------------------------------------------------------------------------------------
# layers  (networks.py:159-209 EdgeAggregation; PyG TAGConv; networks.py:268-269 dropout/relu)
# --------------------------------------------------------------------------------------------


def edge_aggregation(x, edge_index, edge_attr, w1, b1, w2, b2):
    """networks.py:176-181 + :206 with aggr='add' (:164): message MLP on [x_target | x_source | a_e],
    summed into the target node.  The degree norm of :196-200 never reaches `message` and is omitted."""
    src, dst = edge_index[0], edge_index[1]
    feats = torch.cat([x.index_select(0, dst), x.index_select(0, src), edge_attr], dim=-1)
    hidden = torch.relu(torch.addmm(b1, feats, w1.t()))
    msg = torch.addmm(b2, hidden, w2.t())
    return segment_sum(msg, dst, x.shape[0])


def tag_conv(x, edge_index, weights, bias, edge_w=None):
    """PyG TAGConv.forward: out = sum_k (A_hat^k x) W_k^T + b with A_hat from gcn_weights, hop by hop.
    `edge_w` may carry precomputed gcn weights; PyG itself recomputes them in every layer."""
    if edge_w is None:
        edge_w = gcn_weights(edge_index, x.shape[0], x.dtype)
    src, dst = edge_index[0], edge_index[1]
    out = x @ weights[0].t()
    for wk in weights[1:]:
        x = segment_sum(edge_w.unsqueeze(1) * x.index_select(0, src), dst, x.shape[0])
        out = out + x @ wk.t()
    return out + bias


def dropout_relu(x, p, mask=None, generator=None, gate=None, trace=None):
    """networks.py:268-269: a freshly built nn.Dropout is always in training mode, so the mask is
    applied in eval too.  x * (mask / (1 - p)) is torch's CPU formulation.  `mask` (0/1, same shape)
    injects a recorded mask; otherwise one is drawn (p=0 -> identity).

    Test hooks (not reference behaviour): `trace` collects the pre-activation (dropout applied, before the
    ReLU); `gate` (0/1) REPLACES mask and ReLU by a fixed pass pattern, y = x * gate / (1 - p) - used to
    evaluate the gradient at the other side of a ReLU tie (pre-activation ~1e-7 in one fp32
    implementation, <= 0 in another), where relu' is implementation dependent."""
    if gate is not None:
        return x * (gate.to(x.dtype) / (1.0 - p))
    if p > 0.0:
        if mask is None:
            mask = torch.empty_like(x).bernoulli_(1.0 - p, generator=generator)
        x = x * (mask.to(x.dtype) / (1.0 - p))
    if trace is not None:
        trace.append(x.detach())
    return torch.relu(x)


# --------------------------------------------------------------------------------------------
# models, evaluated from a state_dict with the reference parameter names
# --------------------------------------------------------------------------------------------


def _layer_params(sd, prefix):
    k = 0
    ws = []
    while f"{prefix}lins.{k}.weight" in sd:
        ws.append(sd[f"{prefix}lins.{k}.weight"])
        k += 1
    return ws, sd[f"{prefix}bias"]


def mpn_forward(sd, prefix, x, edge_index, edge_attr, p_drop, skip, masks=None, generator=None, gates=None, trace=None):
    """networks.py:260-273 (MPN) and :323-338 (SkipMPN, `skip=True` adds the input back, :336).
    `masks`: optional list with one 0/1 tensor per hidden TAG layer (`gates`, `trace`: test hooks of dropout_relu)."""
    x_in = x
    ei2, ea2 = undirect(edge_index, edge_attr)
    x = edge_aggregation(x, ei2, ea2,
                         sd[f"{prefix}edge_aggr.edge_aggr.0.weight"], sd[f"{prefix}edge_aggr.edge_aggr.0.bias"],
                         sd[f"{prefix}edge_aggr.edge_aggr.2.weight"], sd[f"{prefix}edge_aggr.edge_aggr.2.bias"])
    n_layers = 0
    while f"{prefix}convs.{n_layers}.bias" in sd:
        n_layers += 1
    for layer in range(n_layers):
        ws, b = _layer_params(sd, f"{prefix}convs.{layer}.")
        x = tag_conv(x, ei2, ws, b)
        if layer < n_layers - 1:
            x = dropout_relu(x, p_drop, None if masks is None else masks[layer], generator,
                             gate=None if gates is None else gates[layer], trace=trace)
    return x_in + x if skip else x


def pfn_forward(sd, x, edge_index, edge_attr, p_drop, skip=True, masks=None, generator=None, gates=None, trace=None):
    """networks.py:359-363 (PFN, skip=False) / :384-388 (SkipPFN, skip=True): L stacked sub-nets that
    all receive the same raw edge attributes; the last one is always a plain MPN (:355,:380)."""
    n_sub = 0
    while f"mpns.{n_sub}.convs.0.bias" in sd:
        n_sub += 1
    for s in range(n_sub):
        sub_masks = None if masks is None else masks[s]
        x = mpn_forward(sd, f"mpns.{s}.", x, edge_index, edge_attr, p_drop,
                        skip=(skip and s < n_sub - 1), masks=sub_masks, generator=generator,
                        gates=None if gates is None else gates[s], trace=trace)
    return x


def init_state_dict(kind="SkipPFN", dim_featn=8, dim_feate=6, dim_out=2, dim_hid=32, n_gnn_layers=8, K=2, L=5,
                    seed=0, dtype=torch.float32):
    """Random parameters with the reference's names/shapes (SURVEY.md 5, checkpoint row).  The init
    distribution (uniform +-1/sqrt(fan_in), TAG bias zero) matches torch/PyG Linear defaults, but parity
    always goes through state_dict transfer, never seed replay.  kind: MPN | SkipMPN | PFN | SkipPFN."""
    g = torch.Generator().manual_seed(seed)
    sd = {}

    def lin(name, fan_out, fan_in, bias):
        bound = 1.0 / math.sqrt(fan_in)
        sd[f"{name}.weight"] = ((torch.rand(fan_out, fan_in, generator=g, dtype=torch.float64) * 2 - 1) * bound).to(dtype)
        if bias:
            sd[f"{name}.bias"] = ((torch.rand(fan_out, generator=g, dtype=torch.float64) * 2 - 1) * bound).to(dtype)

    def mpn(prefix, d_out):
        lin(f"{prefix}edge_aggr.edge_aggr.0", dim_hid, 2 * dim_featn + dim_feate, True)
        lin(f"{prefix}edge_aggr.edge_aggr.2", dim_hid, dim_hid, True)
        for layer in range(n_gnn_layers):
            cout = d_out if layer == n_gnn_layers - 1 else dim_hid
            sd[f"{prefix}convs.{layer}.bias"] = torch.zeros(cout, dtype=dtype)
            for k in range(K + 1):
                lin(f"{prefix}convs.{layer}.lins.{k}", cout, dim_hid, False)

    if kind in ("MPN", "SkipMPN"):
        mpn("", dim_out)
    else:
        for s in range(L):
            mpn(f"mpns.{s}.", dim_out if s == L - 1 else dim_featn)
    return sd


# --------------------------------------------------------------------------------------------
# GAT_DSSE (networks.py:113-156): 7 x (GATv2Conv(8, 8, heads=1, edge_dim=6, add_self_loops, fill 'mean') + LeakyReLU(0.01)),
# Linear(8, 32), Linear(32, 2).  SURVEY.md 8f-1: the as-shipped default model of dss2_run.py:86.
# --------------------------------------------------------------------------------------------


def gatv2_layer(x, edge_index, edge_attr, w_l, b_l, w_r, b_r, w_e, att, bias, slope=0.2, self_loops=True):
    """One GATv2Conv (heads = 1) on the ONE-WAY edge list the script passes (networks.py:146 gets `data.edge_index` as is).
    Self loops of the input are dropped, then one loop per node is appended whose attribute is the mean of the attributes of the
    edges pointing at the node (0 without any).  Segment softmax as PyG: max-shifted exp / (sum + 1e-16)."""
    n = x.size(0)
    if self_loops:
        keep = edge_index[0] != edge_index[1]
        src, dst, ea = edge_index[0][keep], edge_index[1][keep], edge_attr[keep]
        cnt = segment_sum(torch.ones(dst.numel(), 1, dtype=x.dtype), dst, n).clamp(min=1)
        loop_attr = segment_sum(ea, dst, n) / cnt
        loop = torch.arange(n)
        src, dst, ea = torch.cat([src, loop]), torch.cat([dst, loop]), torch.cat([ea, loop_attr])
    else:   # add_self_loops=False: the edge list as given (GATv2Conv.forward only touches loops under add_self_loops)
        src, dst, ea = edge_index[0], edge_index[1], edge_attr
    x_l = x @ w_l.t() + b_l
    x_r = x @ w_r.t() + b_r
    s = torch.nn.functional.leaky_relu(x_r[dst] + x_l[src] + ea @ w_e.t(), slope)
    score = (s * att.view(1, -1)).sum(-1)
    smax = torch.full((n,), float("-inf"), dtype=x.dtype).scatter_reduce(0, dst, score.detach(), reduce="amax", include_self=True)
    ex = (score - smax[dst]).exp()
    den = segment_sum(ex.view(-1, 1), dst, n).view(-1) + 1e-16
    alpha = ex / den[dst]
    return segment_sum(x_l[src] * alpha.view(-1, 1), dst, n) + bias


def gat_dsse_forward(sd, x, edge_index, edge_attr, num_layers=8, nonlin="leaky_relu", slope=0.2, self_loops=True):
    """GAT_DSSE.forward (networks.py:155-156) from a reference-named state_dict (`model.module_{i}.*`, PyG Sequential naming)."""
    h = x
    for l in range(num_layers - 1):
        p = f"model.module_{2 * l}."
        H = sd[p + "att"].shape[1]
        if H == 1:
            h = gatv2_layer(h, edge_index, edge_attr, sd[p + "lin_l.weight"], sd[p + "lin_l.bias"], sd[p + "lin_r.weight"], sd[p + "lin_r.bias"],
                            sd[p + "lin_edge.weight"], sd[p + "att"], sd[p + "bias"], slope=slope, self_loops=self_loops)
        else:
            # heads > 1, concat=False (GATv2Conv: out.mean(dim=1) + bias): head k owns rows [k C, (k+1) C) of lin_l / lin_r / lin_edge
            # and att[0, k]; the heads do not interact before the mean
            c = h.size(1)
            heads = [gatv2_layer(h, edge_index, edge_attr, sd[p + "lin_l.weight"][k * c:(k + 1) * c], sd[p + "lin_l.bias"][k * c:(k + 1) * c],
                                 sd[p + "lin_r.weight"][k * c:(k + 1) * c], sd[p + "lin_r.bias"][k * c:(k + 1) * c],
                                 sd[p + "lin_edge.weight"][k * c:(k + 1) * c], sd[p + "att"][0, k], 0.0, slope=slope, self_loops=self_loops)
                     for k in range(H)]
            h = torch.stack(heads, 1).mean(dim=1) + sd[p + "bias"]
        h = {"leaky_relu": lambda t: torch.nn.functional.leaky_relu(t, 0.01), "relu": torch.relu, "tanh": torch.tanh}[nonlin](h)   # :130-137
    i = 2 * (num_layers - 1)
    h = h @ sd[f"model.module_{i}.weight"].t() + sd[f"model.module_{i}.bias"]
    return h @ sd[f"model.module_{i + 1}.weight"].t() + sd[f"model.module_{i + 1}.bias"]


def init_gat_state_dict(dim_feat=8, dim_dense=32, dim_out=2, num_layers=8, edge_dim=6, seed=0, dtype=torch.float32, heads=1):
    """Random GAT_DSSE parameters with the reference's names/shapes; all biases non-zero so every path is exercised."""
    g = torch.Generator().manual_seed(seed)

    def u(*shape, bound):
        return ((torch.rand(*shape, generator=g, dtype=torch.float64) * 2 - 1) * bound).to(dtype)

    sd = {}
    for l in range(num_layers - 1):
        p = f"model.module_{2 * l}."
        sd[p + "att"] = u(1, heads, dim_feat, bound=0.8)
        sd[p + "bias"] = u(dim_feat, bound=0.1)
        sd[p + "lin_l.weight"] = u(heads * dim_feat, dim_feat, bound=0.6)
        sd[p + "lin_l.bias"] = u(heads * dim_feat, bound=0.1)
        sd[p + "lin_r.weight"] = u(heads * dim_feat, dim_feat, bound=0.6)
        sd[p + "lin_r.bias"] = u(heads * dim_feat, bound=0.1)
        sd[p + "lin_edge.weight"] = u(heads * dim_feat, edge_dim, bound=0.6)
    i = 2 * (num_layers - 1)
    sd[f"model.module_{i}.weight"] = u(dim_dense, dim_feat, bound=1.0 / math.sqrt(dim_feat))
    sd[f"model.module_{i}.bias"] = u(dim_dense, bound=1.0 / math.sqrt(dim_feat))
    sd[f"model.module_{i + 1}.weight"] = u(dim_out, dim_dense, bound=1.0 / math.sqrt(dim_dense))
    sd[f"model.module_{i + 1}.bias"] = u(dim_out, bound=1.0 / math.sqrt(dim_dense))
    return sd


# --------------------------------------------------------------------------------------------
# GINE_DSSE (networks.py:71-111): 7 x (GINEConv(nn = ONE Linear(8, 8) shared by all layers, eps, edge_dim=6) + LeakyReLU(0.01)),
# Linear(8, 32), Linear(32, 2).  SURVEY.md 8f-1.
# --------------------------------------------------------------------------------------------


def gine_dsse_forward(sd, x, edge_index, edge_attr, num_layers=8):
    """GINE_DSSE.forward (networks.py:110-111) from a reference-named state_dict: `nn.*` (the shared Linear), per layer
    `model.module_{2l}.lin.*` (edge Linear, with bias) and the buffer `model.module_{2l}.eps`; one-way edge list, no self-loop handling."""
    n = x.size(0)
    src, dst = edge_index[0], edge_index[1]
    h = x
    for l in range(num_layers - 1):
        p = f"model.module_{2 * l}."
        eps = sd[p + "eps"].to(x.dtype) if (p + "eps") in sd else torch.zeros(1, dtype=x.dtype)
        msg = torch.relu(h[src] + edge_attr @ sd[p + "lin.weight"].t() + sd[p + "lin.bias"])
        agg = segment_sum(msg, dst, n)
        h = (agg + (1 + eps) * h) @ sd["nn.weight"].t() + sd["nn.bias"]
        h = torch.nn.functional.leaky_relu(h, 0.01)
    i = 2 * (num_layers - 1)
    h = h @ sd[f"model.module_{i}.weight"].t() + sd[f"model.module_{i}.bias"]
    return h @ sd[f"model.module_{i + 1}.weight"].t() + sd[f"model.module_{i + 1}.bias"]


def init_gine_state_dict(dim_feat=8, dim_dense=32, dim_out=2, num_layers=8, edge_dim=6, seed=0, dtype=torch.float32):
    """Random GINE_DSSE parameters under the names named_parameters() reports (shared `nn.*` once)."""
    g = torch.Generator().manual_seed(seed)

    def u(*shape, bound):
        return ((torch.rand(*shape, generator=g, dtype=torch.float64) * 2 - 1) * bound).to(dtype)

    sd = {"nn.weight": u(dim_feat, dim_feat, bound=0.45), "nn.bias": u(dim_feat, bound=0.1)}
    for l in range(num_layers - 1):
        p = f"model.module_{2 * l}."
        sd[p + "lin.weight"] = u(dim_feat, edge_dim, bound=0.4)
        sd[p + "lin.bias"] = u(dim_feat, bound=0.1)
    i = 2 * (num_layers - 1)
    sd[f"model.module_{i}.weight"] = u(dim_dense, dim_feat, bound=1.0 / math.sqrt(dim_feat))
    sd[f"model.module_{i}.bias"] = u(dim_dense, bound=1.0 / math.sqrt(dim_feat))
    sd[f"model.module_{i + 1}.weight"] = u(dim_out, dim_dense, bound=1.0 / math.sqrt(dim_dense))
    sd[f"model.module_{i + 1}.bias"] = u(dim_out, bound=1.0 / math.sqrt(dim_dense))
    return sd


# --------------------------------------------------------------------------------------------
# gnn_dsse (networks.py:11-69): (num_layers - 1) x [conv + nonlin], Linear(dim_feat, dim_dense), Linear(dim_dense, dim_out);
# forward(x, edge_index) with x_0 = x, on the edge list AS GIVEN (no un-directing).  model='gcn2': GCN2Conv(channels, alpha,
# shared_weights=True, add_self_loops, normalize); model='fagcn': FAConv(channels, eps, dropout, add_self_loops, normalize);
# model='tagcn': TAGConv(channels, channels, K, bias, normalize).
# --------------------------------------------------------------------------------------------


def gcn_norm_self_loops(edge_index, num_nodes, dtype):
    """PyG gcn_norm(add_self_loops=True), which calls add_remaining_self_loops: the self loops of the input are dropped, the other
    edges keep their order and one loop of weight 1 per node is appended; deg = in-degree (input loops not counted) + 1 by target;
    w = deg[src]^-1/2 * deg[dst]^-1/2."""
    loop = torch.arange(num_nodes)
    ei = torch.cat([edge_index[:, edge_index[0] != edge_index[1]], torch.stack([loop, loop])], dim=1)
    return ei, gcn_weights(ei, num_nodes, dtype)


def gnn_dsse_forward(sd, x, edge_index, num_layers, model="gcn2", alpha=0.1, K=3, add_self_loops=True, slope=0.01, nonlin="leaky_relu"):
    """gnn_dsse.forward (networks.py:67-69) from a reference-named state_dict (`model.module_{2l}.weight1` / `.lins.{k}.weight`, `.bias`).
    nonlin: the module's activation after every conv, 'leaky_relu' (negative slope `slope`), 'relu' or 'tanh'."""
    act = {"leaky_relu": lambda t: torch.nn.functional.leaky_relu(t, slope), "relu": torch.relu, "tanh": torch.tanh}[nonlin]
    n = x.size(0)
    x0, h = x, x
    for l in range(num_layers - 1):
        p = f"model.module_{2 * l}."
        if model == "gcn2":
            if add_self_loops:
                ei, w = gcn_norm_self_loops(edge_index, n, x.dtype)
            else:
                ei, w = edge_index, gcn_weights(edge_index, n, x.dtype)
            prop = segment_sum(w.view(-1, 1) * h[ei[0]], ei[1], n)          # GCN2Conv.message / aggr='add'
            out = prop * (1 - alpha) + alpha * x0                           # x.mul_(1 - alpha); x_0 = alpha * x_0; x.add_(x_0)
            h = out @ sd[p + "weight1"]                                     # addmm(out, out, weight1, beta=0, alpha=1)
        elif model == "fagcn":
            # FAConv (PyG): out_i = sum_{j -> i} tanh(att_l x_j + att_r x_i) w_ji x_j + eps x_0_i; `alpha` is FAConv's eps (networks.py:46)
            if add_self_loops:
                ei, w = gcn_norm_self_loops(edge_index, n, x.dtype)
            else:
                ei, w = edge_index, gcn_weights(edge_index, n, x.dtype)
            al, ar = h @ sd[p + "att_l.weight"].t(), h @ sd[p + "att_r.weight"].t()
            coef = torch.tanh(al[ei[0]] + ar[ei[1]]).squeeze(-1) * w
            h = segment_sum(coef.view(-1, 1) * h[ei[0]], ei[1], n)
            if alpha != 0.0:
                h = h + alpha * x0
        elif model == "tagcn":
            ws = []
            k = 0
            while f"{p}lins.{k}.weight" in sd:
                ws.append(sd[f"{p}lins.{k}.weight"])
                k += 1
            h = tag_conv(h, edge_index, ws, sd.get(p + "bias"))
        else:
            raise NotImplementedError(model)
        h = act(h)
    i = 2 * (num_layers - 1)
    h = h @ sd[f"model.module_{i}.weight"].t() + sd[f"model.module_{i}.bias"]
    return h @ sd[f"model.module_{i + 1}.weight"].t() + sd[f"model.module_{i + 1}.bias"]


def init_gnn_state_dict(model="gcn2", dim_feat=8, dim_dense=32, dim_out=2, num_layers=4, K=3, seed=0, dtype=torch.float32):
    """Random parameters under the reference's names (PyG Sequential children `module_{i}`); biases non-zero so that they matter."""
    g = torch.Generator().manual_seed(seed)

    def u(*shape, bound):
        return ((torch.rand(*shape, generator=g) * 2 - 1) * bound).to(dtype)

    sd = {}
    c = dim_feat
    for l in range(num_layers - 1):
        p = f"model.module_{2 * l}."
        if model == "gcn2":
            sd[p + "weight1"] = u(c, c, bound=math.sqrt(6.0 / (2 * c)))
        elif model == "fagcn":
            sd[p + "att_l.weight"] = u(1, c, bound=1.0 / math.sqrt(c))
            sd[p + "att_r.weight"] = u(1, c, bound=1.0 / math.sqrt(c))
        else:
            sd[p + "bias"] = u(c, bound=0.1)
            for k in range(K + 1):
                sd[p + f"lins.{k}.weight"] = u(c, c, bound=1.0 / math.sqrt(c))
    i = 2 * (num_layers - 1)
    sd[f"model.module_{i}.weight"] = u(dim_dense, c, bound=1.0 / math.sqrt(c))
    sd[f"model.module_{i}.bias"] = u(dim_dense, bound=1.0 / math.sqrt(c))
    sd[f"model.module_{i + 1}.weight"] = u(dim_out, dim_dense, bound=1.0 / math.sqrt(dim_dense))
    sd[f"model.module_{i + 1}.bias"] = u(dim_out, bound=1.0 / math.sqrt(dim_dense))
    return sd


# --------------------------------------------------------------------------------------------
# physics: branch flows (data.py:328-390) and the WLS loss (data.py:393-459)
# --------------------------------------------------------------------------------------------


def get_pflow(y, edge_index, node_param, edge_param, phase_shift=True):
    """data.py:328-390.  phase_shift=True is the only way the script calls it (angle shift ignored, :362-363);
    phase_shift=False subtracts the branch's phase-shift column from the angle difference (:364-365).

    y[Nt,2] = (V pu, theta rad); edge_index one-way [2,Et]; node_param[:,0] = vn_kv;
    edge_param = (G, B, Gs, Bs, closed, phase_shift, imax_or_sn).
    Returns (loading_lines, loading_trafo, P_from, Q_from, P_to, Q_to, I_from, I_to)."""
    vn = node_param[:, 0]
    v_hv, v_lv = vn.max(), vn.min()                     # :334-336, over the whole batch
    ratio = (v_hv / v_lv).detach()                      # :338
    frm, to = edge_index[0], edge_index[1]
    vi, vj = y[:, 0][frm], y[:, 0][to]                  # :355-358
    delta = y[:, 1][frm] - y[:, 1][to]                  # shift = 0
    if not phase_shift:
        delta = delta - edge_param[:, 5].detach()       # :365 torch.tensor(edge_param[:,5]) is a detached copy
    g, b, gs, bs = edge_param[:, 0], edge_param[:, 1], edge_param[:, 2], edge_param[:, 3]
    is_trafo = torch.ceil(edge_param[:, 5].detach())    # :367 (3 on Oberrhein: quirk kept)
    rating = edge_param[:, 6].detach()                  # :368
    cosd, sind = torch.cos(delta), torch.sin(delta)
    base = v_lv ** 2
    p_from = (-vi * vj * (g * cosd + b * sind) + (g + gs / 2) * vi ** 2) * base     # :370
    q_from = (vi * vj * (-g * sind + b * cosd) - (b + bs / 2) * vi ** 2) * base     # :372
    p_to = (-vi * vj * (g * cosd - b * sind) + (g + gs / 2) * vj ** 2) * base       # :374
    q_to = (vi * vj * (g * sind + b * cosd) - (b + bs / 2) * vj ** 2) * base        # :376
    sqrt3 = torch.sqrt(torch.tensor(3.0, dtype=torch.float32)).to(y.dtype)          # :378 fp32 sqrt(3)
    i_from = torch.complex(p_from, -q_from).abs() / (vi * v_lv * sqrt3)             # :378
    i_from = i_from / (1.0 - (is_trafo * (1.0 - ratio)))                            # :380
    i_to = torch.complex(p_to, -q_to).abs() / (vj * v_lv * sqrt3)                   # :383
    load_lines = ((1.0 - is_trafo) * torch.maximum(i_from, i_to)) / rating          # :387
    load_trafo = (is_trafo * torch.maximum(i_from * v_hv, i_to * v_lv)) / rating    # :388
    return load_lines, load_trafo, p_from, q_from, p_to, q_to, i_from, i_to


def wls_loss(x, edge_attr, output, x_mean, x_std, edge_mean, edge_std, edge_index, reg_coefs):
    """data.py:393-459 `gsp_wls_edge`, taking the full 11-/13-column tensors (the caller slices them
    into input / node_param / edge_input / edge_param, dss2_run.py:140).  The dead dense Laplacian
    (:422-423) is omitted - it does not influence the result.  `output` is NOT modified in place here
    (the reference zeroes slack theta inside the caller's tensor, :412-413; the effect on the loss is
    identical).  Returns the 0-dim loss."""
    feat, node_param = x[:, :8], x[:, 8:]
    efeat, edge_param = edge_attr[:, :6], edge_attr[:, 6:]
    nt = x.shape[0]
    z, r = feat[:, 0::2], feat[:, 1::2]                               # :397, :403
    ez, er = efeat[:, 0:4:2], efeat[:, 1:4:2]                         # :398, :405
    meas = (z * x_std[0::2] + x_mean[0::2]) * (z != 0)                # :402
    wgt = (r * x_std[1::2] + x_mean[1::2]) * (r != 0)                 # :408
    emeas = (ez * edge_std[0:4:2] + edge_mean[0:4:2]) * (ez != 0)     # :401
    ewgt = (er * edge_std[1:4:2] + edge_mean[1:4:2]) * (er != 0)      # :409
    v = output[:, 0:1] * x_std[:1] + x_mean[:1]                       # :411
    theta = output[:, 1:] * (1.0 - node_param[:, 1:2])                # :412-413
    state = torch.cat([v, theta], dim=1)
    ll, lt, pf, qf, pt, qt, _, _ = get_pflow(state, edge_index, node_param, edge_param)
    loading = ll + lt                                                 # :417
    frm, to = edge_index[0], edge_index[1]
    p_bus = -segment_sum(pt, to, nt) - segment_sum(pf, frm, nt)       # :428
    q_bus = -segment_sum(qt, to, nt) - segment_sum(qf, frm, nt)       # :429
    dtheta = (theta[:, 0][frm] - theta[:, 0][to]).abs()               # :431
    h = torch.cat([v, theta, p_bus[:, None], q_bus[:, None]], dim=1)  # :433
    h_edge = torch.stack([pf, qf], dim=1)                             # :435
    lam_n = torch.tensor([reg_coefs["lam_v"], reg_coefs["lam_v"], reg_coefs["lam_p"], reg_coefs["lam_p"]], dtype=x.dtype)
    lam_e = torch.tensor([reg_coefs["lam_pf"], reg_coefs["lam_pf"]], dtype=x.dtype)
    j_node = (((meas - h) ** 2 * wgt) * lam_n).sum(1)                 # :446
    j_edge = (((emeas - h_edge) ** 2 * ewgt) * lam_e).sum(1)          # :447
    j = j_node.mean() + j_edge.mean()                                 # :450
    lam = reg_coefs["lam_reg"]
    j_v = lam * (torch.relu(v - 1.1) + torch.relu(0.9 - v)).mean() ** 2       # :453
    j_t = lam * torch.relu(dtheta - 0.5).mean() ** 2                          # :454
    j_l = lam * torch.relu(loading - 1.5).mean() ** 2                         # :455
    return j + j_v + j_t + j_l


# --------------------------------------------------------------------------------------------
# optimizer (adjacent row a10: torch.optim.Adamax defaults, dss2_run.py:91-92)
# --------------------------------------------------------------------------------------------


def adamax_step(param, grad, exp_avg, exp_inf, step, lr=3e-3, beta1=0.9, beta2=0.999, eps=1e-8):
    """torch.optim.Adamax single-tensor update (no weight decay); `step` is the 1-based step count.
    exp_avg = b1*exp_avg + (1-b1)*g ; exp_inf = max(b2*exp_inf, |g| + eps) ;
    param -= lr / (1 - b1^step) * exp_avg / exp_inf.  Updates in place, returns param."""
    exp_avg.mul_(beta1).add_(grad, alpha=1 - beta1)
    torch.maximum(exp_inf * beta2, grad.abs() + eps, out=exp_inf)
    clr = lr / (1 - beta1 ** step)
    param.addcdiv_(exp_avg, exp_inf, value=-clr)
    return param


# --------------------------------------------------------------------------------------------
# one training step on CPU (used as the timed CPU baseline "port")
# --------------------------------------------------------------------------------------------


def train_step(sd, batch, stats, reg_coefs, p_drop, opt_state, kind="SkipPFN", generator=None):
    """fwd + loss + bwd (autograd) + Adamax on CPU, mirroring dss2_run.py:137-143.  `sd` values must be
    leaf tensors with requires_grad=True; opt_state = {"step": int, name: (exp_avg, exp_inf)}."""
    for p in sd.values():
        p.grad = None
    out = pfn_forward(sd, batch["x"][:, :8], batch["edge_index"], batch["edge_attr"][:, :6], p_drop,
                      skip=(kind == "SkipPFN"), generator=generator)
    loss = wls_loss(batch["x"], batch["edge_attr"], out, stats["x_mean"], stats["x_std"],
                    stats["edge_mean"], stats["edge_std"], batch["edge_index"], reg_coefs)
    loss.backward()
    opt_state["step"] = opt_state.get("step", 0) + 1
    with torch.no_grad():
        for name, p in sd.items():
            if name not in opt_state:
                opt_state[name] = (torch.zeros_like(p), torch.zeros_like(p))
            adamax_step(p, p.grad, opt_state[name][0], opt_state[name][1], opt_state["step"])
    return loss.detach()


# --------------------------------------------------------------------------------------------
# (f-3) synthetic scenario sampler of the offline generator: loadsampling.py:75-107, toy_network.py:83-129
# --------------------------------------------------------------------------------------------
def mc_uniform(lb, ub, numbersamples, draws=None):
    """loadsampling.py:75-93 `samplermontecarlo`: LB + rand(U, n) * (UB - LB); scalars broadcast to [1, n] like the reference."""
    import numpy as np
    lb, ub = np.atleast_1d(np.asarray(lb, dtype=np.float64)), np.atleast_1d(np.asarray(ub, dtype=np.float64))
    if draws is None:
        draws = np.random.rand(lb.size, numbersamples)           # :91, legacy global stream
    return lb[:, None] + np.multiply(draws, (ub - lb)[:, None])


def mc_normal(mu, sig, numbersamples, draws=None):
    """loadsampling.py:94-107 `samplermontecarlo_normal`: np.random.normal(MMU, MSIG) = MMU + MSIG * gauss on the legacy stream."""
    import numpy as np
    mu, sig = np.atleast_1d(np.asarray(mu, dtype=np.float64)), np.atleast_1d(np.asarray(sig, dtype=np.float64))
    if draws is None:
        draws = np.random.standard_normal((mu.size, numbersamples))
    return mu[:, None] + sig[:, None] * draws


def sample_profiles(base, weight_a, weight_b, profile_a, profile_b, iterations, dist="normal", spread=0.15, draws=None):
    """toy_network.py:104-129: hourly profile of every load (:106-107), unrolled (:111-114), perturbed `iterations` times with the chosen
    sampler (:118-123) and reshaped to [L, H*iterations] (:129)."""
    import numpy as np
    base, wa, wb = (np.asarray(t, dtype=np.float64) for t in (base, weight_a, weight_b))
    pa, pb = np.asarray(profile_a, dtype=np.float64), np.asarray(profile_b, dtype=np.float64)
    prof = np.stack([wa * (base * pa[i]) + wb * (base * pb[i]) for i in range(pa.size)], axis=1)
    unroll = np.reshape(prof, prof.size)
    if dist == "uniform":
        mc = mc_uniform(unroll * (1 - spread), unroll * (1 + spread), iterations, draws)
    else:
        mc = mc_normal(unroll, unroll * spread, iterations, draws)
    return np.reshape(mc, [prof.shape[0], prof.shape[1] * iterations])
