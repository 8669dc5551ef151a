"""Attention dropout of GAT_DSSE (GATv2Conv, networks.py:145-146) and gnn_dsse(model='fagcn') (FAConv, networks.py:46).

PyG applies F.dropout to the normalised attention coefficients in training mode: every coefficient of a softmax segment, the
appended self loop included, is kept with probability 1 - p and scaled by 1 / (1 - p).  The kernels draw the keep bit of a
coefficient from its edge key (one-way edge id e, Et + i for the loop of bus i), so a mask is a uint8 [Et + Nt] per (layer, head).

The masked reference below (fp64 arbiter, fp32 noise) restates the oracle's GAT_DSSE / fagcn forward with injected masks in that
edge-key layout; the CPU tests pin it, and the layout conversion, to the PyG shim's GATv2Conv / FAConv with F.dropout replaced by the
same mask."""
import os
import sys

import pytest
import torch

from conftest import REG_COEFS, ROOT, assert_fp32_parity, permute_edges
import dss2_oracle as orc
import networks

SHIM = os.path.join(ROOT, "oracle", "pyg_shim")
P = 0.3


# ------------------------------------------------------------------------------------------------ masked reference
def edge_keys(edge_index, n, self_loops):
    """Edge key of every attention coefficient in PyG's edge order: with self loops, the input loops removed (GATv2Conv's
    remove_self_loops, FAConv's add_remaining_self_loops) and one loop per bus appended; without, the edge list as given."""
    et = edge_index.size(1)
    ids = torch.arange(et)
    if not self_loops:
        return ids
    ids = ids[edge_index[0] != edge_index[1]]
    return torch.cat([ids, et + torch.arange(n)])


def to_pyg_order(mask, edge_index, n, self_loops):
    """[..., Et + N] edge-key layout -> [..., E'] PyG order."""
    return mask[..., edge_keys(edge_index, n, self_loops)]


def from_pyg_order(mask, edge_index, n, self_loops):
    """[..., E'] PyG order -> [..., Et + N] edge-key layout (keys PyG never visits: 0)."""
    out = torch.zeros(mask.shape[:-1] + (edge_index.size(1) + n,), dtype=mask.dtype)
    out[..., edge_keys(edge_index, n, self_loops)] = mask
    return out


def gatv2_layer(x, edge_index, edge_attr, w_l, b_l, w_r, b_r, w_e, att, bias, slope=0.2, self_loops=True, mask=None, p=0.0, trace=None):
    """orc.gatv2_layer with alpha = alpha * mask[key] / (1 - p) after the softmax (mask: [Et + N] edge-key layout).  trace (test hook):
    collects x_l and x_r, whose per-bus gradients are the terms of the lin_l / lin_r bias gradients."""
    n = x.size(0)
    if self_loops:
        keep = edge_index[0] != edge_index[1]
        src, dst, ea = edge_index[0][keep], edge_index[1][keep], edge_attr[keep]
        cnt = orc.segment_sum(torch.ones(dst.numel(), 1, dtype=x.dtype), dst, n).clamp(min=1)
        loop_attr = orc.segment_sum(ea, dst, n) / cnt
        loop = torch.arange(n)
        src, dst, ea = torch.cat([src, loop]), torch.cat([dst, loop]), torch.cat([ea, loop_attr])
    else:
        src, dst, ea = edge_index[0], edge_index[1], edge_attr
    x_l = x @ w_l.t() + b_l
    x_r = x @ w_r.t() + b_r
    if trace is not None:
        trace += [x_l, x_r]
    s = torch.nn.functional.leaky_relu(x_r[dst] + x_l[src] + ea @ w_e.t(), slope)
    score = (s * att.view(1, -1)).sum(-1)
    smax = torch.full((n,), float("-inf"), dtype=x.dtype).scatter_reduce(0, dst, score.detach(), reduce="amax", include_self=True)
    ex = (score - smax[dst]).exp()
    den = orc.segment_sum(ex.view(-1, 1), dst, n).view(-1) + 1e-16
    alpha = ex / den[dst]
    if mask is not None:
        alpha = alpha * (to_pyg_order(mask, edge_index, n, self_loops).to(x.dtype) / (1.0 - p))
    return orc.segment_sum(x_l[src] * alpha.view(-1, 1), dst, n) + bias


def gat_forward(sd, x, edge_index, edge_attr, num_layers, nonlin="leaky_relu", slope=0.2, self_loops=True, masks=None, p=0.0, trace=None):
    """orc.gat_dsse_forward with per-layer masks [heads, Et + N].  trace (test hook): name -> the tensors whose per-bus gradients,
    concatenated over the columns, are the terms that the gradient of the bias `name` sums over the buses."""
    h = x
    for l in range(num_layers - 1):
        pf = f"model.module_{2 * l}."
        H, c = sd[pf + "att"].shape[1], h.size(1)
        tr = [] if trace is not None else None
        heads = [gatv2_layer(h, edge_index, edge_attr, *[sd[pf + k][j * c:(j + 1) * c] for k in ("lin_l.weight", "lin_l.bias", "lin_r.weight",
                                                                                                "lin_r.bias", "lin_edge.weight")],
                             sd[pf + "att"][0, j], 0.0, slope=slope, self_loops=self_loops, mask=None if masks is None else masks[l][j], p=p,
                             trace=tr)
                 for j in range(H)]
        h = torch.stack(heads, 1).mean(dim=1) + sd[pf + "bias"]
        if trace is not None:
            trace[pf + "lin_l.bias"], trace[pf + "lin_r.bias"], trace[pf + "bias"] = tr[0::2], tr[1::2], [h]
        h = {"leaky_relu": lambda t: torch.nn.functional.leaky_relu(t, 0.01), "relu": torch.relu, "tanh": torch.tanh}[nonlin](h)
    i = 2 * (num_layers - 1)
    h = h @ sd[f"model.module_{i}.weight"].t() + sd[f"model.module_{i}.bias"]
    return h @ sd[f"model.module_{i + 1}.weight"].t() + sd[f"model.module_{i + 1}.bias"]


def fa_layer(h, x0, edge_index, att_l, att_r, eps, self_loops=True, mask=None, p=0.0):
    """One FAConv as the fagcn oracle states it, coef = dropout(tanh(att_l x_j + att_r x_i)) w_ji (mask: [Et + N] edge-key layout)."""
    n = h.size(0)
    if self_loops:
        ei, w = orc.gcn_norm_self_loops(edge_index, n, h.dtype)
    else:
        ei, w = edge_index, orc.gcn_weights(edge_index, n, h.dtype)
    t = torch.tanh((h @ att_l.t())[ei[0]] + (h @ att_r.t())[ei[1]]).squeeze(-1)
    if mask is not None:
        t = t * (to_pyg_order(mask, edge_index, n, self_loops).to(h.dtype) / (1.0 - p))
    out = orc.segment_sum((t * w).view(-1, 1) * h[ei[0]], ei[1], n)
    return out + eps * x0 if eps != 0.0 else out


def fagcn_forward(sd, x, edge_index, num_layers, alpha=0.1, self_loops=True, slope=0.01, masks=None, p=0.0):
    """orc.gnn_dsse_forward(model='fagcn') with per-layer masks [1, Et + N]."""
    h = x
    for l in range(num_layers - 1):
        pf = f"model.module_{2 * l}."
        h = fa_layer(h, x, edge_index, sd[pf + "att_l.weight"], sd[pf + "att_r.weight"], alpha, self_loops,
                     None if masks is None else masks[l][0], p)
        h = torch.nn.functional.leaky_relu(h, slope)
    i = 2 * (num_layers - 1)
    h = h @ sd[f"model.module_{i}.weight"].t() + sd[f"model.module_{i}.bias"]
    return h @ sd[f"model.module_{i + 1}.weight"].t() + sd[f"model.module_{i + 1}.bias"]


def random_masks(num_layers, heads, num_keys, p, seed):
    g = torch.Generator().manual_seed(seed)
    return [(torch.rand(heads, num_keys, generator=g) >= p).to(torch.uint8) for _ in range(num_layers - 1)]


# ------------------------------------------------------------------------------------------------ CPU: the reference against PyG's semantics
def _shim_conv():
    if SHIM not in sys.path:
        sys.path.insert(0, SHIM)
    from torch_geometric.nn import conv
    return conv


# a graph with two input self loops ((2,2), (4,4)), a bus without in-edges (0) and a bus with several (1)
_EI = torch.tensor([[0, 1, 2, 2, 3, 5, 6, 6, 4], [1, 2, 3, 2, 1, 1, 7, 8, 4]])
_EI_NO_LOOPS = torch.tensor([[0, 1, 2, 3, 5, 6, 6, 4], [1, 2, 3, 1, 1, 7, 8, 2]])


def _patched_dropout(monkeypatch, mask_pyg):
    """F.dropout replaced by the recorded mask (what PyG's layer would have drawn), training mode required."""
    def dropout(t, p=0.5, training=True, inplace=False):
        assert training and t.shape == mask_pyg.shape
        return t * (mask_pyg.to(t.dtype) / (1.0 - p))
    monkeypatch.setattr(torch.nn.functional, "dropout", dropout)


@pytest.mark.parametrize("heads", [1, 3])
@pytest.mark.parametrize("self_loops", [True, False])
def test_masked_gatv2_reference_matches_pyg_semantics(monkeypatch, heads, self_loops):
    conv = _shim_conv()
    n = 9
    torch.manual_seed(11)
    x = torch.randn(n, 8, dtype=torch.float64)
    ea = torch.randn(_EI.size(1), 6, dtype=torch.float64)
    sd = orc.init_gat_state_dict(num_layers=2, seed=4, heads=heads, dtype=torch.float64)
    layer = conv.GATv2Conv(8, 8, heads=heads, concat=False, dropout=P, add_self_loops=self_loops, edge_dim=6).double().train()
    with torch.no_grad():
        for k in ("att", "bias", "lin_l.weight", "lin_l.bias", "lin_r.weight", "lin_r.bias", "lin_edge.weight"):
            layer.get_parameter(k).copy_(sd["model.module_0." + k])
    mask = random_masks(2, heads, _EI.size(1) + n, P, seed=heads)[0]
    mask_pyg = to_pyg_order(mask, _EI, n, self_loops)
    assert torch.equal(to_pyg_order(from_pyg_order(mask_pyg, _EI, n, self_loops), _EI, n, self_loops), mask_pyg)
    _patched_dropout(monkeypatch, mask_pyg.t())          # the shim's alpha is [E', heads]
    want = layer(x, _EI, ea)
    c = 8
    got = torch.stack([gatv2_layer(x, _EI, ea, *[sd["model.module_0." + k][j * c:(j + 1) * c] for k in ("lin_l.weight", "lin_l.bias", "lin_r.weight",
                                                                                                         "lin_r.bias", "lin_edge.weight")],
                                   sd["model.module_0.att"][0, j], 0.0, self_loops=self_loops, mask=mask[j], p=P) for j in range(heads)], 1)
    got = got.mean(1) + sd["model.module_0.bias"]
    assert torch.allclose(got, want, rtol=1e-12, atol=1e-12)
    monkeypatch.undo()
    assert not torch.allclose(layer.eval()(x, _EI, ea), want), "the mask matters"


@pytest.mark.parametrize("self_loops", [True, False])
def test_masked_faconv_reference_matches_pyg_semantics(monkeypatch, self_loops):
    """On the loop-free graph and on _EI, whose input loops FAConv's add_remaining_self_loops drops under add_self_loops (their mask
    entries are then never read) and keeps as ordinary edges without it."""
    conv = _shim_conv()
    n = 9
    torch.manual_seed(12)
    x, x0 = torch.randn(n, 8, dtype=torch.float64), torch.randn(n, 8, dtype=torch.float64)
    layer = conv.FAConv(8, eps=0.1, dropout=P, add_self_loops=self_loops).double().train()
    for ei in (_EI_NO_LOOPS, _EI):
        mask = random_masks(2, 1, ei.size(1) + n, P, seed=5)[0][0]
        mask_pyg = to_pyg_order(mask, ei, n, self_loops)
        _patched_dropout(monkeypatch, mask_pyg)
        want = layer(x, x0, ei)
        monkeypatch.undo()
        got = fa_layer(x, x0, ei, layer.att_l.weight.detach(), layer.att_r.weight.detach(), 0.1, self_loops, mask, P)
        assert torch.allclose(got, want, rtol=1e-12, atol=1e-12)


def test_constructors_accept_attention_dropout(monkeypatch):
    monkeypatch.setattr(torch.cuda, "is_available", lambda: True)      # the constructors refuse p > 0 without a device (test below)
    for p in (0.1, 0.5, 0.99):
        for kw in ({}, {"heads": 3, "concat": False}):
            m = networks.GAT_DSSE(dim_feat=8, dim_dense=32, dim_out=2, num_layers=4, edge_dim=6, dropout=p, **kw)
            ref = networks.GAT_DSSE(dim_feat=8, dim_dense=32, dim_out=2, num_layers=4, edge_dim=6, **kw)
            assert [(k, v.shape) for k, v in m.state_dict().items()] == [(k, v.shape) for k, v in ref.state_dict().items()]
        m = networks.gnn_dsse(dim_feat=8, dim_dense=32, dim_out=2, num_layers=4, model="fagcn", dropout=p)
        ref = networks.gnn_dsse(dim_feat=8, dim_dense=32, dim_out=2, num_layers=4, model="fagcn")
        assert [(k, v.shape) for k, v in m.state_dict().items()] == [(k, v.shape) for k, v in ref.state_dict().items()]
    for p, exc in ((1.0, NotImplementedError), (-0.1, ValueError), (1.5, ValueError)):
        with pytest.raises(exc):
            networks.GAT_DSSE(dim_feat=8, dim_dense=32, dim_out=2, num_layers=4, edge_dim=6, dropout=p)
        with pytest.raises(exc):
            networks.gnn_dsse(dim_feat=8, dim_dense=32, dim_out=2, num_layers=4, model="fagcn", dropout=p)
    networks.gnn_dsse(dim_feat=8, dim_dense=32, dim_out=2, num_layers=4, model="gcn2", dropout=0.5)   # ignored, as in the reference
    with pytest.raises(NotImplementedError):      # the other refusals stay
        networks.GAT_DSSE(dim_feat=8, dim_dense=32, dim_out=2, num_layers=4, edge_dim=6, heads=2, concat=True, dropout=0.1)


def test_attention_dropout_needs_a_cuda_device(monkeypatch):
    """Attention dropout exists only in the CUDA kernels: without a device the constructors refuse p > 0 (p = 0 still builds)."""
    monkeypatch.setattr(torch.cuda, "is_available", lambda: False)
    for build in (lambda p: networks.GAT_DSSE(dim_feat=8, dim_dense=32, dim_out=2, num_layers=3, edge_dim=6, dropout=p),
                  lambda p: networks.gnn_dsse(dim_feat=8, dim_dense=32, dim_out=2, num_layers=3, model="fagcn", dropout=p)):
        build(0.0)
        with pytest.raises(NotImplementedError):
            build(0.1)


# ------------------------------------------------------------------------------------------------ GPU
NL = 5
CASES = {   # name -> (model kind, constructor options, environment)
    "gat": ("gat", {}, {}),
    "gat_noslots": ("gat", {}, {"DSS2_GAT_SLOTS": "0"}),
    "gat_heads2": ("gat", {"heads": 2, "concat": False}, {}),
    "gat_heads3": ("gat", {"heads": 3, "concat": False}, {}),
    "gat_noloop_tanh": ("gat", {"self_loops": False, "nonlin": "tanh"}, {}),
    "fagcn": ("fagcn", {}, {}),
}


def _batch(case, nb, seed):
    from dss2 import batching, synth
    st = synth.synthetic_store(synth.load_grid(case), nb, seed=seed).to("cuda")
    return batching.pack_batch(st, list(range(nb))), [t.cpu() for t in (st.x_mean, st.x_std, st.edge_mean, st.edge_std)]


def _model(name, p, seed):
    kind, opts, _ = CASES[name]
    if kind == "gat":
        sd = orc.init_gat_state_dict(num_layers=NL, seed=seed, heads=opts.get("heads", 1))
        m = networks.GAT_DSSE(dim_feat=8, dim_dense=32, dim_out=2, num_layers=NL, edge_dim=6, dropout=p, **opts)
    else:
        sd = orc.init_gnn_state_dict("fagcn", num_layers=NL, seed=seed)
        m = networks.gnn_dsse(dim_feat=8, dim_dense=32, dim_out=2, num_layers=NL, model="fagcn", dropout=p, **opts)
    m.load_state_dict(sd, strict=True)
    return m.cuda().train(), sd


def _call(name, model, x, ei, ea):
    return model(x, ei, ea) if CASES[name][0] == "gat" else model(x, ei)


def _oracle(name, sd, x, ei, ea, masks, dtype, trace=None):
    kind, opts, _ = CASES[name]
    p = {k: v.to(dtype) for k, v in sd.items()}
    if kind == "gat":
        return gat_forward(p, x, ei, ea, NL, nonlin=opts.get("nonlin", "leaky_relu"), self_loops=opts.get("self_loops", True), masks=masks, p=P,
                           trace=trace)
    return fagcn_forward(p, x, ei, NL, masks=masks, p=P)


def _oracle_run(name, sd, x, ea, ei, stats, masks, dtype, grad_out=None):
    """fp32 / fp64 reference: output, loss (WLS or sum(out * grad_out)), parameter gradients, gradient w.r.t. the 8 input features,
    and name -> per-bus terms [N, .] of every bias gradient that is a plain sum over the buses."""
    p = {k: v.to(dtype).clone().requires_grad_(True) for k, v in sd.items()}
    xin = x[:, :8].to(dtype).clone().requires_grad_(True)
    trace = {}
    out = _oracle(name, p, xin, ei, ea[:, :6].to(dtype), masks, dtype, trace)
    for ts in trace.values():
        for t_ in ts:
            t_.retain_grad()
    if grad_out is None:
        loss = orc.wls_loss(x.to(dtype), ea.to(dtype), out, *[s.to(dtype) for s in stats], ei, REG_COEFS)
    else:
        loss = (out * grad_out.to(dtype)).sum()
    loss.backward()
    terms = {k: torch.cat([t_.grad for t_ in ts], 1) for k, ts in trace.items()}
    return out.detach(), loss.detach(), {k: v.grad for k, v in p.items()}, xin.grad, terms


def _permuted(x, ea, ei, masks, seed):
    """The same batch with the edge list in another order, and the masks moved with their edges (another valid fp32 evaluation)."""
    et = ei.size(1)
    perm = torch.randperm(et, generator=torch.Generator().manual_seed(seed))
    pb = permute_edges({"edge_index": ei, "edge_attr": ea}, seed)
    assert torch.equal(pb["edge_index"], ei[:, perm])
    pm = [torch.cat([m[:, :et][:, perm], m[:, et:]], 1) for m in masks]
    return pb["edge_attr"], pb["edge_index"], pm


def _check_step(name, model, b, stats, masks):
    """One training step of the drop-in module (masks: injected, or None for its Philox stream): output, loss through gsp_wls_edge,
    parameter gradients, gradient w.r.t. the 8 input features, and the upstream gradient d loss / d out the loss kernel produced."""
    import data
    x, ea, ei = b.x, b.edge_attr, b.edge_index
    xin = x[:, :8].clone().requires_grad_(True)
    if masks is not None:
        model._dss2_attn_masks = masks
    out = _call(name, model, xin, ei, ea[:, :6])
    up = []
    out.register_hook(up.append)
    out_before = out.detach().clone()
    # (gsp_wls_edge zeroes the slack angle inside the tensor it gets, as the reference does: it gets a copy, so that the hook above sees
    # d loss / d out)
    loss = data.gsp_wls_edge(input=x[:, :8], edge_input=ea[:, :6], output=out.clone(), x_mean=stats[0], x_std=stats[1], edge_mean=stats[2],
                             edge_std=stats[3], edge_index=ei, reg_coefs=REG_COEFS, num_samples=None, node_param=x[:, 8:], edge_param=ea[:, 6:])
    loss.backward()
    return out_before, loss.detach(), {k: v.grad.clone() for k, v in model.named_parameters()}, xin.grad.clone(), up[0].clone()


def _compare(name, model, b, stats, sd, masks, ours):
    """`ours` (from _check_step) against the masked reference with `masks`: output, loss, every parameter gradient and the gradient
    w.r.t. x end to end, then the backward kernels on a fixed upstream gradient - at the criteria of
    test_gpu_parity.test_gat_dsse_matches_reference_run."""
    out_before, loss, grads, gx, gout = ours
    xc, eac, eic = b.x.cpu(), b.edge_attr.cpu(), b.edge_index.cpu()
    r64 = _oracle_run(name, sd, xc, eac, eic, stats, masks, torch.float64)
    runs = [_oracle_run(name, sd, xc, eac, eic, stats, masks, torch.float32)]
    for s_ in (1, 2):
        pea, pei, pm = _permuted(xc, eac, eic, masks, s_)
        runs.append(_oracle_run(name, sd, xc, pea, pei, stats, pm, torch.float32))
    assert_fp32_parity(out_before, [r[0] for r in runs], r64[0], "out")
    l_ref = {dt: orc.wls_loss(xc.to(dt), eac.to(dt), out_before.cpu().to(dt), *[t_.to(dt) for t_ in stats], eic, REG_COEFS)
             for dt in (torch.float32, torch.float64)}
    assert_fp32_parity(loss, l_ref[torch.float32], l_ref[torch.float64], "loss (of our output)")
    assert_fp32_parity(loss, [r[1] for r in runs], r64[1], "loss vs the masked reference", rtol=1e-4, noise_mult=16.0)
    # gradients end to end.  d loss / d out carries the loss's conditioning (a 1e-7 change of `out` moves the loss by 1e-5), so the
    # chain is judged in its two pieces: the upstream gradient our loss kernel produced, against the reference's at the output it
    # received, and the model's gradients, against the reference's backward fed with that same upstream gradient (end-to-end criterion
    # of the reference-run tests)
    g_up = {}
    for dt in (torch.float32, torch.float64):
        o_ = out_before.cpu().to(dt).requires_grad_(True)
        l_ = orc.wls_loss(xc.to(dt), eac.to(dt), o_, *[t_.to(dt) for t_ in stats], eic, REG_COEFS)
        g_up[dt] = torch.autograd.grad(l_, o_)[0]
    assert_fp32_parity(gout, g_up[torch.float32], g_up[torch.float64], "d loss / d out (of our output)", rtol=1e-4, noise_mult=16.0)
    chain = {dt: _oracle_run(name, sd, xc, eac, eic, stats, masks, dt, grad_out=gout.cpu()) for dt in (torch.float32, torch.float64)}
    for k in sd:
        assert_fp32_parity(grads[k], chain[torch.float32][2][k], chain[torch.float64][2][k], k + " (end to end)", rtol=1e-4, noise_mult=16.0,
                           sum_of=chain[torch.float64][4].get(k))
    assert_fp32_parity(gx, chain[torch.float32][3], chain[torch.float64][3], "grad_x (end to end)", rtol=1e-4, noise_mult=16.0)
    # the backward kernels alone, on a fixed upstream gradient (both sides differentiate sum(out * grad_out)), with the same masks
    go = torch.linspace(-1, 1, out_before.numel()).view_as(out_before.cpu())
    model.zero_grad()
    xin = b.x[:, :8].clone().requires_grad_(True)
    model._dss2_attn_masks = masks
    _call(name, model, xin, b.edge_index, b.edge_attr[:, :6]).backward(go.cuda())
    lin = {dt: _oracle_run(name, sd, xc, eac, eic, stats, masks, dt, grad_out=go) for dt in (torch.float32, torch.float64)}
    terms = dict(lin[torch.float64][4], **{f"model.module_{2 * (NL - 1) + 1}.bias": go})   # bias gradients: column sums over the buses
    for k, p_ in model.named_parameters():
        assert_fp32_parity(p_.grad, lin[torch.float32][2][k], lin[torch.float64][2][k], k + " (fixed grad_out)", sum_of=terms.get(k))
    assert_fp32_parity(xin.grad, lin[torch.float32][3], lin[torch.float64][3], "grad_x (fixed grad_out)")


@pytest.mark.gpu
@pytest.mark.parametrize("case,nb", [("cigre14", 6), ("ober_sub", 3)])
@pytest.mark.parametrize("name", list(CASES))
def test_injected_masks_match_reference(monkeypatch, name, case, nb):
    for k, v in CASES[name][2].items():
        monkeypatch.setenv(k, v)
    b, stats = _batch(case, nb, seed=17)
    model, sd = _model(name, P, seed=9)
    heads = CASES[name][1].get("heads", 1)
    masks = random_masks(NL, heads, b.edge_index.size(1) + b.x.size(0), P, seed=23)
    ours = _check_step(name, model, b, stats, masks)
    _compare(name, model, b, stats, sd, masks, ours)


def _philox_masks(rng_state, heads, et, nt, p=P):
    """What the kernels' Philox stream applies, per layer [heads, Et + Nt], from dss2_attn_drop_mask."""
    from dss2 import _lib
    lib = _lib.load()
    out = []
    for l in range(NL - 1):
        m = torch.empty(heads, et + nt, dtype=torch.uint8, device="cuda")
        for h in range(heads):
            _lib.check(lib.dss2_attn_drop_mask(_lib.attn_drop(p, l, h, rng_state=rng_state), et, nt, _lib.ptr(m[h]), _lib.stream()),
                       "dss2_attn_drop_mask")
        out.append(m.cpu())
    return out


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["gat", "gat_heads3", "fagcn"])
def test_philox_masks_forward_and_backward_draw_the_same_bits(monkeypatch, name):
    """A training step with the in-kernel Philox stream; its masks, materialised by dss2_attn_drop_mask, fed to the reference: forward
    and every gradient match, so the forward, the statistics pass and both backward branches drew the same bits."""
    from dss2 import gat, gnn
    b, stats = _batch("ober_sub", 3, seed=18)
    model, sd = _model(name, P, seed=10)
    rng = torch.tensor([987654321987, 5], dtype=torch.int64, device="cuda")
    monkeypatch.setattr(gat if CASES[name][0] == "gat" else gnn, "fresh_rng_state", lambda device: rng.clone())
    ours = _check_step(name, model, b, stats, None)
    masks = _philox_masks(rng, CASES[name][1].get("heads", 1), b.edge_index.size(1), b.x.size(0))
    kept = torch.cat([m.flatten().float() for m in masks]).mean()
    assert 0.5 < float(kept) < 0.9, kept
    _compare(name, model, b, stats, sd, masks, ours)


@pytest.mark.gpu
def test_philox_mask_statistics_and_streams():
    """Oberrhein, B = 4096: the keep fraction over every (layer, head, edge key) lies within 5 sigma of 1 - p; masks differ between
    layers, heads and steps; the same {seed, step} gives the same mask."""
    from dss2 import synth
    grid = synth.load_grid("ober_sub")
    st = synth.synthetic_store(grid, 1, seed=1)
    B, heads = 4096, 2
    et, nt = B * st.max_edges, B * st.max_nodes
    rng = torch.tensor([1234567, 0], dtype=torch.int64, device="cuda")
    for p in (0.1, P):
        masks = _philox_masks(rng, heads, et, nt, p)
        allm = torch.stack(masks)
        n = allm.numel()
        frac = float(allm.double().mean())
        sigma = ((1 - p) * p / n) ** 0.5
        assert abs(frac - (1 - p)) <= 5 * sigma, (p, frac, sigma)
        for l in range(1, NL - 1):
            assert not torch.equal(masks[l], masks[0]), l
        assert not torch.equal(masks[0][0], masks[0][1])
        again = _philox_masks(rng.clone(), heads, et, nt, p)
        assert all(torch.equal(a, b_) for a, b_ in zip(masks, again))
        nxt = rng.clone()
        nxt[1] += 1
        assert not torch.equal(_philox_masks(nxt, heads, et, nt, p)[0], masks[0])
        # the coefficients are kept independently: neighbouring keys agree as often as chance says
        agree = float((masks[0][0][1:] == masks[0][0][:-1]).double().mean())
        assert abs(agree - ((1 - p) ** 2 + p ** 2)) < 0.01, agree


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["gat", "gat_heads2", "fagcn"])
def test_eval_mode_has_no_attention_dropout(name):
    """PyG honours self.training: after model.eval() the output is bit-identical to dropout=0 with the same weights; in train() mode
    under torch.no_grad() the masks apply."""
    b, _ = _batch("cigre14", 4, seed=19)
    model, sd = _model(name, P, seed=11)
    plain, _ = _model(name, 0.0, seed=11)
    x, ei, ea = b.x[:, :8], b.edge_index, b.edge_attr[:, :6]
    with torch.no_grad():
        model.eval()
        plain.eval()
        ev = _call(name, model, x, ei, ea)
        assert torch.equal(ev, _call(name, plain, x, ei, ea))
        plain.train()
        assert torch.equal(ev, _call(name, plain, x, ei, ea))
        model.train()
        tr = _call(name, model, x, ei, ea)
        assert not torch.equal(tr, ev)
        torch.manual_seed(3)
        a1 = _call(name, model, x, ei, ea)
        torch.manual_seed(3)
        assert torch.equal(a1, _call(name, model, x, ei, ea)), "torch.manual_seed makes the masks repeatable"


@pytest.mark.gpu
def test_graphed_trainer_gat_attention_dropout(monkeypatch):
    """GraphedTrainer(network='gat', spec=GATSpec(..., dropout=0.1)): the eager step equals the drop-in module's step given the same
    {seed, step} (loss and gradient bit for bit), the first replayed CUDA-graph step equals the eager step, and the replayed steps draw
    new masks (the graph reads the advancing step counter from the device)."""
    import data
    from dss2 import batching, gat, synth
    from dss2.gat import GATSpec
    from dss2.trainer import GraphedTrainer
    store = synth.synthetic_store(synth.load_grid("ober_sub"), 8, seed=6).to("cuda")
    nb = 5
    ids = torch.tensor([3, 0, 7, 1, 4], device="cuda")
    spec = GATSpec(dim_feat=8, dim_dense=32, dim_out=2, num_layers=8, edge_dim=6, dropout=0.1)
    tr = GraphedTrainer(store, nb, spec=spec, reg_coefs=REG_COEFS, lr=3e-3, seed=3, use_cuda_graph=True, network="gat")
    model = networks.GAT_DSSE(dim_feat=8, dim_dense=32, dim_out=2, heads=1, num_layers=8, edge_dim=6, dropout=0.1).cuda().train()
    with torch.no_grad():
        for name, p_ in model.named_parameters():
            off, n = tr.runner.table[name]
            p_.copy_(tr.flat[off:off + n].view_as(p_))
    stats = [t.cuda() for t in (store.x_mean, store.x_std, store.edge_mean, store.edge_std)]
    monkeypatch.setattr(gat, "fresh_rng_state", lambda device: tr.step_state.clone())
    tr.ids.copy_(ids)
    tr._enqueue(with_optimizer=False)
    torch.cuda.synchronize()
    b = batching.pack_batch(store, ids)
    out = model(b.x[:, :8], b.edge_index, b.edge_attr[:, :6])
    loss_m = data.gsp_wls_edge(input=b.x[:, :8], edge_input=b.edge_attr[:, :6], output=out, x_mean=stats[0], x_std=stats[1],
                               edge_mean=stats[2], edge_std=stats[3], edge_index=b.edge_index, reg_coefs=REG_COEFS, num_samples=None,
                               node_param=b.x[:, 8:], edge_param=b.edge_attr[:, 6:])
    loss_m.backward()
    assert torch.equal(tr.loss, loss_m.detach())
    for name, p_ in model.named_parameters():
        off, n = tr.runner.table[name]
        assert torch.equal(tr.flat_grad[off:off + n], p_.grad.reshape(-1)), name
    # the same step without dropout differs (the masks are in effect)
    plain = GraphedTrainer(store, nb, reg_coefs=REG_COEFS, lr=3e-3, seed=3, use_cuda_graph=False, network="gat")
    plain.ids.copy_(ids)
    plain._enqueue(with_optimizer=False)
    assert not torch.equal(plain.loss, tr.loss)
    loss_first = tr.loss.clone()
    tr.capture()
    assert torch.equal(tr.step(ids).clone(), loss_first), "the first replayed step is the eager step"
    torch.cuda.synchronize()
    keep = [t.clone() for t in (tr.flat, tr.exp_avg, tr.exp_inf, tr.step_state)]
    assert int(keep[3][1]) == 1
    loss_r2 = tr.step(ids).clone()          # replay at step 1
    torch.cuda.synchronize()
    for t, k in zip((tr.flat, tr.exp_avg, tr.exp_inf, tr.step_state), keep):
        t.copy_(k)
    tr._enqueue(with_optimizer=False)       # eager, same parameters, step 1
    torch.cuda.synchronize()
    assert torch.equal(tr.loss, loss_r2), "the replay used the step counter of the device"
    tr.step_state[1] = 0
    tr._enqueue(with_optimizer=False)       # same parameters, step 0's masks
    torch.cuda.synchronize()
    assert not torch.equal(tr.loss, loss_r2), "step 1 draws other masks than step 0"
