"""Host side of gnn_dsse (reference networks.py:11-69, the rest of SURVEY.md 8f-1): `model='gcn2'` (GCN2Conv stack, the default),
`model='fagcn'` (FAConv stack, with its attention dropout) and `model='tagcn'` (TAGConv stack) at width dim_feat == 8, followed by Linear(dim_feat, dim_dense), Linear(dim_dense, dim_out).
Spec, flat parameter layout under the names named_parameters() reports (`model.module_{2l}.weight1`, `.att_l.weight`, `.att_r.weight`, `.lins.{k}.weight`,
`model.module_{2l}.bias`, the head), launch sequence, autograd bridge.  All arithmetic is in csrc/gat.cu (k_gcn_dinv, k_prop8,
k_lin8_fwd/bwd, k_fa_fwd/bwd, k_outer_reduce, the mlp2 head); there is no CPU fallback.

Reference behaviours kept: the model takes the edge list AS GIVEN (one-way for the reference's data: no un-directing, networks.py:67-69),
so the propagation is not symmetric and the backward walks the out-edges; `x_0` is the model input (networks.py:68).  Not reproduced:
`cached=True` keeps the normalised adjacency of the FIRST batch forever (networks.py:12,39-43; SURVEY appendix A) - here it is
recomputed per batch, which is what the cache holds as long as the batch topology does not change."""
import ctypes
from dataclasses import dataclass

import torch

from . import _lib
from .head import head_bwd, head_fwd
from .ops import ParamPack, _align4, fresh_rng_state, require_cuda, resolve_graph, stage_rows

C = 8
ACTS = {"none": 0, "leaky_relu": 1, "relu": 2, "tanh": 3}


@dataclass(frozen=True)
class GNNSpec:
    model: str            # 'gcn2' | 'fagcn' | 'tagcn'
    dim_feat: int
    dim_dense: int
    dim_out: int
    num_layers: int
    alpha: float = 0.1    # main_param: GCN2Conv's alpha, FAConv's eps
    K: int = 3            # TAGConv
    bias: bool = True     # TAGConv
    self_loops: bool = True
    normalize: bool = True
    act: str = "leaky_relu"
    act_slope: float = 0.01
    dropout: float = 0.0  # FAConv's attention dropout (networks.py:46), applied when the caller asks for it; gcn2 / tagcn ignore it

    @property
    def n_conv(self):
        return self.num_layers - 1

    @property
    def M(self):
        return 1 if self.model == "gcn2" else self.K + 1

    def layout(self):
        off, table = 0, {}

        def put(name, n):
            nonlocal off
            table[name] = (off, n)
            off += n

        c = self.dim_feat
        for l in range(self.n_conv):
            p = f"model.module_{2 * l}."
            if self.model == "gcn2":
                put(p + "weight1", c * c)
            elif self.model == "fagcn":
                put(p + "att_l.weight", c)      # Linear(channels, 1, bias=False) x 2, contiguous: one 16-float gradient slot
                put(p + "att_r.weight", c)
            else:
                if self.bias:
                    put(p + "bias", c)
                    off = _align4(off + 0)
                    off = (off + 7) // 8 * 8      # the K+1 matrices start 32-byte aligned and contiguous
                for k in range(self.K + 1):
                    put(p + f"lins.{k}.weight", c * c)
            off = _align4(off)
        i = 2 * self.n_conv
        put(f"model.module_{i}.weight", self.dim_dense * c)
        put(f"model.module_{i}.bias", self.dim_dense)
        put(f"model.module_{i + 1}.weight", self.dim_out * self.dim_dense)
        put(f"model.module_{i + 1}.bias", self.dim_out)
        return table, _align4(off) + 16      # 16 floats of scratch behind the parameters (bias-sum slot of layers without a bias)


def validate(sp):
    if sp.model not in ("gcn2", "fagcn", "tagcn"):
        raise Exception("invalid model type")
    if sp.dim_feat != C:
        raise NotImplementedError(f"gnn_dsse kernels are built for dim_feat == {C}, got {sp.dim_feat}")
    if not (1 <= sp.dim_dense <= 32 and 1 <= sp.dim_out <= 8 and sp.num_layers >= 2):
        raise NotImplementedError(f"gnn_dsse kernels support dim_dense <= 32, dim_out <= 8, num_layers >= 2; got {sp}")
    if sp.model == "tagcn" and not (1 <= sp.K <= 3):
        raise NotImplementedError("gnn_dsse tagcn kernels support K in 1..3")
    if not sp.normalize:
        raise NotImplementedError("gnn_dsse kernels cover normalize=True (the reference default)")
    if sp.act not in ACTS:
        raise Exception("invalid activation type")


class GNNRunner:
    def __init__(self, spec):
        validate(spec)
        self.spec = spec
        self.table, self.flat_size = spec.layout()
        self.scratch_off = self.flat_size - 16
        self.lib = _lib.load()
        self.num_partials = self.lib.dss2_num_partials()

    def _p(self, t, name):
        return ctypes.c_void_p(t.data_ptr() + 4 * self.table[name][0])

    def _w(self, flat, l):
        p = f"model.module_{2 * l}."
        return self._p(flat, p + ("weight1" if self.spec.model == "gcn2" else "lins.0.weight"))

    def _w_off(self, l):
        p = f"model.module_{2 * l}."
        return self.table[p + ("weight1" if self.spec.model == "gcn2" else "lins.0.weight")][0]

    def alloc(self, num_nodes, device, need_grad=True):
        sp = self.spec
        f32 = dict(dtype=torch.float32, device=device)
        nlev = sp.K if sp.model == "tagcn" else 1         # per layer: h (gcn2), hop levels 1..K (tagcn); fagcn keeps none
        b = {"dinv": torch.empty(num_nodes, **f32), "acts": torch.empty(sp.n_conv, num_nodes, C, **f32),
             "lev": torch.empty(sp.n_conv, nlev, num_nodes, C, **f32), "h": torch.empty(num_nodes, sp.dim_dense, **f32),
             "out": torch.empty(num_nodes, sp.dim_out, **f32)}
        if need_grad:
            b["g8"] = [torch.empty(num_nodes, C, **f32) for _ in range(2)]
            b["gz"] = torch.empty(num_nodes, C, **f32)
            b["gin"] = torch.empty(sp.M, num_nodes, C, **f32)
            b["u"] = [torch.empty(num_nodes, C, **f32) for _ in range(2)]
            b["gx0"] = torch.zeros(num_nodes, C, **f32)
            b["gh"] = torch.empty(num_nodes, sp.dim_dense, **f32)
            b["partials"] = torch.zeros(self.num_partials, self.flat_size, **f32)
        return b

    @staticmethod
    def _ptr_array(tensors):
        arr = (ctypes.c_void_p * len(tensors))(*[t.data_ptr() for t in tensors])
        return arr

    @staticmethod
    def _stride_array(strides):
        return (ctypes.c_int64 * len(strides))(*strides)

    def _layer_inputs(self, bufs, l, x, xs):
        """(tensors, strides) of the M inputs of layer l's dense stage: gcn2: [h]; tagcn: [x_l, A x_l, ..., A^K x_l]."""
        sp = self.spec
        if sp.model == "gcn2":
            return [bufs["lev"][l, 0]], [C]
        xin, stride = (x, xs) if l == 0 else (bufs["acts"][l - 1], C)
        return [xin] + [bufs["lev"][l, k] for k in range(sp.K)], [stride] + [C] * sp.K

    def _drop(self, l, rng_state, masks):
        return _lib.attn_drop(self.spec.dropout, l, 0, rng_state, None if masks is None else masks[l][0])

    def forward(self, graph, x, xs, flat, bufs, rng_state=None, masks=None):
        """fagcn: attention dropout (p = spec.dropout) when the caller passes the device {seed, step} `rng_state` (Philox, layer uid =
        layer index) or `masks` (per layer uint8 [1, Et + Nt], dss2_attn_drop_t's edge-key layout); the backward must get the same."""
        sp, lib, st, g = self.spec, self.lib, _lib.stream(), graph.ref
        loops = 1 if (sp.self_loops and sp.model != "tagcn") else 0      # TAGConv: gcn_norm(add_self_loops=False)
        _lib.check(lib.dss2_gcn_dinv(g, loops, _lib.ptr(bufs["dinv"]), st), "dss2_gcn_dinv")
        for l in range(sp.n_conv):
            xin, stride = (x, xs) if l == 0 else (bufs["acts"][l - 1], C)
            if sp.model == "fagcn":
                p = f"model.module_{2 * l}."
                _lib.check(lib.dss2_fa_fwd_drop(g, _lib.ptr(bufs["dinv"]), loops, _lib.ptr(xin), stride, _lib.ptr(x), xs,
                                                self._p(flat, p + "att_l.weight"), self._p(flat, p + "att_r.weight"), sp.alpha, ACTS[sp.act],
                                                sp.act_slope, self._drop(l, rng_state, masks), _lib.ptr(bufs["acts"][l]), st), "dss2_fa_fwd_drop")
                continue
            if sp.model == "gcn2":
                # h = (1 - alpha) A x + alpha x_0   (GCN2Conv.forward: x.mul_(1 - alpha); x_0 = alpha * x_0; out = x.add_(x_0))
                _lib.check(lib.dss2_gcn_prop8(g, _lib.ptr(bufs["dinv"]), loops, 0, _lib.ptr(xin), stride, 1.0 - sp.alpha, _lib.ptr(x), xs, sp.alpha,
                                              _lib.ptr(bufs["lev"][l, 0]), st), "dss2_gcn_prop8")
            else:
                src, ss = xin, stride
                for k in range(sp.K):
                    _lib.check(lib.dss2_gcn_prop8(g, _lib.ptr(bufs["dinv"]), 0, 0, _lib.ptr(src), ss, 1.0, None, 0, 0.0, _lib.ptr(bufs["lev"][l, k]), st),
                               "dss2_gcn_prop8")
                    src, ss = bufs["lev"][l, k], C
            ins, strides = self._layer_inputs(bufs, l, x, xs)
            bias = self._p(flat, f"model.module_{2 * l}.bias") if (sp.model == "tagcn" and sp.bias) else None
            _lib.check(lib.dss2_lin8_fwd(graph.num_nodes, sp.M, 0 if sp.model == "gcn2" else 1, self._ptr_array(ins), self._stride_array(strides),
                                         self._w(flat, l), bias, ACTS[sp.act], sp.act_slope, _lib.ptr(bufs["acts"][l]), st), "dss2_lin8_fwd")
        i = 2 * sp.n_conv
        head_fwd(lib, graph.num_nodes, _lib.ptr(bufs["acts"][sp.n_conv - 1]), C, self._p(flat, f"model.module_{i}.weight"),
                 self._p(flat, f"model.module_{i}.bias"), sp.dim_dense, self._p(flat, f"model.module_{i + 1}.weight"),
                 self._p(flat, f"model.module_{i + 1}.bias"), sp.dim_out, _lib.ptr(bufs["h"]), _lib.ptr(bufs["out"]), st)
        return bufs["out"]

    def backward(self, graph, x, xs, flat, bufs, grad_out, flat_grad, rng_state=None, masks=None):
        """grad_out [Nt, dim_out] dense -> flat parameter gradient; returns grad wrt x [Nt, 8].  rng_state / masks: those of the forward."""
        sp, lib, st, g = self.spec, self.lib, _lib.stream(), graph.ref
        part, pstride = bufs["partials"], self.flat_size
        loops = 1 if (sp.self_loops and sp.model != "tagcn") else 0

        def pp(off):
            return ctypes.c_void_p(part.data_ptr() + 4 * off)

        i = 2 * sp.n_conv
        gy = bufs["g8"][0]
        head_bwd(lib, graph.num_nodes, _lib.ptr(bufs["acts"][sp.n_conv - 1]), C, self._p(flat, f"model.module_{i}.weight"),
                 self._p(flat, f"model.module_{i}.bias"), sp.dim_dense, self._p(flat, f"model.module_{i + 1}.weight"), sp.dim_out,
                 _lib.ptr(bufs["h"]), _lib.ptr(grad_out), _lib.ptr(bufs["gh"]), _lib.ptr(gy), pp(self.table[f"model.module_{i}.weight"][0]), pstride, st)
        bufs["gx0"].zero_()
        for l in reversed(range(sp.n_conv)):
            if sp.model == "fagcn":
                p = f"model.module_{2 * l}."
                xin, stride = (x, xs) if l == 0 else (bufs["acts"][l - 1], C)
                gx = bufs["g8"][(sp.n_conv - l) & 1]
                _lib.check(lib.dss2_fa_bwd_drop(g, _lib.ptr(bufs["dinv"]), loops, _lib.ptr(xin), stride, self._p(flat, p + "att_l.weight"),
                                                self._p(flat, p + "att_r.weight"), sp.alpha, ACTS[sp.act], sp.act_slope, self._drop(l, rng_state, masks),
                                                _lib.ptr(bufs["acts"][l]), _lib.ptr(gy), _lib.ptr(gx), _lib.ptr(bufs["gx0"]) if sp.alpha != 0.0 else None,
                                                pp(self.table[p + "att_l.weight"][0]), pstride, st), "dss2_fa_bwd_drop")
                if l == 0 and sp.alpha != 0.0:
                    gx.add_(bufs["gx0"])          # the x_0 path (eps * sum_l grad_z_l) joins the gradient of the model input
                gy = gx
                continue
            ins, strides = self._layer_inputs(bufs, l, x, xs)
            gins = [bufs["gin"][m] for m in range(sp.M)]
            w_off = self._w_off(l)
            has_bias = sp.model == "tagcn" and sp.bias
            b_off = (self.table[f"model.module_{2 * l}.bias"][0] if has_bias else self.scratch_off) - w_off
            _lib.check(lib.dss2_lin8_bwd(graph.num_nodes, sp.M, 0 if sp.model == "gcn2" else 1, self._ptr_array(ins), self._stride_array(strides),
                                         self._w(flat, l), ACTS[sp.act], sp.act_slope, _lib.ptr(bufs["acts"][l]), _lib.ptr(gy), _lib.ptr(bufs["gz"]),
                                         self._ptr_array(gins), _lib.ptr(bufs["gx0"]) if sp.model == "gcn2" else None, sp.alpha, pp(w_off), pstride,
                                         b_off, st), "dss2_lin8_bwd")
            gx = bufs["g8"][(sp.n_conv - l) & 1]
            if sp.model == "gcn2":
                # grad x_l = (1 - alpha) A^T grad_h; at layer 0 the accumulated x_0 path (alpha * sum_l grad_h_l) joins
                add = bufs["gx0"] if l == 0 else None
                _lib.check(lib.dss2_gcn_prop8(g, _lib.ptr(bufs["dinv"]), loops, 1, _lib.ptr(gins[0]), C, 1.0 - sp.alpha, _lib.ptr(add), C, 1.0,
                                              _lib.ptr(gx), st), "dss2_gcn_prop8")
            else:
                # Horner over the transposed hops: u = g_K; u = A^T u + g_m for m = K-1 .. 0
                u = gins[sp.K]
                for m in reversed(range(sp.K)):
                    dst = gx if m == 0 else bufs["u"][m & 1]
                    _lib.check(lib.dss2_gcn_prop8(g, _lib.ptr(bufs["dinv"]), 0, 1, _lib.ptr(u), C, 1.0, _lib.ptr(gins[m]), C, 1.0, _lib.ptr(dst), st),
                               "dss2_gcn_prop8")
                    u = dst
            gy = gx
        _lib.check(lib.dss2_reduce_partials(_lib.ptr(part), pstride, self.num_partials, self.flat_size, _lib.ptr(flat_grad), 0, st),
                   "dss2_reduce_partials")
        return gy


class _GNNFunction(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, edge_index, runner, pack, names, drop, masks, *params):
        require_cuda()
        out_device = x.device
        named = dict(zip(names, params))
        xg, xs = stage_rows(x)
        if xg.size(1) != C:
            raise _lib.Dss2Error(f"gnn_dsse kernels need {C} node features, got {xg.size(1)}")
        graph = resolve_graph(edge_index, xg.size(0))
        if graph.c.undirected != 1:
            raise _lib.Dss2Error("gnn_dsse expects the one-way edge list of the reference's data (from_bus -> to_bus)")
        rng_state = None
        with torch.cuda.device(xg.device):
            if drop and masks is not None:
                masks = [m.to(device=xg.device, dtype=torch.uint8).contiguous() for m in masks]
            elif drop:
                rng_state = fresh_rng_state(xg.device)
            else:
                masks = None
            flat = pack.gather(named)
            bufs = runner.alloc(xg.size(0), xg.device, need_grad=any(ctx.needs_input_grad))
            out = runner.forward(graph, xg, xs, flat, bufs, rng_state=rng_state, masks=masks)
        ctx.runner, ctx.pack, ctx.names, ctx.graph, ctx.params = runner, pack, names, graph, params
        ctx.saved = (xg, xs, flat, bufs, rng_state, masks)
        ctx.x_needs_grad, ctx.x_device = x.requires_grad, x.device
        result = out.clone()
        return result if out_device.type == "cuda" else result.to(out_device)

    @staticmethod
    def backward(ctx, grad_out):
        xg, xs, flat, bufs, rng_state, masks = ctx.saved
        runner = ctx.runner
        go = grad_out.to(device=xg.device, dtype=torch.float32).contiguous()
        with torch.cuda.device(xg.device):
            flat_grad = torch.empty(runner.flat_size, dtype=torch.float32, device=xg.device)
            gx = runner.backward(ctx.graph, xg, xs, flat, bufs, go, flat_grad, rng_state=rng_state, masks=masks)
        grads = ctx.pack.scatter_grads(flat_grad, dict(zip(ctx.names, ctx.params)))
        gx_ret = gx.clone().to(ctx.x_device) if ctx.x_needs_grad else None
        return (gx_ret, None, None, None, None, None, None, *grads)


def gnn_apply(runner, pack, named_params, x, edge_index, drop=False, masks=None):
    """drop: apply FAConv's attention dropout of runner.spec (training mode) - with `masks` (per layer uint8 [1, Et + Nt], 1 = keep) when
    given, else with a fresh Philox seed from torch's global generator."""
    names = tuple(named_params.keys())
    return _GNNFunction.apply(x, edge_index, runner, pack, names, drop, masks, *named_params.values())


def make_machinery(spec):
    return GNNRunner(spec), ParamPack(spec)
