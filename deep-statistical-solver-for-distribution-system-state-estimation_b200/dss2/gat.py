"""Host side of GAT_DSSE (reference networks.py:113-156, SURVEY.md 8f-1): architecture spec, flat parameter layout in the
reference's state_dict names (`model.module_{i}.*`, PyG `nn.Sequential` naming), kernel launch sequence, autograd bridge.

7 x [GATv2Conv(8, 8, heads=1, edge_dim) + LeakyReLU(0.01)] -> Linear(8, dim_dense) -> Linear(dim_dense, dim_out).
heads = H in 2..4 with concat=False (the only multi-head setting the reference model can run: with concat=True the next layer's
in_channels no longer match, networks.py:145): every head runs the single-head kernels on its slice of the parameters without bias and
activation, and the per-bus 8x8 kernels (dss2_lin8_fwd/bwd with weight blocks I / H) average the heads, add the bias and apply the
non-linearity.  All arithmetic is in csrc/gat.cu; there is no CPU fallback."""
import ctypes
import os
from dataclasses import dataclass

import torch

from . import _lib
from .head import head_bwd, head_fwd
from .ops import ParamPack, _align4, fresh_rng_state, require_cuda, resolve_graph, stage_rows

GAT_C = 8   # channels the kernels are built for (dim_feat of dss2_run.py:73)
GAT_SLOTS = 8   # constant-memory weight slots of csrc/gat.cu


@dataclass(frozen=True)
class GATSpec:
    dim_feat: int
    dim_dense: int
    dim_out: int
    num_layers: int       # the reference builds num_layers - 1 GATv2 layers (networks.py:144)
    edge_dim: int
    att_slope: float = 0.2
    act_slope: float = 0.01   # torch.nn.LeakyReLU() default (networks.py:137); 0 for nonlin='relu'
    act: str = "leaky_relu"   # nonlin of networks.py:130-137: 'leaky_relu' | 'relu' | 'tanh'
    self_loops: bool = True   # add_self_loops of the GATv2 layers (networks.py:145)
    heads: int = 1            # > 1: concat=False (mean over the heads)
    dropout: float = 0.0      # attention dropout of the GATv2 layers (networks.py:145-146), applied when the caller asks for it

    @property
    def act_code(self):
        """`act` argument of dss2_gat_fwd / dss2_gat_bwd (include/dss2_b200.h)."""
        return (2 if self.act == "tanh" else 1) | (0 if self.self_loops else 0x100)

    @property
    def n_conv(self):
        return self.num_layers - 1

    def param_names(self):
        """Reference parameter names (named_parameters() order of PyG's modules) with their shapes."""
        out = []
        for l in range(self.n_conv):
            p = f"model.module_{2 * l}."
            hc = self.heads * self.dim_feat
            out += [(p + "att", (1, self.heads, self.dim_feat)), (p + "bias", (self.dim_feat,)),
                    (p + "lin_l.weight", (hc, self.dim_feat)), (p + "lin_l.bias", (hc,)),
                    (p + "lin_r.weight", (hc, self.dim_feat)), (p + "lin_r.bias", (hc,)),
                    (p + "lin_edge.weight", (hc, self.edge_dim))]
        i = 2 * self.n_conv
        out += [(f"model.module_{i}.weight", (self.dim_dense, self.dim_feat)), (f"model.module_{i}.bias", (self.dim_dense,)),
                (f"model.module_{i + 1}.weight", (self.dim_out, self.dim_dense)), (f"model.module_{i + 1}.bias", (self.dim_out,))]
        return out

    def layout(self):
        """name -> (offset, numel) in the flat fp32 buffer.  Per GATv2 layer [lin_l.w | lin_r.w | lin_l.b | lin_r.b | lin_edge.w | att |
        bias] (all sizes are multiples of 4 floats for dim_feat = 8 and even edge_dim); the backward gets the blocks' offsets
        (`part_off`), the head is [w1 | b1 | w2 | b2]."""
        off, table = 0, {}

        def put(name, n):
            nonlocal off
            table[name] = (off, n)
            off += n

        c, fe, H = self.dim_feat, self.edge_dim, self.heads
        for l in range(self.n_conv):
            p = f"model.module_{2 * l}."
            put(p + "lin_l.weight", H * c * c)     # H > 1: every parameter holds its heads one after the other (PyG's [H * C, ...] rows)
            put(p + "lin_r.weight", H * c * c)     # the two Linears' weights, then their biases, adjacent: one gradient reduction for both
            put(p + "lin_l.bias", H * c)
            put(p + "lin_r.bias", H * c)
            put(p + "lin_edge.weight", H * c * fe)
            put(p + "att", H * c)
            put(p + "bias", c)
            off = _align4(off)
        i = 2 * self.n_conv
        put(f"model.module_{i}.weight", self.dim_dense * c)
        put(f"model.module_{i}.bias", self.dim_dense)
        put(f"model.module_{i + 1}.weight", self.dim_out * self.dim_dense)
        put(f"model.module_{i + 1}.bias", self.dim_out)
        off = _align4(off)
        if H > 1:      # not parameters: the head-averaging blocks [H][8][8] = I / H, a zero bias, and a gradient slot nobody reads
            put("_mean_blocks", H * c * c)
            put("_zero_bias", c)
            put("_scratch", c)
        return table, _align4(off)


def validate_gat_spec(sp):
    if sp.dim_feat != GAT_C:
        raise NotImplementedError(f"GAT_DSSE kernels are built for dim_feat == {GAT_C} (dss2_run.py:73), got {sp.dim_feat}")
    if not 1 <= sp.heads <= 4:
        raise NotImplementedError(f"GAT_DSSE kernels support heads in 1..4, got {sp.heads}")
    if not (1 <= sp.edge_dim <= 8 and 1 <= sp.dim_dense <= 32 and 1 <= sp.dim_out <= 8 and sp.num_layers >= 2):
        raise NotImplementedError(f"GAT_DSSE kernels support edge_dim <= 8, dim_dense <= 32, dim_out <= 8, num_layers >= 2; got {sp}")


class GATRunner:
    def __init__(self, spec):
        validate_gat_spec(spec)
        self.spec = spec
        self.table, self.flat_size = spec.layout()
        self.lib = _lib.load()
        self.num_partials = self.lib.dss2_num_partials()
        self._lin8_act = {"leaky_relu": 1, "relu": 2, "tanh": 3}[spec.act]      # act codes of dss2_lin8_fwd / bwd

    def _p(self, flat, name):
        return ctypes.c_void_p(flat.data_ptr() + 4 * self.table[name][0])

    def _layer(self, flat, l):
        p = f"model.module_{2 * l}."
        return [self._p(flat, p + k) for k in ("lin_l.weight", "lin_l.bias", "lin_r.weight", "lin_r.bias", "lin_edge.weight", "att", "bias")]

    # ---- single-head layers: weights in constant-memory slots (csrc/gat.cu, dss2_gat_upload) ----
    def use_slots(self):
        return self.spec.heads == 1 and self.spec.n_conv <= GAT_SLOTS and os.environ.get("DSS2_GAT_SLOTS", "1") != "0"

    def upload(self, flat):
        sp = self.spec
        arr = ctypes.c_void_p * sp.n_conv
        cols = [arr(*[self._layer(flat, l)[k] for l in range(sp.n_conv)]) for k in range(7)]
        _lib.check(self.lib.dss2_gat_upload(0, sp.n_conv, *cols, sp.edge_dim, _lib.stream()), "dss2_gat_upload")

    _HEAD_BLOCKS = (("lin_l.weight", GAT_C * GAT_C), ("lin_l.bias", GAT_C), ("lin_r.weight", GAT_C * GAT_C), ("lin_r.bias", GAT_C),
                    ("lin_edge.weight", None), ("att", GAT_C))

    def _layer_offsets(self, l):
        """part_off of layer l relative to its lin_l.weight (single head)."""
        p = f"model.module_{2 * l}."
        base = self.table[p + "lin_l.weight"][0]
        return (ctypes.c_int64 * 7)(*[self.table[p + k][0] - base for k in ("lin_l.weight", "lin_l.bias", "lin_r.weight", "lin_r.bias",
                                                                              "lin_edge.weight", "att", "bias")])

    def _head_offsets(self, l, h):
        """Flat offsets of head h's slice of the six per-head parameters of layer l, then of the unused bias slot."""
        p = f"model.module_{2 * l}."
        offs = [self.table[p + k][0] + h * (n if n is not None else GAT_C * self.spec.edge_dim) for k, n in self._HEAD_BLOCKS]
        return offs + [self.table["_scratch"][0]]

    def _head(self, flat, l, h):
        offs = self._head_offsets(l, h)
        ptrs = [ctypes.c_void_p(flat.data_ptr() + 4 * o) for o in offs[:6]]
        return ptrs + [self._p(flat, "_zero_bias")]

    def prepare(self, flat):
        """heads > 1: (re)write the constant tail of the flat buffer (I / H blocks, zero bias) - the optimizer may have touched it."""
        sp = self.spec
        if sp.heads > 1:
            off, n = self.table["_mean_blocks"]
            eye = torch.eye(GAT_C, dtype=torch.float32, device=flat.device) / sp.heads
            flat[off:off + n].copy_(eye.repeat(sp.heads, 1, 1).reshape(-1))
            for name in ("_zero_bias", "_scratch"):
                off, n = self.table[name]
                flat[off:off + n].zero_()

    @staticmethod
    def _arr(tensors):
        return (ctypes.c_void_p * len(tensors))(*[t.data_ptr() for t in tensors])

    @staticmethod
    def _strides(n):
        return (ctypes.c_int64 * n)(*([GAT_C] * n))

    def alloc(self, num_nodes, device, need_grad=True):
        sp = self.spec
        f32 = dict(dtype=torch.float32, device=device)
        b = {"acts": torch.empty(sp.n_conv, num_nodes, GAT_C, **f32),      # outputs of the GATv2 layers
             "h": torch.empty(num_nodes, sp.dim_dense, **f32), "out": torch.empty(num_nodes, sp.dim_out, **f32)}
        if sp.heads > 1:
            b["raw"] = torch.empty(sp.n_conv, sp.heads, num_nodes, GAT_C, **f32)    # per-head outputs before mean / bias / activation
            if need_grad:
                b["graw"] = torch.empty(sp.heads, num_nodes, GAT_C, **f32)
                b["gxh"] = torch.empty(sp.heads, num_nodes, GAT_C, **f32)
                b["gz"] = torch.empty(num_nodes, GAT_C, **f32)
        if need_grad:
            b["g8"] = [torch.empty(num_nodes, GAT_C, **f32) for _ in range(2)]
            b["gh"] = torch.empty(num_nodes, sp.dim_dense, **f32)
            b["ws"] = torch.empty(self.lib.dss2_gat_ws_bytes(num_nodes) // 4, **f32)
            b["partials"] = torch.zeros(self.num_partials, self.flat_size, **f32)
        return b

    def _drop(self, l, h, rng_state, masks):
        return _lib.attn_drop(self.spec.dropout, l, h, rng_state, None if masks is None else masks[l][h])

    def forward(self, graph, x, xs, ea, eas, flat, bufs, rng_state=None, masks=None):
        """Attention dropout (p = spec.dropout) is applied when the caller passes the device {seed, step} `rng_state` (Philox, layer uid =
        layer index, one stream per head) or `masks` (per layer uint8 [heads, Et + Nt], dss2_attn_drop_t's edge-key layout); the backward
        must get the same."""
        sp, lib, st = self.spec, self.lib, _lib.stream()
        g = graph.ref
        H = sp.heads
        if H > 1:
            self.prepare(flat)
        slots = self.use_slots()
        if slots:
            self.upload(flat)
        for l in range(sp.n_conv):
            xin, stride = (x, xs) if l == 0 else (bufs["acts"][l - 1], GAT_C)
            if H > 1:
                raw = bufs["raw"][l]
                for h in range(H):
                    _lib.check(lib.dss2_gat_fwd_drop(g, _lib.ptr(xin), stride, _lib.ptr(ea), eas, sp.edge_dim, -1, *self._head(flat, l, h),
                                                     sp.att_slope, sp.act_code & 0x100, 0.0, self._drop(l, h, rng_state, masks), _lib.ptr(raw[h]), st),
                               "dss2_gat_fwd_drop")
                # y = act(sum_h raw_h (I / H) + bias)
                _lib.check(lib.dss2_lin8_fwd(graph.num_nodes, H, 1, self._arr([raw[h] for h in range(H)]), self._strides(H),
                                             self._p(flat, "_mean_blocks"), self._p(flat, f"model.module_{2 * l}.bias"), self._lin8_act,
                                             sp.act_slope, _lib.ptr(bufs["acts"][l]), st), "dss2_lin8_fwd")
                continue
            # slots: the weights are immediate operands from constant-memory slot l (the pointers are not read)
            _lib.check(lib.dss2_gat_fwd_drop(g, _lib.ptr(xin), stride, _lib.ptr(ea), eas, sp.edge_dim, l if slots else -1, *self._layer(flat, l),
                                             sp.att_slope, sp.act_code, sp.act_slope, self._drop(l, 0, rng_state, masks), _lib.ptr(bufs["acts"][l]),
                                             st), "dss2_gat_fwd_drop")
        i = 2 * sp.n_conv
        head_fwd(lib, graph.num_nodes, _lib.ptr(bufs["acts"][sp.n_conv - 1]), GAT_C, self._p(flat, f"model.module_{i}.weight"),
                 self._p(flat, f"model.module_{i}.bias"), sp.dim_dense, self._p(flat, f"model.module_{i + 1}.weight"),
                 self._p(flat, f"model.module_{i + 1}.bias"), sp.dim_out, _lib.ptr(bufs["h"]), _lib.ptr(bufs["out"]), st)
        return bufs["out"]

    def backward(self, graph, x, xs, ea, eas, flat, bufs, grad_out, flat_grad, need_gx=False, uploaded=False, rng_state=None, masks=None):
        """grad_out [Nt, dim_out] dense -> flat parameter gradient (and grad wrt x when need_gx).  uploaded: the constant-memory slots
        still hold this model's weights (the captured step: forward and backward of one step, nothing in between).  rng_state / masks:
        those of the forward."""
        sp, lib, st = self.spec, self.lib, _lib.stream()
        g = graph.ref
        slots = self.use_slots()
        if slots and not uploaded:
            self.upload(flat)
        part, pstride = bufs["partials"], self.flat_size

        def pp(name):
            return ctypes.c_void_p(part.data_ptr() + 4 * self.table[name][0])

        i = 2 * sp.n_conv
        gy = bufs["g8"][0]
        head_bwd(lib, graph.num_nodes, _lib.ptr(bufs["acts"][sp.n_conv - 1]), GAT_C, self._p(flat, f"model.module_{i}.weight"),
                 self._p(flat, f"model.module_{i}.bias"), sp.dim_dense, self._p(flat, f"model.module_{i + 1}.weight"), sp.dim_out,
                 _lib.ptr(bufs["h"]), _lib.ptr(grad_out), _lib.ptr(bufs["gh"]), _lib.ptr(gy), pp(f"model.module_{i}.weight"), pstride, st)
        gx_out = None
        for l in reversed(range(sp.n_conv)):
            xin, stride = (x, xs) if l == 0 else (bufs["acts"][l - 1], GAT_C)
            want_gx = l > 0 or need_gx
            gx = bufs["g8"][(sp.n_conv - l) & 1] if want_gx else None
            if sp.heads > 1:
                H, raw, graw, gxh = sp.heads, bufs["raw"][l], bufs["graw"], bufs["gxh"]
                base = self.table[f"model.module_{2 * l}.lin_l.weight"][0]
                # grad_raw_h = grad_z / H, bias gradient (weight_is_out_by_in = 1: the bias column sums grad_z); the (unused) gradient of the
                # constant I / H blocks lands behind the parameters
                mb = self.table["_mean_blocks"][0]
                _lib.check(lib.dss2_lin8_bwd(graph.num_nodes, H, 1, self._arr([raw[h] for h in range(H)]), self._strides(H),
                                             self._p(flat, "_mean_blocks"), self._lin8_act, sp.act_slope, _lib.ptr(bufs["acts"][l]), _lib.ptr(gy),
                                             _lib.ptr(bufs["gz"]), self._arr([graw[h] for h in range(H)]), None, 0.0,
                                             ctypes.c_void_p(part.data_ptr() + 4 * mb), pstride, self.table[f"model.module_{2 * l}.bias"][0] - mb, st),
                           "dss2_lin8_bwd")
                for h in range(H):
                    offs = (ctypes.c_int64 * 7)(*[o - base for o in self._head_offsets(l, h)])
                    _lib.check(lib.dss2_gat_bwd_drop(g, _lib.ptr(xin), stride, _lib.ptr(ea), eas, sp.edge_dim, -1, *self._head(flat, l, h),
                                                     sp.att_slope, sp.act_code & 0x100, 0.0, self._drop(l, h, rng_state, masks), _lib.ptr(raw[h]),
                                                     _lib.ptr(graw[h]), _lib.ptr(gxh[h]) if want_gx else None, _lib.ptr(bufs["ws"]),
                                                     bufs["ws"].numel() * 4, pp(f"model.module_{2 * l}.lin_l.weight"), pstride, offs, st),
                               "dss2_gat_bwd_drop")
                if want_gx:     # grad_x = sum over the heads (identity blocks = H * (I / H): scale folded into one more 8x8 pass)
                    _lib.check(lib.dss2_lin8_fwd(graph.num_nodes, H, 1, self._arr([gxh[h] for h in range(H)]), self._strides(H),
                                                 self._p(flat, "_mean_blocks"), None, 0, 0.0, _lib.ptr(gx), st), "dss2_lin8_fwd")
                    gx.mul_(float(H))
                gy = gx
                gx_out = gx
                continue
            _lib.check(lib.dss2_gat_bwd_drop(g, _lib.ptr(xin), stride, _lib.ptr(ea), eas, sp.edge_dim, l if slots else -1, *self._layer(flat, l),
                                             sp.att_slope, sp.act_code, sp.act_slope, self._drop(l, 0, rng_state, masks), _lib.ptr(bufs["acts"][l]),
                                             _lib.ptr(gy), _lib.ptr(gx), _lib.ptr(bufs["ws"]), bufs["ws"].numel() * 4,
                                             pp(f"model.module_{2 * l}.lin_l.weight"), pstride, self._layer_offsets(l), st), "dss2_gat_bwd_drop")
            gy = gx
            gx_out = gx
        _lib.check(lib.dss2_reduce_partials(_lib.ptr(part), pstride, self.num_partials, self.flat_size, _lib.ptr(flat_grad), 0, st),
                   "dss2_reduce_partials")
        return gx_out


class _GATFunction(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, edge_attr, edge_index, runner, pack, names, drop, masks, *params):
        require_cuda()
        out_device = x.device
        named = dict(zip(names, params))
        xg, xs = stage_rows(x)
        eag, eas = stage_rows(edge_attr)
        graph = resolve_graph(edge_index, xg.size(0))
        rng_state = None
        with torch.cuda.device(xg.device):
            if drop and masks is not None:
                masks = [m.to(device=xg.device, dtype=torch.uint8).contiguous() for m in masks]
            elif drop:
                rng_state = fresh_rng_state(xg.device)
            else:
                masks = None
            flat = pack.gather(named)
            bufs = runner.alloc(xg.size(0), xg.device, need_grad=any(ctx.needs_input_grad))   # False under torch.no_grad()
            out = runner.forward(graph, xg, xs, eag, eas, flat, bufs, rng_state=rng_state, masks=masks)
        ctx.runner, ctx.pack, ctx.names, ctx.graph, ctx.params = runner, pack, names, graph, params
        ctx.saved = (xg, xs, eag, eas, flat, bufs, rng_state, masks)
        ctx.x_needs_grad, ctx.x_shape, ctx.x_device = x.requires_grad, x.shape, x.device
        result = out.clone()
        return result if out_device.type == "cuda" else result.to(out_device)

    @staticmethod
    def backward(ctx, grad_out):
        xg, xs, eag, eas, flat, bufs, rng_state, masks = ctx.saved
        runner = ctx.runner
        go = grad_out.to(device=xg.device, dtype=torch.float32).contiguous()
        with torch.cuda.device(xg.device):
            flat_grad = torch.empty(runner.flat_size, dtype=torch.float32, device=xg.device)
            gx = runner.backward(ctx.graph, xg, xs, eag, eas, flat, bufs, go, flat_grad, need_gx=ctx.x_needs_grad, rng_state=rng_state, masks=masks)
        grads = ctx.pack.scatter_grads(flat_grad, dict(zip(ctx.names, ctx.params)))
        gx_ret = gx.clone().to(ctx.x_device) if ctx.x_needs_grad else None
        return (gx_ret, None, None, None, None, None, None, None, *grads)


def gat_apply(runner, pack, named_params, x, edge_index, edge_attr, drop=False, masks=None):
    """drop: apply the attention dropout of runner.spec (training mode) - with `masks` (per layer uint8 [heads, Et + Nt], 1 = keep) when
    given, else with a fresh Philox seed from torch's global generator (so torch.manual_seed makes runs repeatable)."""
    names = tuple(named_params.keys())
    return _GATFunction.apply(x, edge_attr, edge_index, runner, pack, names, drop, masks, *named_params.values())


def make_machinery(spec):
    return GATRunner(spec), ParamPack(spec)
