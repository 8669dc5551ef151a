"""Host side of the layer kernels: model spec + flat parameter layout, the launch sequence of a whole
(Skip)PFN forward / backward, and the torch.autograd bridges used by the drop-in `networks` / `data`
modules.  All arithmetic happens in libdss2_b200.so; torch supplies device memory and streams.
"""
import ctypes
import os
from dataclasses import dataclass

import torch

from . import _lib
from .graph import BatchGraph, graph_for

MAX_EA_SLOTS = 7   # constant-memory slots of the prepared-weights EdgeAggregation path (include/dss2_b200.h)
HID = _lib.HID
# which TAG-layer kernels the runner launches (all are CUDA; there is no CPU path):
#   "ffma": CUDA-core forward and backward (tag.cu)
#   "tc2" : tcgen05 forward AND backward (tag_tc3.cu TMA-fed, tag_tc2.cu direct loads); tiles of up to 256 rows (two MMA blocks)
# Unsupported shapes (K = 3, oversize tiles) fall back to the CUDA-core kernels.
TAG_IMPL = os.environ.get("DSS2_TAG_IMPL", "tc2")
# weight-gradient pass behind the tc2 backward: "tc" = tcgen05 3xTF32 GEMM (68.7 us on the bench layer), "ffma" = exact fp32 streaming
# kernel on the CUDA cores (82.5 us; profiles/r1k_bench.json) - the tensor cores are used because they measure faster
GW_IMPL = os.environ.get("DSS2_GW_IMPL", "tc")
# consecutive TAG layers of a sub-net linked per tile (programmatic dependent launch + tile marks) instead of per grid: DSS2_CHAIN=0 disables
CHAIN = os.environ.get("DSS2_CHAIN", "1") != "0"
# backward: chained backward-to-input launches on the current stream, weight-gradient passes on a second one (DSS2_CHAIN_BWD=0 disables)
CHAIN_BWD = CHAIN and os.environ.get("DSS2_CHAIN_BWD", "1") != "0"


def tile_cap():
    """Max node rows of a shared-memory tile the batch structure is built for (all layer kernels accept up to 256)."""
    return int(os.environ.get("DSS2_TILE_CAP", _lib.TILE_CAP))


def _align4(n):
    return (n + 3) & ~3


@dataclass(frozen=True)
class PFNSpec:
    """Architecture of MPN / SkipMPN / PFN / SkipPFN (networks.py:212-388) as one stack of sub-nets.
    Sub-net s: EdgeAggregation(fn -> 32) then n_layers TAGConv(K); the last TAGConv maps 32 -> out_s
    with out_s = dim_out for the last sub-net and fn otherwise (networks.py:355-357,380-382)."""
    fn: int
    fe: int
    dim_out: int
    n_layers: int
    K: int
    L: int
    p_drop: float
    skip: tuple          # per sub-net: add the input back (SkipMPN, networks.py:336)
    prefix_fmt: str      # "mpns.{s}." for PFN/SkipPFN, "" for a single MPN/SkipMPN
    hid: int = HID

    def out_dim(self, s):
        return self.dim_out if s == self.L - 1 else self.fn

    def param_names(self):
        """Reference parameter names in named_parameters() order with their shapes."""
        out = []
        for s in range(self.L):
            pre = self.prefix_fmt.format(s=s)
            ld = 2 * self.fn + self.fe
            out += [(pre + "edge_aggr.edge_aggr.0.weight", (self.hid, ld)), (pre + "edge_aggr.edge_aggr.0.bias", (self.hid,)),
                    (pre + "edge_aggr.edge_aggr.2.weight", (self.hid, self.hid)), (pre + "edge_aggr.edge_aggr.2.bias", (self.hid,))]
            for l in range(self.n_layers):
                cout = self.out_dim(s) if l == self.n_layers - 1 else self.hid
                out.append((pre + f"convs.{l}.bias", (cout,)))
                for k in range(self.K + 1):
                    out.append((pre + f"convs.{l}.lins.{k}.weight", (cout, self.hid)))
        return out

    def layout(self):
        """name -> (offset, numel) in the flat fp32 buffer; every tensor starts 16-byte aligned and the
        K+1 matrices of one TAGConv are contiguous ([K+1, cout, 32])."""
        off, table = 0, {}
        for name, shape in self.param_names():
            n = 1
            for d in shape:
                n *= d
            table[name] = (off, n)
            off += _align4(n)
        return table, off


def validate_spec(spec):
    if spec.hid != HID:
        raise _lib.Dss2Error(f"dim_hid={spec.hid}: the sm_100a layer kernels are specialised for dim_hid={HID}")
    if not (1 <= spec.fn <= 8 and 1 <= spec.fe <= 8):
        raise _lib.Dss2Error("EdgeAggregation kernels support 1..8 node and edge features")
    if not (1 <= spec.K <= 3):
        raise _lib.Dss2Error("TAGConv kernels support K in 1..3")
    if not (1 <= spec.dim_out <= HID):
        raise _lib.Dss2Error("dim_out must be in 1..32")
    if any(spec.skip[s] and spec.out_dim(s) != spec.fn for s in range(spec.L)):
        raise _lib.Dss2Error("skip connection needs dim_out == dim_featn (networks.py:336)")


class PFNRunner:
    """Launch sequence of one forward / backward over raw device buffers (no autograd, no allocation after
    `alloc`): used by the autograd bridge below and, with static buffers, by the CUDA-graph trainer."""

    def __init__(self, spec):
        validate_spec(spec)
        self.spec = spec
        self.table, self.flat_size = spec.layout()
        self.lib = _lib.load()
        self.num_partials = self.lib.dss2_num_partials()

    # ---- buffers ----
    def alloc(self, num_nodes, device, need_grad=True, pipelined=False):
        sp = self.spec
        f32 = dict(dtype=torch.float32, device=device)
        b = {
            "acts": torch.empty(sp.L, sp.n_layers, num_nodes, HID, **f32),    # [s][l] = input of TAG layer l
            # one sign word per node; rows padded to 64 words so every [s, l] slice starts 256-byte aligned (bulk-copy source)
            "bits": torch.empty(sp.L, max(sp.n_layers - 1, 1), (num_nodes + 63) // 64 * 64, dtype=torch.int32, device=device),
            "outs": [torch.empty(num_nodes, sp.out_dim(s), **f32) for s in range(sp.L)],
            # per-tile completion marks of every forward layer launch (layer chaining; one 32-bit word per tile, 256-tile upper bound per row)
            "marks": torch.zeros(sp.L, sp.n_layers, (num_nodes + 255) // 256 * 256 + 256, dtype=torch.int32, device=device),
        }
        if need_grad:
            b["g32"] = [torch.empty(num_nodes, HID, **f32) for _ in range(2)]
            b["gsub"] = [torch.empty(num_nodes, sp.fn, **f32) for _ in range(2)]
            b["partials"] = torch.zeros(self.num_partials, self.flat_size, **f32)
            b["lvl"] = torch.empty(self.lib.dss2_tag_bwd_tc2_workspace_bytes(num_nodes, sp.K) // 4, **f32)
            if pipelined:
                # two-stream backward (see backward()): the gradient of every layer input and the spilled hop levels of every layer stay
                # alive until that layer's weight-gradient pass has read them on the second stream
                b["gchain"] = torch.empty(sp.n_layers, num_nodes, HID, **f32)
                b["lvls"] = torch.empty(sp.n_layers, b["lvl"].numel(), **f32)
                b["marks_b"] = torch.zeros_like(b["marks"])
        return b

    def _p(self, flat, name):
        off, _ = self.table[name]
        return ctypes.c_void_p(flat.data_ptr() + 4 * off)

    # ---- EdgeAggregation weights -> constant-memory slots (thread-per-row kernels, csrc/edgeagg_row.cu) ----
    def _ea_names(self, s):
        pre = self.spec.prefix_fmt.format(s=s) + "edge_aggr.edge_aggr."
        return pre + "0.weight", pre + "0.bias", pre + "2.weight", pre + "2.bias"

    def ea_slots(self, graph, x_stride, ea_stride):
        """True when every EdgeAggregation of the model can run from prepared constant-memory slots (one per sub-net)."""
        sp = self.spec
        if sp.L > MAX_EA_SLOTS or os.environ.get("DSS2_EA_IMPL", "row")[:1] == "w":
            return False
        return bool(self.lib.dss2_edgeagg_slots_ok(graph.ref, max(x_stride, sp.fn), ea_stride, sp.fe))

    def ea_upload(self, flat):
        """One layout kernel + one device-to-device copy node for all sub-nets (capturable)."""
        sp = self.spec
        arr = ctypes.c_void_p * sp.L
        cols = [arr(*[self._p(flat, self._ea_names(s)[k]) for s in range(sp.L)]) for k in range(4)]
        _lib.check(self.lib.dss2_edgeagg_upload(0, sp.L, *cols, sp.fn, sp.fe, _lib.stream()), "dss2_edgeagg_upload")

    # ---- forward ----
    def forward(self, graph, x, x_stride, ea, ea_stride, flat, bufs, drop_mode=1, rng_state=None, masks=None, ea_uploaded=False):
        """x: tensor whose data_ptr is row 0 / col 0 of the [Nt, fn] input with row stride x_stride.
        masks: optional [L][n_layers-1] uint8 [Nt,32] tensors (drop_mode 2).  ea_uploaded: the caller has already run ea_upload(flat)
        for this step (the trainer does, beside the batch packer).  Returns bufs['outs'][-1]."""
        sp, lib, st = self.spec, self.lib, _lib.stream()
        g = graph.ref
        use_tc2 = TAG_IMPL == "tc2" and bool(lib.dss2_tag_tc2_supported(g, sp.K))
        slots = self.ea_slots(graph, x_stride, ea_stride)
        if slots and not ea_uploaded:
            self.ea_upload(flat)
        chain = use_tc2 and CHAIN and rng_state is not None and "marks" in bufs
        for s in range(sp.L):
            pre = sp.prefix_fmt.format(s=s)
            xin, xs = (x, x_stride) if s == 0 else (bufs["outs"][s - 1], sp.fn)
            if slots:
                _lib.check(lib.dss2_edgeagg_fwd_slot(g, _lib.ptr(xin), xs, sp.fn, _lib.ptr(ea), ea_stride, sp.fe, s, _lib.ptr(bufs["acts"][s, 0]), st),
                           "dss2_edgeagg_fwd_slot")
            else:
                _lib.check(lib.dss2_edgeagg_fwd(g, _lib.ptr(xin), xs, sp.fn, _lib.ptr(ea), ea_stride, sp.fe,
                                                *[self._p(flat, n) for n in self._ea_names(s)], _lib.ptr(bufs["acts"][s, 0]), st), "dss2_edgeagg_fwd")
            for l in range(sp.n_layers):
                last = l == sp.n_layers - 1
                cout = sp.out_dim(s) if last else HID
                y = bufs["outs"][s] if last else bufs["acts"][s, l + 1]
                mask = None
                mode = 0 if last else drop_mode
                if not last and drop_mode == 2:
                    mask = masks[s][l]
                res, rs = (xin, xs) if (last and sp.skip[s]) else (None, 0)
                args = (g, _lib.ptr(bufs["acts"][s, l]), self._p(flat, pre + f"convs.{l}.lins.0.weight"),
                        self._p(flat, pre + f"convs.{l}.bias"), cout, sp.K, 0 if last else 1, sp.p_drop, mode,
                        _lib.ptr(rng_state), s * sp.n_layers + l, _lib.ptr(mask), _lib.ptr(res), rs,
                        _lib.ptr(y), None if last else _lib.ptr(bufs["bits"][s, l]))
                if chain:   # layers of a sub-net linked per tile: layer l+1 starts on the SMs layer l's CTAs leave (csrc/tc2_shared.cuh)
                    marks = bufs["marks"]
                    _lib.check(lib.dss2_tag_fwd_tc2_chain(*args, None if last else _lib.ptr(marks[s, l]), _lib.ptr(marks[s, l - 1]) if l > 0 else None,
                                                          st), "dss2_tag_fwd_tc2_chain")
                else:
                    _lib.check((lib.dss2_tag_fwd_tc2 if use_tc2 else lib.dss2_tag_fwd)(*args, st), "dss2_tag_fwd")
        return bufs["outs"][-1]

    # ---- backward ----
    def backward(self, graph, x, x_stride, ea, ea_stride, flat, bufs, grad_out, flat_grad, accumulate=False, ea_uploaded=False, rng_state=None,
                 bucket_hook=None):
        """grad_out [Nt, dim_out] dense.  Writes the flat parameter gradient into flat_grad.  ea_uploaded: the constant-memory slots
        still hold this model's EdgeAggregation weights (the captured step: forward and backward of one step, nothing in between).
        rng_state (device {seed, step}) with buffers from alloc(pipelined=True) selects the two-stream schedule (_backward_pipelined).
        bucket_hook(lo, hi): two-stream schedule only - called on the second stream once flat_grad[lo:hi] (one sub-net) is final, e.g. to
        all-reduce it while the next sub-net's backward runs; self.bucketed tells whether the hook was used."""
        sp, lib, st = self.spec, self.lib, _lib.stream()
        self.bucketed = False
        if (CHAIN_BWD and rng_state is not None and "gchain" in bufs and TAG_IMPL == "tc2" and GW_IMPL == "tc"
                and bool(lib.dss2_tag_tc2_supported(graph.ref, sp.K))):
            return self._backward_pipelined(graph, x, x_stride, ea, ea_stride, flat, bufs, grad_out, flat_grad, accumulate, ea_uploaded, rng_state,
                                            bucket_hook)
        g = graph.ref
        slots = self.ea_slots(graph, x_stride, ea_stride)
        if slots and not ea_uploaded:
            self.ea_upload(flat)
        part = bufs["partials"]
        pstride = self.flat_size

        def pp(name):
            return ctypes.c_void_p(part.data_ptr() + 4 * self.table[name][0])

        use_tc2 = TAG_IMPL == "tc2" and bool(lib.dss2_tag_tc2_supported(g, sp.K))
        gy = grad_out
        for s in reversed(range(sp.L)):
            pre = sp.prefix_fmt.format(s=s)
            xin, xs = (x, x_stride) if s == 0 else (bufs["outs"][s - 1], sp.fn)
            g_sub = gy                                  # grad wrt this sub-net's output (needed again for the skip path)
            for l in reversed(range(sp.n_layers)):
                last = l == sp.n_layers - 1
                cout = sp.out_dim(s) if last else HID
                gx = bufs["g32"][l & 1]
                w_off, b_off = self.table[pre + f"convs.{l}.lins.0.weight"][0], self.table[pre + f"convs.{l}.bias"][0]
                common = (g, _lib.ptr(bufs["acts"][s, l]), self._p(flat, pre + f"convs.{l}.lins.0.weight"), cout, sp.K,
                          0 if last else 1, sp.p_drop, None if last else _lib.ptr(bufs["bits"][s, l]),
                          _lib.ptr(gy), _lib.ptr(gx), pp(pre + f"convs.{l}.lins.0.weight"), pstride, b_off - w_off)
                if use_tc2 and GW_IMPL == "tc":
                    _lib.check(lib.dss2_tag_bwd_tc2(*common, _lib.ptr(bufs["lvl"]), bufs["lvl"].numel() * 4, st), "dss2_tag_bwd_tc2")
                elif use_tc2:
                    (_, xl, wl, _, _, actl, _, bitsl, gyl, gxl, partl, _, boff) = common
                    ws, nws = _lib.ptr(bufs["lvl"]), bufs["lvl"].numel() * 4
                    _lib.check(lib.dss2_tag_bwd_tc2_gx(g, wl, cout, sp.K, actl, sp.p_drop, bitsl, gyl, gxl, ws, nws, st), "dss2_tag_bwd_tc2_gx")
                    _lib.check(lib.dss2_tag_gw_ffma(graph.num_nodes, xl, cout, sp.K, actl, sp.p_drop, bitsl, gyl, partl, pstride, boff,
                                                    ws, nws, st), "dss2_tag_gw_ffma")
                else:
                    _lib.check(lib.dss2_tag_bwd(*common, st), "dss2_tag_bwd")
                gy = gx
            need_gx = s > 0
            gprev = bufs["gsub"][s & 1] if need_gx else None
            skip_grad = g_sub if (sp.skip[s] and need_gx) else None
            if slots:
                _lib.check(lib.dss2_edgeagg_bwd_slot(g, _lib.ptr(xin), xs, sp.fn, _lib.ptr(ea), ea_stride, sp.fe, s, _lib.ptr(gy), _lib.ptr(skip_grad),
                                                     sp.fn if skip_grad is not None else 0, _lib.ptr(gprev), pp(pre + "edge_aggr.edge_aggr.0.weight"),
                                                     pstride, st), "dss2_edgeagg_bwd_slot")
            else:
                _lib.check(lib.dss2_edgeagg_bwd(g, _lib.ptr(xin), xs, sp.fn, _lib.ptr(ea), ea_stride, sp.fe,
                                                *[self._p(flat, n) for n in self._ea_names(s)],
                                                _lib.ptr(gy), _lib.ptr(skip_grad), sp.fn if skip_grad is not None else 0,
                                                _lib.ptr(gprev), pp(pre + "edge_aggr.edge_aggr.0.weight"), pstride, st), "dss2_edgeagg_bwd")
            gy = gprev
        _lib.check(lib.dss2_reduce_partials(_lib.ptr(part), pstride, self.num_partials, self.flat_size, _lib.ptr(flat_grad),
                                            1 if accumulate else 0, st), "dss2_reduce_partials")
        return flat_grad

    def _subnet_range(self, s):
        """[lo, hi) of sub-net s in the flat parameter buffer (the layout is ordered by sub-net)."""
        sp = self.spec
        lo = min(off for name, (off, _) in self.table.items() if name.startswith(sp.prefix_fmt.format(s=s)))
        if s + 1 < sp.L:
            hi = min(off for name, (off, _) in self.table.items() if name.startswith(sp.prefix_fmt.format(s=s + 1)))
        else:
            hi = self.flat_size
        return (0 if s == 0 else lo), hi

    def _backward_pipelined(self, graph, x, x_stride, ea, ea_stride, flat, bufs, grad_out, flat_grad, accumulate, ea_uploaded, rng_state,
                            bucket_hook=None):
        """Same arithmetic as backward(), scheduled on two streams.  The backward-to-input launches of a sub-net form a per-tile chain on
        the current stream (layer l-1 needs only the same tile of layer l's output: dss2_tag_bwd_tc2_gx_chain); the weight-gradient pass
        of each layer needs that layer's whole launch (its spilled hop levels), so it runs behind an event on a second stream and fills
        the SMs the chain leaves idle.  Every layer keeps its own input gradient and level workspace until its pass has run; the streams
        join before the next sub-net reuses them.  Each kernel still writes only its own columns of the per-CTA partials, and the
        partial reduction of a sub-net's columns (+ bucket_hook: its all-reduce) runs on the second stream under the next sub-net."""
        sp, lib = self.spec, self.lib
        g = graph.ref
        main = torch.cuda.current_stream()
        if getattr(self, "_side", None) is None or self._side.device != main.device:
            self._side = torch.cuda.Stream(device=main.device)
        side = self._side
        st, st2 = ctypes.c_void_p(main.cuda_stream), ctypes.c_void_p(side.cuda_stream)
        slots = self.ea_slots(graph, x_stride, ea_stride)
        if slots and not ea_uploaded:
            self.ea_upload(flat)
        part, pstride = bufs["partials"], self.flat_size

        def pp(name):
            return ctypes.c_void_p(part.data_ptr() + 4 * self.table[name][0])

        G, LV, marks = bufs["gchain"], bufs["lvls"], bufs["marks_b"]
        nws = LV[0].numel() * 4
        gy = grad_out
        ev_gw = None
        for s in reversed(range(sp.L)):
            pre = sp.prefix_fmt.format(s=s)
            xin, xs = (x, x_stride) if s == 0 else (bufs["outs"][s - 1], sp.fn)
            g_sub = gy
            if ev_gw is not None:
                main.wait_event(ev_gw)      # the previous sub-net's weight-gradient passes have read G / LV / g_sub
            for l in reversed(range(sp.n_layers)):
                last = l == sp.n_layers - 1
                cout = sp.out_dim(s) if last else HID
                act = 0 if last else 1
                bits = None if last else _lib.ptr(bufs["bits"][s, l])
                w_off, b_off = self.table[pre + f"convs.{l}.lins.0.weight"][0], self.table[pre + f"convs.{l}.bias"][0]
                _lib.check(lib.dss2_tag_bwd_tc2_gx_chain(g, self._p(flat, pre + f"convs.{l}.lins.0.weight"), cout, sp.K, act, sp.p_drop, bits,
                                                         _lib.ptr(gy), _lib.ptr(G[l]), _lib.ptr(LV[l]), nws, _lib.ptr(rng_state),
                                                         _lib.ptr(marks[s, l]) if l > 0 else None, None if last else _lib.ptr(marks[s, l + 1]), st),
                           "dss2_tag_bwd_tc2_gx_chain")
                ev = torch.cuda.Event()
                ev.record(main)
                side.wait_event(ev)
                _lib.check(lib.dss2_tag_bwd_tc2_gw(graph.num_nodes, _lib.ptr(bufs["acts"][s, l]), cout, sp.K, act, sp.p_drop, bits, _lib.ptr(gy),
                                                   pp(pre + f"convs.{l}.lins.0.weight"), pstride, b_off - w_off, _lib.ptr(LV[l]), nws, st2),
                           "dss2_tag_bwd_tc2_gw")
                gy = G[l]
            need_gx = s > 0
            gprev = bufs["gsub"][s & 1] if need_gx else None
            skip_grad = g_sub if (sp.skip[s] and need_gx) else None
            if slots:
                _lib.check(lib.dss2_edgeagg_bwd_slot(g, _lib.ptr(xin), xs, sp.fn, _lib.ptr(ea), ea_stride, sp.fe, s, _lib.ptr(gy), _lib.ptr(skip_grad),
                                                     sp.fn if skip_grad is not None else 0, _lib.ptr(gprev), pp(pre + "edge_aggr.edge_aggr.0.weight"),
                                                     pstride, st), "dss2_edgeagg_bwd_slot")
            else:
                _lib.check(lib.dss2_edgeagg_bwd(g, _lib.ptr(xin), xs, sp.fn, _lib.ptr(ea), ea_stride, sp.fe,
                                                *[self._p(flat, n) for n in self._ea_names(s)],
                                                _lib.ptr(gy), _lib.ptr(skip_grad), sp.fn if skip_grad is not None else 0,
                                                _lib.ptr(gprev), pp(pre + "edge_aggr.edge_aggr.0.weight"), pstride, st), "dss2_edgeagg_bwd")
            gy = gprev
            ev_gw = torch.cuda.Event()
            ev_gw.record(side)
            # this sub-net's columns are final once its EdgeAggregation backward (this stream) and weight-gradient passes (second stream) are
            ev = torch.cuda.Event()
            ev.record(main)
            side.wait_event(ev)
            lo, hi = self._subnet_range(s)
            _lib.check(lib.dss2_reduce_partials(ctypes.c_void_p(part.data_ptr() + 4 * lo), pstride, self.num_partials, hi - lo,
                                                ctypes.c_void_p(flat_grad.data_ptr() + 4 * lo), 1 if accumulate else 0, st2), "dss2_reduce_partials")
            if bucket_hook is not None:
                with torch.cuda.stream(side):
                    bucket_hook(lo, hi)
        main.wait_stream(side)
        self.bucketed = bucket_hook is not None
        return flat_grad


# ---------------------------------------------------------------------------------------------------
# flat parameter packing for nn.Modules
# ---------------------------------------------------------------------------------------------------
class ParamPack:
    """Keeps a module's parameters in ONE flat CUDA buffer laid out by PFNSpec.layout().  CUDA parameters
    are re-pointed into the buffer (their `.data` become views, so optimizers keep working and no copy is
    needed per step); CPU parameters (unmodified dss2_run.py never moves the model) are staged every call."""

    def __init__(self, spec):
        self.spec = spec
        self.table, self.flat_size = spec.layout()
        self.flat = None

    def gather(self, named_params):
        """named_params: dict name -> Parameter.  Returns the flat CUDA buffer holding their current values."""
        first = next(iter(named_params.values()))
        if first.device.type == "cuda":
            if self.flat is None or self.flat.device != first.device or not self._is_packed(named_params):
                flat = torch.zeros(self.flat_size, dtype=torch.float32, device=first.device)
                with torch.no_grad():
                    for name, p in named_params.items():
                        off, n = self.table[name]
                        view = flat[off:off + n].view(p.shape)
                        view.copy_(p.data)
                        p.data = view
                self.flat = flat
            return self.flat
        # CPU parameters: one host staging buffer in the layout's order + one H2D copy
        host = torch.zeros(self.flat_size, dtype=torch.float32)
        for name, p in named_params.items():
            off, n = self.table[name]
            host[off:off + n] = p.data.reshape(-1).float()
        return host.cuda(non_blocking=True)

    def _is_packed(self, named_params):
        base = self.flat.data_ptr()
        for name, p in named_params.items():
            if p.data_ptr() != base + 4 * self.table[name][0]:
                return False
        return True

    def scatter_grads(self, flat_grad, named_params):
        """Per-parameter gradient views of a flat gradient (moved to the parameter's device)."""
        first = next(iter(named_params.values()))
        if first.device.type != "cuda":
            flat_grad = flat_grad.cpu()
        out = []
        for name, p in named_params.items():
            off, n = self.table[name]
            out.append(flat_grad[off:off + n].view(p.shape))
        return out


# ---------------------------------------------------------------------------------------------------
# helpers for device-following inputs
# ---------------------------------------------------------------------------------------------------
def require_cuda():
    _lib.load(require_cuda=True)


def stage_rows(t):
    """CUDA fp32 tensor + row stride for a 2-D (possibly column-sliced) view; copies only if needed."""
    if t.dtype != torch.float32:
        t = t.float()
    if t.device.type != "cuda":
        t = t.cuda(non_blocking=True)
    if t.dim() != 2 or (t.size(1) > 1 and t.stride(1) != 1) or t.stride(0) < t.size(1):
        t = t.contiguous()
    return t, (t.stride(0) if t.size(0) > 1 else max(t.stride(0), t.size(1)))


def resolve_graph(edge_index, num_nodes):
    """BatchGraph for `edge_index` (CPU or CUDA).  Cached on the tensor object, keyed by its version."""
    cached = getattr(edge_index, "_dss2_graph", None)
    if (cached is not None and cached.num_nodes == num_nodes and getattr(edge_index, "_dss2_graph_version", None) == edge_index._version
            and cached.tile_cap <= tile_cap() and cached.hop_keys == _lib.hop_keys_default()):
        return cached
    ei = edge_index if edge_index.device.type == "cuda" else edge_index.cuda(non_blocking=True)
    g = BatchGraph(ei.long(), num_nodes, ptr=getattr(edge_index, "_dss2_ptr", None), tile_cap=tile_cap())
    try:
        edge_index._dss2_graph = g
        edge_index._dss2_graph_version = edge_index._version
    except AttributeError:
        pass
    return g


# ---------------------------------------------------------------------------------------------------
# autograd bridge for whole models
# ---------------------------------------------------------------------------------------------------
class _PFNFunction(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, edge_attr, edge_index, runner, pack, names, masks, rng_state, *params):
        require_cuda()
        out_device = x.device
        named = dict(zip(names, params))
        xg, xs = stage_rows(x)
        eag, eas = stage_rows(edge_attr)
        graph = resolve_graph(edge_index, xg.size(0))
        with torch.cuda.device(xg.device):
            flat = pack.gather(named)
            # inside Function.forward grad mode is always off: whether a backward can follow is what needs_input_grad says
            # (False under torch.no_grad(), e.g. the script's validation loop: no gradient workspaces are allocated then)
            need_grad = any(ctx.needs_input_grad[8:])
            bufs = runner.alloc(xg.size(0), xg.device, need_grad=need_grad)
            if masks is not None:
                mode = 2
                masks = [[m.to(device=xg.device, dtype=torch.uint8).contiguous() for m in sub] for sub in masks]
            else:
                mode = 1 if runner.spec.p_drop > 0 else 0
            if mode == 1 and rng_state is None:
                rng_state = fresh_rng_state(xg.device)
            out = runner.forward(graph, xg, xs, eag, eas, flat, bufs, drop_mode=mode, rng_state=rng_state, masks=masks)
        if getattr(runner, "keep_last_bufs", False):     # tests read the sign words of the last forward
            runner.last_bufs = bufs
        ctx.runner, ctx.pack, ctx.names, ctx.graph = runner, pack, names, graph
        ctx.saved = (xg, xs, eag, eas, flat, bufs, masks, rng_state)
        ctx.param_devices_cpu = params[0].device.type != "cuda"
        ctx.params = params
        result = out.clone()      # bufs are owned by this call; hand out an independent tensor
        return result if out_device.type == "cuda" else result.to(out_device)

    @staticmethod
    def backward(ctx, grad_out):
        xg, xs, eag, eas, flat, bufs, masks, rng_state = ctx.saved
        runner = ctx.runner
        go = grad_out.to(device=xg.device, dtype=torch.float32).contiguous()
        with torch.cuda.device(xg.device):
            flat_grad = torch.empty(runner.flat_size, dtype=torch.float32, device=xg.device)
            runner.backward(ctx.graph, xg, xs, eag, eas, flat, bufs, go, flat_grad)
        named = dict(zip(ctx.names, ctx.params))
        grads = ctx.pack.scatter_grads(flat_grad, named)
        return (None, None, None, None, None, None, None, None, *grads)


def fresh_rng_state(device):
    """{seed, step} for the in-kernel Philox dropout, drawn from torch's global generator so that
    torch.manual_seed() makes runs repeatable."""
    seed = int(torch.randint(0, 2 ** 62, (1,)).item())
    return torch.tensor([seed, 0], dtype=torch.int64, device=device)


def pfn_apply(runner, pack, named_params, x, edge_index, edge_attr, masks=None, rng_state=None):
    if torch.is_grad_enabled() and (x.requires_grad or edge_attr.requires_grad):
        raise _lib.Dss2Error("MPN / SkipMPN / PFN / SkipPFN: gradients are computed w.r.t. the parameters only; x / edge_attr with "
                             "requires_grad=True would silently get none (the reference's data tensors never require grad, "
                             "dss2_run.py:138) - detach them first")
    names = tuple(named_params.keys())
    return _PFNFunction.apply(x, edge_attr, edge_index, runner, pack, names, masks, rng_state, *named_params.values())


# ---------------------------------------------------------------------------------------------------
# stand-alone layers (EdgeAggregation / TAGConv modules used on their own)
# ---------------------------------------------------------------------------------------------------
class _EdgeAggFunction(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, edge_attr, edge_index, w1, b1, w2, b2):
        require_cuda()
        lib = _lib.load()
        dev_out = x.device
        xg, xs = stage_rows(x)
        eag, eas = stage_rows(edge_attr)
        graph = resolve_graph(edge_index, xg.size(0))
        ws = [t.detach().to(device=xg.device, dtype=torch.float32).contiguous() for t in (w1, b1, w2, b2)]
        if ws[2].size(0) != HID or ws[0].size(0) != HID:
            raise _lib.Dss2Error(f"EdgeAggregation kernels need dim_hid == dim_out == {HID}")
        fn, fe = xg.size(1), eag.size(1)
        out = torch.empty(xg.size(0), HID, dtype=torch.float32, device=xg.device)
        with torch.cuda.device(xg.device):
            _lib.check(lib.dss2_edgeagg_fwd(graph.ref, _lib.ptr(xg), xs, fn, _lib.ptr(eag), eas, fe, *[_lib.ptr(t) for t in ws],
                                            _lib.ptr(out), _lib.stream()), "dss2_edgeagg_fwd")
        ctx.saved = (xg, xs, eag, eas, graph, ws, fn, fe)
        ctx.in_devices = (x.device, w1.device)
        ctx.need_x = x.requires_grad
        return out if dev_out.type == "cuda" else out.to(dev_out)

    @staticmethod
    def backward(ctx, grad_out):
        lib = _lib.load()
        xg, xs, eag, eas, graph, ws, fn, fe = ctx.saved
        go = grad_out.to(device=xg.device, dtype=torch.float32).contiguous()
        npart = lib.dss2_num_partials()
        count = HID * (2 * fn + fe) + HID + HID * HID + HID
        part = torch.empty(npart, count, dtype=torch.float32, device=xg.device)
        gx = torch.empty(xg.size(0), fn, dtype=torch.float32, device=xg.device)
        flat = torch.empty(count, dtype=torch.float32, device=xg.device)
        with torch.cuda.device(xg.device):
            _lib.check(lib.dss2_edgeagg_bwd(graph.ref, _lib.ptr(xg), xs, fn, _lib.ptr(eag), eas, fe, *[_lib.ptr(t) for t in ws],
                                            _lib.ptr(go), None, 0, _lib.ptr(gx), _lib.ptr(part), count, _lib.stream()), "dss2_edgeagg_bwd")
            _lib.check(lib.dss2_reduce_partials(_lib.ptr(part), count, npart, count, _lib.ptr(flat), 0, _lib.stream()), "dss2_reduce_partials")
        ld = 2 * fn + fe
        sizes = [HID * ld, HID, HID * HID, HID]
        gw1, gb1, gw2, gb2 = torch.split(flat, sizes)
        xdev, wdev = ctx.in_devices
        grads = [gw1.view(HID, ld), gb1, gw2.view(HID, HID), gb2]
        grads = [t.to(wdev) for t in grads]
        return (gx.to(xdev) if ctx.need_x else None, None, None, *grads)


class _TagFunction(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, edge_index, bias, K, *weights):
        require_cuda()
        lib = _lib.load()
        dev_out = x.device
        xg, xs = stage_rows(x)
        if xg.size(1) != HID:
            raise _lib.Dss2Error(f"TAGConv kernels need in_channels == {HID}")
        if xs != HID:
            xg = xg.contiguous()
        graph = resolve_graph(edge_index, xg.size(0))
        w = torch.stack([t.detach().to(device=xg.device, dtype=torch.float32) for t in weights]).contiguous()
        b = bias.detach().to(device=xg.device, dtype=torch.float32).contiguous()
        cout = w.size(1)
        y = torch.empty(xg.size(0), cout, dtype=torch.float32, device=xg.device)
        with torch.cuda.device(xg.device):
            _lib.check(lib.dss2_tag_fwd(graph.ref, _lib.ptr(xg), _lib.ptr(w), _lib.ptr(b), cout, K, 0, 0.0, 0, None, 0, None, None, 0,
                                        _lib.ptr(y), None, _lib.stream()), "dss2_tag_fwd")
        ctx.saved = (xg, graph, w, cout, K)
        ctx.in_devices = (x.device, bias.device)
        return y if dev_out.type == "cuda" else y.to(dev_out)

    @staticmethod
    def backward(ctx, grad_y):
        lib = _lib.load()
        xg, graph, w, cout, K = ctx.saved
        gy = grad_y.to(device=xg.device, dtype=torch.float32).contiguous()
        npart = lib.dss2_num_partials()
        nw = (K + 1) * cout * HID
        count = nw + _align4(cout)
        part = torch.empty(npart, count, dtype=torch.float32, device=xg.device)
        flat = torch.empty(count, dtype=torch.float32, device=xg.device)
        gx = torch.empty(xg.size(0), HID, dtype=torch.float32, device=xg.device)
        with torch.cuda.device(xg.device):
            _lib.check(lib.dss2_tag_bwd(graph.ref, _lib.ptr(xg), _lib.ptr(w), cout, K, 0, 0.0, None, _lib.ptr(gy), _lib.ptr(gx),
                                        _lib.ptr(part), count, nw, _lib.stream()), "dss2_tag_bwd")
            _lib.check(lib.dss2_reduce_partials(_lib.ptr(part), count, npart, nw + cout, _lib.ptr(flat), 0, _lib.stream()), "dss2_reduce_partials")
        xdev, wdev = ctx.in_devices
        gw = flat[:nw].view(K + 1, cout, HID).to(wdev)
        gb = flat[nw:nw + cout].to(wdev)
        return (gx.to(xdev), None, gb, None, *[gw[k] for k in range(K + 1)])


def edge_aggregation(x, edge_index, edge_attr, w1, b1, w2, b2):
    return _EdgeAggFunction.apply(x, edge_attr, edge_index, w1, b1, w2, b2)


def tag_conv(x, edge_index, weights, bias):
    return _TagFunction.apply(x, edge_index, bias, len(weights) - 1, *weights)
