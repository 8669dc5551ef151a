"""ctypes binding of libdss2_b200.so (the C ABI declared in include/dss2_b200.h).

There is no CPU fallback: if the library is missing, or no CUDA device is present, every compute
entry point raises.  The library is built in-tree by `__graft_entry__.build()` / `make -C csrc`.
"""
import ctypes
import os
from ctypes import POINTER, Structure, c_char_p, c_float, c_int, c_int32, c_int64, c_size_t, c_uint32, c_void_p

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(os.path.dirname(_HERE), "csrc", "libdss2_b200.so")

HID = 32
TILE_CAP = 256
# swizzle-key policies of dss2_graph_build (DSS2_HOP_KEYS_* in the header)
HOP_KEYS = {"identity": 0, "color": 1}
ELL_DEG_MASK = 0x1FFFF
ELL_KEY_SHIFT = 17


def hop_keys_default():
    """Policy for graphs built without an explicit one: $DSS2_HOP_KEYS (identity | color), read at every build; color when unset."""
    name = os.environ.get("DSS2_HOP_KEYS", "color")
    if name not in HOP_KEYS:
        raise ValueError(f"DSS2_HOP_KEYS={name!r}: expected one of {sorted(HOP_KEYS)}")
    return name


class GraphStruct(Structure):
    """Mirror of `dss2_graph_t`."""
    _fields_ = [
        ("num_nodes", c_int64), ("num_edges", c_int64), ("nnz", c_int64),
        ("num_graphs", c_int32), ("undirected", c_int32), ("graphs_per_tile", c_int32), ("num_tiles", c_int32),
        ("max_tile_nodes", c_int32), ("max_tile_nnz", c_int32), ("max_tile_edges", c_int32), ("hop_keys", c_int32),
        ("edge_index", c_void_p), ("ptr", c_void_p), ("eptr", c_void_p), ("rowptr", c_void_p), ("col", c_void_p),
        ("eid", c_void_p), ("dis", c_void_p), ("w", c_void_p), ("ell_w", c_void_p), ("ell_ci", c_void_p),
        ("scratch", c_void_p), ("scratch_bytes", c_size_t), ("hop_key", c_void_p),
    ]


class AttnDrop(Structure):
    """Mirror of `dss2_attn_drop_t` (attention dropout of one GATv2Conv / FAConv layer and head)."""
    _fields_ = [("p", c_float), ("mode", c_int), ("rng_state", c_void_p), ("layer_uid", c_uint32), ("head", c_uint32), ("mask", c_void_p)]


class PfTopology(Structure):
    """Mirror of `dss2_pf_topology_t` (one power-flow topology, dss2.powerflow)."""
    _fields_ = [
        ("num_buses", c_int32), ("slack", c_int32), ("num_pq", c_int32), ("num_blocks", c_int32),
        ("num_updates", c_int32), ("num_edges", c_int32), ("v_lv", ctypes.c_double),
        ("y_ptr", c_void_p), ("y_col", c_void_p), ("y_gb", c_void_p), ("bus", c_void_p), ("blk_ptr", c_void_p),
        ("blk_col", c_void_p), ("blk_y", c_void_p), ("diag", c_void_p), ("upd_ptr", c_void_p), ("upd", c_void_p),
        ("edge_ft", c_void_p), ("edge_gb", c_void_p),
    ]


class SeTopology(Structure):
    """Mirror of `dss2_se_topology_t` (one state-estimation topology, dss2.estimation)."""
    _fields_ = [
        ("num_buses", c_int32), ("num_edges", c_int32), ("slack", c_int32), ("num_blocks", c_int32), ("num_updates", c_int32),
        ("num_pairs", c_int32), ("max_support", c_int32),
        ("edge_ft", c_void_p), ("inc_ptr", c_void_p), ("inc", c_void_p), ("sup_ptr", c_void_p), ("sup_pos", c_void_p),
        ("pair_ptr", c_void_p), ("pair_blk", c_void_p), ("edge_blk", c_void_p), ("bus", c_void_p), ("blk_ptr", c_void_p),
        ("blk_col", c_void_p), ("diag", c_void_p), ("upd_ptr", c_void_p), ("upd", c_void_p),
    ]


_P = c_void_p
_G = POINTER(GraphStruct)
_D = POINTER(AttnDrop)
_T = POINTER(PfTopology)
_ST = POINTER(SeTopology)
_SIGNATURES = {
    "dss2_last_error": (c_char_p, []),
    "dss2_version": (c_int, []),
    "dss2_launch_count": (c_int64, []),
    "dss2_graph_workspace_bytes": (c_size_t, [c_int64, c_int64, c_int32]),
    "dss2_generic_scratch_bytes": (c_size_t, [c_int64]),
    "dss2_graph_build": (c_int, [_G, _P, c_int64, c_int64, _P, c_int32, c_int, c_int, c_int, _P, c_size_t, _P]),
    "dss2_hop_keys_host": (c_int, [_P, _P, c_int32, c_int, _P]),
    "dss2_pack_batch": (c_int, [_P, _P, _P, _P, c_int64, _P, _P, _P, c_int32, _P, _P, c_int64, _P, _P, _P, _P, _P, _P, _P]),
    "dss2_col_minmax": (c_int, [_P, c_int64, c_int, c_int64, _P, _P]),
    "dss2_edgeagg_fwd": (c_int, [_G, _P, c_int64, c_int, _P, c_int64, c_int, _P, _P, _P, _P, _P, _P]),
    "dss2_edgeagg_bwd": (c_int, [_G, _P, c_int64, c_int, _P, c_int64, c_int, _P, _P, _P, _P, _P, _P, c_int64, _P, _P, c_int64, _P]),
    "dss2_tag_fwd": (c_int, [_G, _P, _P, _P, c_int, c_int, c_int, c_float, c_int, _P, c_uint32, _P, _P, c_int64, _P, _P, _P]),
    "dss2_tag_tc2_supported": (c_int, [_G, c_int]),
    "dss2_tag_fwd_tc2": (c_int, [_G, _P, _P, _P, c_int, c_int, c_int, c_float, c_int, _P, c_uint32, _P, _P, c_int64, _P, _P, _P]),
    "dss2_tag_fwd_tc2_chain": (c_int, [_G, _P, _P, _P, c_int, c_int, c_int, c_float, c_int, _P, c_uint32, _P, _P, c_int64, _P, _P, _P, _P, _P]),
    "dss2_tag_bwd_tc2_workspace_bytes": (c_size_t, [c_int64, c_int]),
    "dss2_tag_bwd_tc2": (c_int, [_G, _P, _P, c_int, c_int, c_int, c_float, _P, _P, _P, _P, c_int64, c_int64, _P, c_size_t, _P]),
    "dss2_tag_bwd_tc2_gx": (c_int, [_G, _P, c_int, c_int, c_int, c_float, _P, _P, _P, _P, c_size_t, _P]),
    "dss2_tag_bwd_tc2_gx_chain": (c_int, [_G, _P, c_int, c_int, c_int, c_float, _P, _P, _P, _P, c_size_t, _P, _P, _P, _P]),
    "dss2_tag_bwd_tc2_gw": (c_int, [c_int64, _P, c_int, c_int, c_int, c_float, _P, _P, _P, c_int64, c_int64, _P, c_size_t, _P]),
    "dss2_tag_gw_ffma": (c_int, [c_int64, _P, c_int, c_int, c_int, c_float, _P, _P, _P, c_int64, c_int64, _P, c_size_t, _P]),
    "dss2_tc_selftest": (c_int, [_P, _P, _P, _P]),
    "dss2_tc_selftest_mn": (c_int, [_P, _P, _P, _P]),
    "dss2_tag_bwd": (c_int, [_G, _P, _P, c_int, c_int, c_int, c_float, _P, _P, _P, _P, c_int64, c_int64, _P]),
    "dss2_num_partials": (c_int, []),
    "dss2_reduce_partials": (c_int, [_P, c_int64, c_int, c_int64, _P, c_int, _P]),
    "dss2_wls_workspace_bytes": (c_size_t, [_G]),
    "dss2_wls_fwd_bwd": (c_int, [_G, _P, c_int64, _P, c_int64, _P, _P, c_float, c_float, c_float, c_float, _P, c_int, _P, _P, _P,
                                 _P, c_size_t, _P]),
    "dss2_wls_pass": (c_int, [c_int, _G, _P, c_int64, _P, c_int64, _P, _P, c_float, c_float, c_float, c_float, _P, c_int, _P, _P, _P,
                                 _P, c_size_t, _P]),
    "dss2_wls_sums": (ctypes.c_void_p, [_P]),
    "dss2_edgeagg_slots_ok": (c_int, [_G, c_int64, c_int64, c_int]),
    "dss2_edgeagg_upload": (c_int, [c_int, c_int, _P, _P, _P, _P, c_int, c_int, _P]),
    "dss2_edgeagg_fwd_slot": (c_int, [_G, _P, c_int64, c_int, _P, c_int64, c_int, c_int, _P, _P]),
    "dss2_edgeagg_bwd_slot": (c_int, [_G, _P, c_int64, c_int, _P, c_int64, c_int, c_int, _P, _P, c_int64, _P, _P, c_int64, _P]),
    "dss2_build_scenarios_workspace_bytes": (c_size_t, []),
    "dss2_build_scenarios": (c_int, [_P, _P, _P, _P, _P, _P, _P, c_int64, c_int, c_int, _P, _P, _P, _P, c_size_t, _P]),
    "dss2_load_profiles": (c_int, [_P, _P, _P, _P, _P, c_int, c_int, c_int, ctypes.c_double, _P, _P, _P]),
    "dss2_mc_sample": (c_int, [_P, _P, c_int64, c_int, c_int, _P, _P, _P]),
    "dss2_powerflow_workspace_bytes": (c_size_t, [_T, c_int64]),
    "dss2_powerflow": (c_int, [_T, c_int64, _P, _P, _P, ctypes.c_double, c_int, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, c_size_t,
                               c_int64, _P]),
    "dss2_wls_estimate_workspace_bytes": (c_size_t, [_ST, c_int64]),
    "dss2_wls_estimate": (c_int, [_ST, c_int64, _P, c_int64, _P, c_int64, _P, ctypes.c_double, ctypes.c_double, ctypes.c_double,
                                  ctypes.c_double, c_int, _P, _P, _P, _P, _P, _P, _P, _P, c_size_t, c_int64, _P]),
    "dss2_pflow": (c_int, [_P, c_int64, _P, c_int64, _P, c_int64, _P, _P, _P]),
    "dss2_pflow_ex": (c_int, [_P, c_int64, _P, c_int64, _P, c_int64, _P, c_int, _P, _P]),
    "dss2_pflow_bwd": (c_int, [_G, _P, c_int64, _P, c_int64, _P, c_int, _P, _P, _P]),
    "dss2_pflow_est": (c_int, [_P, c_int64, _P, c_int64, _P, c_int64, c_float, c_float, _P, c_int64, _P, _P, _P]),
    "dss2_adamax_step": (c_int, [_P, _P, _P, _P, c_int64, c_float, c_float, c_float, c_float, c_float, _P, c_int, _P]),
    "dss2_step_advance": (c_int, [_P, _P]),
    "dss2_eval_workspace_bytes": (c_size_t, []),
    "dss2_eval_metrics": (c_int, [_P, c_int64, c_int64, _P, c_int64, _P, c_int64, _P, c_int64, _P, c_int64, c_float, c_float, _P, _P, _P,
                                  c_size_t, _P]),
    "dss2_eval_metrics_acc": (c_int, [_P, c_int64, c_int64, _P, c_int64, _P, c_int64, _P, c_int64, _P, c_int64, c_float, c_float, _P, _P,
                                      _P, c_size_t, _P]),
    "dss2_gat_ws_bytes": (c_size_t, [c_int64]),
    "dss2_gat_fwd": (c_int, [_G, _P, c_int64, _P, c_int64, c_int, _P, _P, _P, _P, _P, _P, _P, c_float, c_int, c_float, _P, _P]),
    "dss2_gat_bwd": (c_int, [_G, _P, c_int64, _P, c_int64, c_int, _P, _P, _P, _P, _P, _P, _P, c_float, c_int, c_float,
                             _P, _P, _P, _P, c_size_t, _P, c_int64, _P]),
    "dss2_gat_upload": (c_int, [c_int, c_int, _P, _P, _P, _P, _P, _P, _P, c_int, _P]),
    "dss2_gat_fwd_slot": (c_int, [_G, _P, c_int64, _P, c_int64, c_int, c_int, c_float, c_int, c_float, _P, _P]),
    "dss2_gat_bwd_slot": (c_int, [_G, _P, c_int64, _P, c_int64, c_int, c_int, c_float, c_int, c_float, _P, _P, _P, _P, c_size_t, _P,
                                  c_int64, _P, _P]),
    "dss2_gat_bwd_ex": (c_int, [_G, _P, c_int64, _P, c_int64, c_int, _P, _P, _P, _P, _P, _P, _P, c_float, c_int, c_float,
                                _P, _P, _P, _P, c_size_t, _P, c_int64, _P, _P]),
    "dss2_gine_ws_bytes": (c_size_t, [c_int64]),
    "dss2_gine_fwd": (c_int, [_G, _P, c_int64, _P, c_int64, c_int, _P, _P, _P, _P, c_float, c_int, c_float, _P, _P]),
    "dss2_gine_fwd_ex": (c_int, [_G, _P, c_int64, _P, c_int64, c_int, _P, _P, _P, _P, c_float, _P, c_int, c_float, _P, _P]),
    "dss2_gine_bwd_ex": (c_int, [_G, _P, c_int64, _P, c_int64, c_int, _P, _P, _P, _P, c_float, _P, c_int, c_float, _P, _P, _P, _P, c_size_t,
                                 _P, _P, c_int64, _P]),
    "dss2_gine_bwd": (c_int, [_G, _P, c_int64, _P, c_int64, c_int, _P, _P, _P, _P, c_float, c_int, c_float, _P, _P, _P, _P, c_size_t,
                              _P, _P, c_int64, _P]),
    "dss2_gcn_dinv": (c_int, [_G, c_int, _P, _P]),
    "dss2_gcn_prop8": (c_int, [_G, _P, c_int, c_int, _P, c_int64, c_float, _P, c_int64, c_float, _P, _P]),
    "dss2_lin8_fwd": (c_int, [c_int64, c_int, c_int, _P, _P, _P, _P, c_int, c_float, _P, _P]),
    "dss2_lin8_bwd": (c_int, [c_int64, c_int, c_int, _P, _P, _P, c_int, c_float, _P, _P, _P, _P, _P, c_float, _P, c_int64, c_int64, _P]),
    "dss2_fa_fwd": (c_int, [_G, _P, c_int, _P, c_int64, _P, c_int64, _P, _P, c_float, c_int, c_float, _P, _P]),
    "dss2_fa_bwd": (c_int, [_G, _P, c_int, _P, c_int64, _P, _P, c_float, c_int, c_float, _P, _P, _P, _P, _P, c_int64, _P]),
    "dss2_gat_fwd_drop": (c_int, [_G, _P, c_int64, _P, c_int64, c_int, c_int, _P, _P, _P, _P, _P, _P, _P, c_float, c_int, c_float, _D, _P, _P]),
    "dss2_gat_bwd_drop": (c_int, [_G, _P, c_int64, _P, c_int64, c_int, c_int, _P, _P, _P, _P, _P, _P, _P, c_float, c_int, c_float, _D,
                                  _P, _P, _P, _P, c_size_t, _P, c_int64, _P, _P]),
    "dss2_fa_fwd_drop": (c_int, [_G, _P, c_int, _P, c_int64, _P, c_int64, _P, _P, c_float, c_int, c_float, _D, _P, _P]),
    "dss2_fa_bwd_drop": (c_int, [_G, _P, c_int, _P, c_int64, _P, _P, c_float, c_int, c_float, _D, _P, _P, _P, _P, _P, c_int64, _P]),
    "dss2_attn_drop_mask": (c_int, [_D, c_int64, c_int64, _P, _P]),
    "dss2_mlp2_fwd": (c_int, [c_int64, _P, c_int, _P, _P, c_int, _P, _P, c_int, _P, _P, _P]),
    "dss2_mlp2_bwd": (c_int, [c_int64, _P, c_int, _P, c_int, _P, c_int, _P, _P, _P, _P, _P, c_int64, _P]),
    "dss2_mlp2_nh_supported": (c_int, [c_int, c_int, c_int]),
    "dss2_mlp2_bwd_nh": (c_int, [c_int64, _P, c_int, _P, _P, c_int, _P, c_int, _P, _P, _P, c_int64, _P]),
}

_lib = None


class Dss2Error(RuntimeError):
    pass


def exported_symbols():
    """Names the header declares (used by the CPU test that checks the library exports all of them)."""
    return sorted(_SIGNATURES)


def load(require_cuda=True):
    """Load the shared library (once).  Raises if it has not been built - there is no fallback path."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise Dss2Error(f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                            "or `make -C <package>/csrc`. There is no CPU fallback.")
        lib = ctypes.CDLL(LIB_PATH)
        for name, (res, args) in _SIGNATURES.items():
            fn = getattr(lib, name)
            fn.restype = res
            fn.argtypes = args
        _lib = lib
    if require_cuda and not torch.cuda.is_available():
        raise Dss2Error("dss2_b200 needs a CUDA device (sm_100a); there is no CPU fallback for the hot path.")
    return _lib


def check(rc, what):
    if rc != 0:
        raise Dss2Error(f"{what} failed ({rc}): {load(False).dss2_last_error().decode()}")


def ptr(t):
    """Device pointer of a tensor (None -> NULL)."""
    return None if t is None else c_void_p(t.data_ptr())


def attn_drop(p, layer_uid, head=0, rng_state=None, mask=None):
    """`dss2_attn_drop_t *` of one layer and head: the caller's mask (uint8 [Et + Nt]) when given, else the Philox stream of the device
    {seed, step} `rng_state`; None (no dropout) when p == 0 or neither is given."""
    if p == 0.0 or (rng_state is None and mask is None):
        return None
    return ctypes.pointer(AttnDrop(float(p), 2 if mask is not None else 1, None if rng_state is None else rng_state.data_ptr(), layer_uid, head,
                                   None if mask is None else mask.data_ptr()))


def stream():
    return c_void_p(torch.cuda.current_stream().cuda_stream)


def launch_count():
    return int(load(False).dss2_launch_count())
