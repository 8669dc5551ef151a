"""Kernel-private structure of one batch (doubled-graph CSR, degree norm, tiling) and its cache.

The reference rebuilds the undirected edge list in each of the 5 sub-nets (networks.py:236-258, with a
host sync in `is_directed`) and PyG recomputes `gcn_norm` in each of the 40 TAGConv layers.  Here the
structure is built once per batch topology by `dss2_graph_build` and shared by every layer and by the
loss.  Batches produced by `dss2.batching` carry their structure with them (attribute `_dss2_graph` on
the edge_index tensor); foreign tensors get one built on first use.
"""
import ctypes

import numpy as np
import torch

from . import _lib


class BatchGraph:
    """Owns the device workspace behind a `dss2_graph_t`."""

    def __init__(self, edge_index, num_nodes, ptr=None, undirect=-1, tile_cap=_lib.TILE_CAP, hop_keys=None):
        """hop_keys: swizzle-key policy of the layer kernels' shared-memory tiles ("identity" or "color", see
        DSS2_HOP_KEYS_COLOR in dss2_b200.h); None = `_lib.hop_keys_default()`.  Results do not depend on it."""
        lib = _lib.load()
        self.hop_keys = _lib.hop_keys_default() if hop_keys is None else hop_keys
        if self.hop_keys not in _lib.HOP_KEYS:
            raise ValueError(f"hop_keys={self.hop_keys!r}: expected one of {sorted(_lib.HOP_KEYS)}")
        if edge_index.device.type != "cuda":
            raise _lib.Dss2Error("BatchGraph needs CUDA tensors")
        if edge_index.dtype != torch.long or edge_index.dim() != 2 or edge_index.size(0) != 2:
            raise ValueError("edge_index must be int64 [2, E]")
        self.edge_index = edge_index.contiguous()
        self.num_nodes = int(num_nodes)
        self.tile_cap = int(tile_cap)
        self.num_edges = int(edge_index.size(1))
        if ptr is None:
            ptr = discover_segments(self.edge_index, self.num_nodes)
        self.ptr = ptr.to(device=edge_index.device, dtype=torch.long).contiguous()
        self.num_graphs = self.ptr.numel() - 1
        nbytes = lib.dss2_graph_workspace_bytes(self.num_nodes, self.num_edges, self.num_graphs)
        self.ws = torch.zeros(nbytes, dtype=torch.uint8, device=edge_index.device)
        self.c = _lib.GraphStruct()
        with torch.cuda.device(edge_index.device):
            rc = lib.dss2_graph_build(ctypes.byref(self.c), _lib.ptr(self.edge_index), self.num_edges, self.num_nodes,
                                      _lib.ptr(self.ptr), self.num_graphs, undirect, tile_cap, _lib.HOP_KEYS[self.hop_keys],
                                      _lib.ptr(self.ws), nbytes,
                                      _lib.stream())
        _lib.check(rc, "dss2_graph_build")
        self._wls_ws = None
        self.scratch = None
        if self.c.num_tiles == 0:      # a graph exceeds a tile: the large-graph kernels need scratch
            n = lib.dss2_generic_scratch_bytes(self.num_nodes)
            self.scratch = torch.empty(n, dtype=torch.uint8, device=edge_index.device)
            self.c.scratch = self.scratch.data_ptr()
            self.c.scratch_bytes = n

    @property
    def ref(self):
        return ctypes.byref(self.c)

    @property
    def device(self):
        return self.edge_index.device

    def wls_workspace(self):
        if self._wls_ws is None:
            n = _lib.load().dss2_wls_workspace_bytes(self.ref)
            self._wls_ws = torch.zeros(n, dtype=torch.uint8, device=self.device)
        return self._wls_ws

    # views of the kernel-private arrays (tests / debugging)
    def arrays(self):
        def view(addr, n, dtype):
            if n == 0:
                return torch.empty(0, dtype=dtype, device=self.device)
            off = addr - self.ws.data_ptr()
            nbytes = n * torch.empty(0, dtype=dtype).element_size()
            return self.ws[off:off + nbytes].view(dtype)
        c = self.c
        return {
            "rowptr": view(c.rowptr, c.num_nodes + 1, torch.int32), "col": view(c.col, c.nnz, torch.int32),
            "eid": view(c.eid, c.nnz, torch.int32), "dis": view(c.dis, c.num_nodes, torch.float32),
            "eptr": view(c.eptr, c.num_graphs + 1, torch.int64), "w": view(c.w, c.nnz, torch.float32),
            "ell_ci": view(c.ell_ci, 2 * c.num_nodes if c.num_tiles else 0, torch.int32),
            "hop_key": view(c.hop_key, c.num_nodes if c.num_tiles else 0, torch.uint8),
        }


def discover_segments(edge_index, num_nodes):
    """Node offsets of the independent segments of a batch when the caller did not supply `ptr`
    (the reference's model signature carries no batch vector, dss2_run.py:138).  A boundary b is a cut
    iff no edge spans it; plain tensor ops on the device, one host sync for the count."""
    dev = edge_index.device
    if edge_index.numel() == 0 or num_nodes == 0:
        return torch.tensor([0, num_nodes], dtype=torch.long, device=dev)
    lo = torch.minimum(edge_index[0], edge_index[1])
    hi = torch.maximum(edge_index[0], edge_index[1])
    span = torch.zeros(num_nodes + 1, dtype=torch.long, device=dev)
    span.index_add_(0, lo + 1, torch.ones_like(lo))
    span.index_add_(0, hi + 1, -torch.ones_like(hi))
    open_edges = torch.cumsum(span, 0)[:num_nodes]          # edges crossing the boundary before node b
    cuts = torch.nonzero(open_edges == 0).flatten()         # includes b = 0
    return torch.cat([cuts, torch.tensor([num_nodes], dtype=torch.long, device=dev)])


def graph_for(edge_index, num_nodes):
    """The cached BatchGraph attached to `edge_index`, building (and attaching) it if needed."""
    g = getattr(edge_index, "_dss2_graph", None)
    if (g is not None and g.num_nodes == num_nodes and g.edge_index.data_ptr() == edge_index.data_ptr()
            and g.hop_keys == _lib.hop_keys_default()):
        return g
    g = BatchGraph(edge_index, num_nodes)
    try:
        edge_index._dss2_graph = g
    except AttributeError:
        pass
    return g


# ---- host model of the tiling, the ELL view and the swizzle keys of dss2_graph_build (tests, tools/hop_conflicts.py) ----

def host_ell(edge_index, ptr, tile_cap=_lib.TILE_CAP, undirect=True):
    """(ell_ci uint32 [Nt, 2], tile_ptr int64 [num_tiles + 1]) as dss2_graph_build makes them before packing the keys: column 0 =
    4 x 8-bit tile-local sources of a row's first 4 entries in PyG scatter order (padding = the row itself), column 1 = degree.
    None when a graph exceeds `tile_cap`."""
    ei = np.asarray(edge_index, dtype=np.int64)
    ptr = np.asarray(ptr, dtype=np.int64)
    nt, b = int(ptr[-1]), len(ptr) - 1
    seg = int(np.diff(ptr).max())
    if seg == 0 or seg > tile_cap:
        return None
    src, dst = (np.concatenate([ei[0], ei[1]]), np.concatenate([ei[1], ei[0]])) if undirect else (ei[0], ei[1])
    order = np.lexsort((np.arange(dst.size), dst))    # by destination, then by doubled edge id
    src, dst = src[order], dst[order]
    deg = np.bincount(dst, minlength=nt)
    rowptr = np.concatenate([[0], np.cumsum(deg)])
    per = tile_cap // seg
    tile_ptr = ptr[np.r_[np.arange(0, b, per), b]]
    n0 = np.repeat(tile_ptr[:-1], np.diff(tile_ptr))
    rows = np.arange(nt)
    ci = np.zeros((nt, 2), dtype=np.uint32)
    for d in range(4):
        has = deg > d
        col = rows.copy()
        col[has] = src[rowptr[:-1][has] + d]
        ci[:, 0] |= (((col - n0) & 0xff) << (8 * d)).astype(np.uint32)
    ci[:, 1] = np.minimum(deg, _lib.ELL_DEG_MASK)
    return ci, tile_ptr


def host_hop_keys(ell_ci, tile_ptr, policy):
    """The keys (uint8 [Nt]) dss2_graph_build assigns under `policy` ("identity" or "color"), computed by the library on the host."""
    ci = np.ascontiguousarray(ell_ci, dtype=np.uint32)
    tp = np.ascontiguousarray(tile_ptr, dtype=np.int64)
    keys = np.zeros(ci.shape[0], dtype=np.uint8)
    lib = _lib.load(require_cuda=False)
    _lib.check(lib.dss2_hop_keys_host(ci.ctypes.data, tp.ctypes.data, len(tp) - 1, _lib.HOP_KEYS[policy], keys.ctypes.data),
               "dss2_hop_keys_host")
    return keys


def hop_wavefronts(ell_ci, tile_ptr, keys):
    """Shared-memory wavefronts of the layer kernels' 128-bit accesses to the plain level tiles, against the conflict-free count:
    {"gather": (wavefronts, ideal), "store": (wavefronts, ideal)}.  One access phase = 8 consecutive rows of a tile; rows with
    different addresses and equal keys share banks, so a phase takes as many wavefronts as the most frequent key among its
    distinct rows (gathers: the rows' active slot-d sources, one count per slot; stores: the rows themselves)."""
    ci = np.asarray(ell_ci, dtype=np.uint32)
    tile_ptr = np.asarray(tile_ptr, dtype=np.int64)
    keys = np.asarray(keys, dtype=np.int64)
    n0 = np.repeat(tile_ptr[:-1], np.diff(tile_ptr))
    rows = np.arange(ci.shape[0])
    group = np.repeat(np.arange(len(tile_ptr) - 1), np.diff(tile_ptr)) * (_lib.TILE_CAP // 8) + (rows - n0) // 8

    def waves(grp, member):
        u = np.unique(np.stack([grp, member]), axis=1)               # distinct rows per phase
        gk = np.unique(np.stack([u[0], keys[u[1]]]), axis=1, return_counts=True)
        per = np.zeros(int(grp.max()) + 1, dtype=np.int64)
        np.maximum.at(per, gk[0][0], gk[1])
        return int(per.sum()), int(np.count_nonzero(per))

    deg = np.minimum(ci[:, 1] & _lib.ELL_DEG_MASK, 4)
    gg, gm = [], []
    for d in range(4):
        act = deg > d
        gg.append(group[act] * 4 + d)
        gm.append(n0[act] + ((ci[act, 0] >> (8 * d)) & 0xff))
    return {"gather": waves(np.concatenate(gg), np.concatenate(gm)), "store": waves(group, rows)}
