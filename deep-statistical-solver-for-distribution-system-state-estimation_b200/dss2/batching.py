"""(a) Batching: PyG `DataLoader` / `Batch.from_data_list` replacement backed by the CUDA packer.

`pack_batch(store, ids)` gathers the chosen scenarios of a device-resident ScenarioStore into PyG's
disjoint-union layout (bit-exact with PyG: x / edge_attr / y concatenated graph-major, edge_index offset by
the running node count, `batch`, `ptr`) with `dss2_pack_batch`, and attaches the kernel-private graph
structure so that the model and the loss do not rebuild it.  `DataLoader` mirrors the PyG loader the
reference uses (dss2_run.py:68-69): list of graphs in, shuffled mini-batches out, last batch partial.
"""
import torch

from . import _lib
from .dataset import ScenarioStore
from .graph import BatchGraph


class Data:
    """One graph: x[N,11], edge_index[2,E] (local ids), edge_attr[E,13], y[N,2] (the slice of PyG `Data` DSS2 uses)."""

    def __init__(self, x=None, edge_index=None, edge_attr=None, y=None):
        self.x, self.edge_index, self.edge_attr, self.y = x, edge_index, edge_attr, y

    @property
    def num_nodes(self):
        return self.x.size(0)

    def validate(self, raise_on_error=True):
        ei = self.edge_index
        ok = ei.dim() == 2 and ei.size(0) == 2 and ei.dtype == torch.long and (
            ei.numel() == 0 or (int(ei.min()) >= 0 and int(ei.max()) < self.num_nodes))
        if not ok and raise_on_error:
            raise ValueError("invalid edge_index")
        return ok


class Batch:
    """Disjoint-union batch (attributes as PyG's `Batch`)."""

    def __init__(self, x, edge_index, edge_attr, y, batch, ptr, num_graphs, vminmax=None):
        self.x, self.edge_index, self.edge_attr, self.y = x, edge_index, edge_attr, y
        self.batch, self.ptr, self.num_graphs, self.vminmax = batch, ptr, num_graphs, vminmax

    def to(self, device):
        for k, v in list(self.__dict__.items()):
            if torch.is_tensor(v):
                setattr(self, k, v.to(device))
        return self


def store_from_graphs(graphs, device="cuda"):
    """Concatenate a python list of graphs into a (possibly ragged) device-resident ScenarioStore."""
    dev = torch.device(device)
    nn = torch.tensor([0] + [g.x.size(0) for g in graphs], dtype=torch.long)
    ne = torch.tensor([0] + [g.edge_index.size(1) for g in graphs], dtype=torch.long)
    z8, z6 = torch.zeros(8), torch.zeros(6)
    return ScenarioStore(
        x=torch.cat([g.x for g in graphs]).float().contiguous().to(dev),
        edge_attr=torch.cat([g.edge_attr for g in graphs]).float().contiguous().to(dev),
        y=torch.cat([g.y for g in graphs]).float().contiguous().to(dev),
        edge_index=torch.cat([g.edge_index for g in graphs], dim=1).long().contiguous().to(dev),
        node_off=torch.cumsum(nn, 0).to(dev), edge_off=torch.cumsum(ne, 0).to(dev),
        x_mean=z8, x_std=z8, edge_mean=z6, edge_std=z6,
        max_nodes=int(nn.max()), max_edges=int(ne.max()))


class BatchBuffers:
    """Pre-sized output buffers of the packer for up to `max_graphs` graphs (reused across steps)."""

    def __init__(self, store, max_graphs):
        dev = store.x.device
        nt, et = max_graphs * store.max_nodes, max_graphs * store.max_edges
        self.x = torch.empty(nt, 11, dtype=torch.float32, device=dev)
        self.edge_attr = torch.empty(et, 13, dtype=torch.float32, device=dev)
        self.y = torch.empty(nt, 2, dtype=torch.float32, device=dev)
        self.edge_index = torch.empty(2, et, dtype=torch.long, device=dev)
        self.batch = torch.empty(nt, dtype=torch.long, device=dev)
        self.ptr = torch.empty(max_graphs + 1, dtype=torch.long, device=dev)
        self.eptr = torch.empty(max_graphs + 1, dtype=torch.long, device=dev)
        self.vminmax = torch.empty(2, dtype=torch.float32, device=dev)


def launch_pack(store, ids, out, num_nodes, num_edges):
    """Enqueue dss2_pack_batch for `ids` (device int64 [B]) into tensors of `out` sliced to the batch size.
    Graph-capturable.  The edge_index view is [2, num_edges] inside a buffer with `out.edge_index.size(1)` columns."""
    lib = _lib.load()
    rc = lib.dss2_pack_batch(_lib.ptr(store.x), _lib.ptr(store.edge_attr), _lib.ptr(store.y), _lib.ptr(store.edge_index),
                             store.edge_index.size(1), _lib.ptr(store.node_off), _lib.ptr(store.edge_off), _lib.ptr(ids), ids.numel(),
                             _lib.ptr(out["x"]), _lib.ptr(out["edge_index"]), out["edge_index"].size(1), _lib.ptr(out["edge_attr"]),
                             _lib.ptr(out["y"]), _lib.ptr(out["batch"]), _lib.ptr(out["ptr"]), _lib.ptr(out["eptr"]),
                             _lib.ptr(out["vminmax"]), _lib.stream())
    _lib.check(rc, "dss2_pack_batch")


def _tile_cap():
    from . import ops
    return ops.tile_cap()


def pack_batch(store, ids, graph_cache=None):
    """Fresh Batch for scenario ids (sequence or tensor).  Sizes come from the host copy of the offsets."""
    _lib.load()
    dev = store.x.device
    if dev.type != "cuda":
        raise _lib.Dss2Error("pack_batch needs a CUDA-resident ScenarioStore (store.to('cuda'))")
    ids_host = torch.as_tensor(ids, dtype=torch.long).cpu()
    if not hasattr(store, "_host_off"):
        store._host_off = (store.node_off.cpu(), store.edge_off.cpu())
    hn, he = store._host_off
    nt = int((hn[ids_host + 1] - hn[ids_host]).sum())
    et = int((he[ids_host + 1] - he[ids_host]).sum())
    b = ids_host.numel()
    ids_dev = ids_host.to(dev)
    out = {
        "x": torch.empty(nt, 11, dtype=torch.float32, device=dev), "edge_attr": torch.empty(et, 13, dtype=torch.float32, device=dev),
        "y": torch.empty(nt, 2, dtype=torch.float32, device=dev), "edge_index": torch.empty(2, et, dtype=torch.long, device=dev),
        "batch": torch.empty(nt, dtype=torch.long, device=dev), "ptr": torch.empty(b + 1, dtype=torch.long, device=dev),
        "eptr": torch.empty(b + 1, dtype=torch.long, device=dev), "vminmax": torch.empty(2, dtype=torch.float32, device=dev),
    }
    with torch.cuda.device(dev):
        launch_pack(store, ids_dev, out, nt, et)
        batch = Batch(out["x"], out["edge_index"], out["edge_attr"], out["y"], out["batch"], out["ptr"], b, out["vminmax"])
        # structure: identical for every batch drawn from a uniform-topology store with the same graph count
        key = None
        if graph_cache is not None and _uniform(store):
            key = (b, store.max_nodes, store.max_edges, _tile_cap(), _lib.hop_keys_default())
        g = graph_cache.get(key) if key is not None else None
        if g is None:
            if key is not None:
                # a cached structure must not alias this batch's tensors: it keeps private copies
                g = BatchGraph(batch.edge_index.clone(), nt, ptr=batch.ptr.clone(), tile_cap=_tile_cap())
                graph_cache[key] = g
            else:
                g = BatchGraph(batch.edge_index, nt, ptr=batch.ptr, tile_cap=_tile_cap())
    batch.edge_index._dss2_graph = g
    batch.edge_index._dss2_graph_version = batch.edge_index._version
    return batch


def _uniform(store):
    """All scenarios share one topology (checked once per store)."""
    flag = getattr(store, "_uniform", None)
    if flag is None:
        s = store.num_scenarios
        n, e = store.max_nodes, store.max_edges
        flag = bool(store.x.size(0) == s * n and store.edge_index.size(1) == s * e)
        if flag and s > 1 and e > 0:
            ei = store.edge_index.view(2, s, e)
            flag = bool((ei == ei[:, :1, :]).all())
        store._uniform = flag
    return flag


class DataLoader:
    """Mini-batch iterator over a list of graphs (PyG loader semantics: `shuffle` re-draws a permutation from
    torch's global generator every epoch, the last batch may be partial).  Batches are packed on the GPU;
    `device=None` returns tensors on the device of the input graphs (CPU for the reference's dataset)."""

    def __init__(self, dataset, batch_size=1, shuffle=False, device=None):
        self.dataset, self.batch_size, self.shuffle = dataset, batch_size, shuffle
        self.out_device = torch.device(device) if device is not None else dataset[0].x.device
        self.store = store_from_graphs(dataset, "cuda")
        self._graphs = {}

    def __len__(self):
        return (len(self.dataset) + self.batch_size - 1) // self.batch_size

    def __iter__(self):
        n = len(self.dataset)
        order = torch.randperm(n) if self.shuffle else torch.arange(n)
        for i in range(0, n, self.batch_size):
            batch = pack_batch(self.store, order[i:i + self.batch_size], self._graphs)
            if self.out_device.type != "cuda":
                g = batch.edge_index._dss2_graph
                batch = batch.to(self.out_device)
                batch.edge_index._dss2_graph = g
                batch.edge_index._dss2_graph_version = batch.edge_index._version
            yield batch
