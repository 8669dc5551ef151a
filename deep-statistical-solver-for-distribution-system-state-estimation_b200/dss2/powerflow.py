"""Batched AC power flow on the device (scope row 8f-2): the pandapower `runpp` stage of the reference's offline generator
(toy_network.py:160-250) on the reference's own pi-model (data.py:370-376, phase shift ignored as in data.py:362-363), so that sampled
loads (`dss2.sampling`) become solved, labelled scenarios for `dss2.dataset.build_scenario_store`.

One slack bus (fixed V, theta = 0) and PQ buses; the topology is shared by all scenarios of a call.  Newton-Raphson in polar form, fp64,
in csrc/powerflow.cu (`dss2_powerflow`): one thread per scenario, the reduced Jacobian held as 2x2 blocks per bus pair and factorised
in an elimination order chosen here once per topology (leaves first, then minimum degree: no fill on radial grids).  No dense Jacobian,
no host synchronisation inside the solve, no CPU fallback.
"""
import ctypes
import heapq

import numpy as np
import torch

from . import _lib
from .synth import _bfs_tree, branch_flows

WORKSPACE_BUDGET = 1 << 30   # bytes of per-chunk workspace solve() aims for: the chunk is the largest scenario count that fits


def symbolic(grid):
    """Host analysis of one topology: admittance matrix, elimination order and the 2x2-block pattern of the reduced Jacobian with fill.

    Returns a dict of numpy arrays (int32 index lists, float64 values) and counts:
      y_ptr/y_col/y_gb  Y * V_lv^2 over all N buses as CSR (columns ascending; parallel edges summed in edge order), [nnz, 2] = (G, B)
      bus[k]            bus eliminated at position k (the slack is not in the reduced system); pos[i] its inverse (-1 at the slack)
      blk_ptr/blk_col   CSR of the factor's block pattern in position order, columns ascending; blk_y[p] = Y entry of the block, -1 = fill
      diag[k]           block (k, k)
      upd_ptr/upd       per lower block p = (k, m): the pairs (block (k, j), block (m, j)) over the upper entries j > m of row m,
                        i.e. A[k, j] -= L[k, m] A[m, j] of the row-wise (IKJ) block LU
      fill              number of fill pairs (blocks off the Y pattern, counted once per bus pair)
    Raises ValueError when the grid's slack count is not 1 or it is not connected through its closed edges."""
    bus_param, edge_param = np.asarray(grid["bus_param"], dtype=np.float64), np.asarray(grid["edge_param"], dtype=np.float64)
    N = bus_param.shape[0]
    slacks = np.nonzero(bus_param[:, 1] == 1.0)[0]
    if slacks.size != 1:
        raise ValueError(f"powerflow: the grid has {slacks.size} slack buses; one is supported")
    slack = int(slacks[0])
    closed = edge_param[:, 6] == 1.0
    ce = edge_param[closed]
    frm, to = ce[:, 0].astype(np.int64), ce[:, 1].astype(np.int64)
    _bfs_tree(N, frm, to, slack)   # raises ValueError: not connected through the closed edges
    v_lv = float(bus_param[:, 0].min())

    # Y (pi-model, data.py:370-376), scaled to MVA at 1 pu
    ydict = {}
    for f, t, g, b, gs, bs in zip(frm, to, ce[:, 2], ce[:, 3], ce[:, 4], ce[:, 5]):
        for key, val in (((f, f), complex(g + gs / 2, b + bs / 2)), ((t, t), complex(g + gs / 2, b + bs / 2)),
                         ((f, t), complex(-g, -b)), ((t, f), complex(-g, -b))):
            ydict[key] = ydict.get(key, 0j) + val
    keys = sorted(ydict)
    y_row = np.array([k[0] for k in keys], dtype=np.int64)
    y_col = np.array([k[1] for k in keys], dtype=np.int32)
    y_ptr = np.searchsorted(y_row, np.arange(N + 1)).astype(np.int32)
    y_gb = np.array([[ydict[k].real, ydict[k].imag] for k in keys], dtype=np.float64) * v_lv ** 2
    y_index = {k: i for i, k in enumerate(keys)}

    # elimination order on the PQ graph (the slack is not in the reduced system)
    adj = [set() for _ in range(N)]
    for (i, j) in keys:
        if i != j and i != slack and j != slack:
            adj[i].add(j)
    el = block_elimination(adj, [i for i in range(N) if i != slack])
    bus, rows = el["bus"], el["rows"]
    blk_y = np.array([y_index.get((int(bus[k]), int(bus[c])), -1) for k, r in enumerate(rows) for c in r], dtype=np.int32)
    blk_ptr, blk_col, diag, upd_ptr, upd, fill, pos = (el[k] for k in ("blk_ptr", "blk_col", "diag", "upd_ptr", "upd", "fill", "pos"))
    return {"num_buses": N, "slack": slack, "v_lv": v_lv, "closed": np.nonzero(closed)[0], "edge_ft": np.stack([frm, to], 1).astype(np.int32),
            "edge_gb": np.ascontiguousarray(ce[:, 2:6]), "y_ptr": y_ptr, "y_col": y_col, "y_gb": y_gb, "bus": bus, "pos": pos,
            "blk_ptr": blk_ptr, "blk_col": blk_col, "blk_y": blk_y, "diag": diag, "upd_ptr": upd_ptr, "upd": upd, "fill": fill}


def block_elimination(adj, nodes):
    """Minimum-degree elimination of the graph `adj` (list of neighbour sets indexed by bus; consumed) restricted to `nodes`, and the
    2x2-block pattern with fill and the update lists of the row-wise block LU in csrc/block_lu.cuh.  Buses of degree 0/1 (the leaves)
    come first, ties by bus id.  Returns a dict:
      bus[k]            bus eliminated at position k; pos[i] its inverse (-1 off `nodes`)
      rows[k]           columns of block row k, ascending (host lists)
      blk_ptr/blk_col   CSR of the factor's block pattern in position order, columns ascending
      diag[k]           block (k, k); where[k][m] the block (k, m) (host dicts)
      upd_ptr/upd       per lower block p = (k, m): the pairs (block (k, j), block (m, j)) over the upper entries j > m of row m,
                        i.e. A[k, j] -= L[k, m] A[m, j]
      fill              number of fill pairs (blocks off the graph, counted once per bus pair)"""
    N = len(adj)
    heap = [(len(adj[i]), i) for i in nodes]
    heapq.heapify(heap)
    done = np.zeros(N, dtype=bool)
    order, upper, fill = [], {}, 0
    while heap:
        d, v = heapq.heappop(heap)
        if done[v] or d != len(adj[v]):
            continue
        done[v] = True
        order.append(v)
        nb = sorted(adj[v])
        upper[v] = nb
        for a in nb:
            adj[a].discard(v)
        for ia, a in enumerate(nb):
            for b in nb[ia + 1:]:
                if b not in adj[a]:
                    adj[a].add(b)
                    adj[b].add(a)
                    fill += 1
        for a in nb:
            heapq.heappush(heap, (len(adj[a]), a))
    n = len(order)
    bus = np.array(order, dtype=np.int32)
    pos = np.full(N, -1, dtype=np.int64)
    pos[bus] = np.arange(n)

    # block pattern: row k = diagonal + upper entries (later neighbours at elimination) + lower entries (mirror)
    rows = [[k] for k in range(n)]
    for k in range(n):
        for j in upper[int(bus[k])]:
            pj = int(pos[j])
            rows[k].append(pj)
            rows[pj].append(k)
    rows = [sorted(r) for r in rows]
    blk_ptr = np.zeros(n + 1, dtype=np.int32)
    blk_ptr[1:] = np.cumsum([len(r) for r in rows])
    blk_col = np.array([c for r in rows for c in r], dtype=np.int32)
    where = [{c: int(blk_ptr[k]) + i for i, c in enumerate(r)} for k, r in enumerate(rows)]
    diag = np.array([where[k][k] for k in range(n)], dtype=np.int32)
    upd_ptr = np.zeros(blk_col.size + 1, dtype=np.int32)
    upd = []
    for k in range(n):
        for m in rows[k]:
            p = where[k][m]
            if m < k:
                upd.extend((where[k][j], where[m][j]) for j in rows[m] if j > m)
            upd_ptr[p + 1] = len(upd)
    upd = np.array(upd, dtype=np.int32).reshape(-1, 2)
    return {"bus": bus, "pos": pos, "rows": rows, "where": where, "blk_ptr": blk_ptr, "blk_col": blk_col, "diag": diag,
            "upd_ptr": upd_ptr, "upd": upd, "fill": fill}


_CACHE = {}


def _topology(grid, device):
    """symbolic() uploaded once per (topology, device): the device arrays and the `dss2_pf_topology_t` that points at them."""
    key = (np.asarray(grid["bus_param"], dtype=np.float64).tobytes(), np.asarray(grid["edge_param"], dtype=np.float64).tobytes(), str(device))
    hit = _CACHE.get(key)
    if hit is None:
        sym = symbolic(grid)
        dev = {k: torch.as_tensor(np.ascontiguousarray(sym[k]), device=device)
               for k in ("y_ptr", "y_col", "y_gb", "bus", "blk_ptr", "blk_col", "blk_y", "diag", "upd_ptr", "upd", "edge_ft", "edge_gb")}
        topo = _lib.PfTopology(sym["num_buses"], sym["slack"], sym["num_buses"] - 1, sym["blk_col"].size, sym["upd"].shape[0],
                          sym["edge_ft"].shape[0], sym["v_lv"], *[dev[k].data_ptr() for k in (
                              "y_ptr", "y_col", "y_gb", "bus", "blk_ptr", "blk_col", "blk_y", "diag", "upd_ptr", "upd", "edge_ft", "edge_gb")])
        hit = _CACHE[key] = (sym, dev, topo)
    return hit


def workspace_bytes(grid, chunk):
    """Device workspace of a solve that runs `chunk` scenarios per launch."""
    sym = symbolic(grid)
    topo = _lib.PfTopology(sym["num_buses"], sym["slack"], sym["num_buses"] - 1, sym["blk_col"].size, sym["upd"].shape[0], sym["edge_ft"].shape[0])
    return int(_lib.load(require_cuda=False).dss2_powerflow_workspace_bytes(ctypes.byref(topo), int(chunk)))


def solve(grid, p_mw, q_mvar, v_slack=1.03, tol_mva=1e-8, max_iter=10, chunk=None):
    """AC power flow of S scenarios of `grid` (synth.load_grid / replicate_feeder) on the CUDA device of p_mw.

    p_mw, q_mvar: [S, N] fp64 load-positive bus injections (data.py:428-429); the slack's entries are ignored.  v_slack: float or [S].
    chunk: scenarios per kernel launch (default: as many as fit WORKSPACE_BUDGET); results do not depend on it.
    Returns a dict of fp64 CUDA tensors: vm_pu, va_rad [S,N]; p_mw, q_mvar [S,N] (the inputs with the computed slack injection);
    p_from, q_from, p_to, q_to [S,E_closed] (closed edges in grid order); iterations [S] int32; converged [S] bool; max_mismatch_mva [S].
    A scenario that did not converge (max_iter reached or a singular pivot) has converged False and undefined outputs; the others are
    unaffected.  Nothing here synchronises with the host."""
    if not torch.cuda.is_available():
        raise _lib.Dss2Error("dss2: no CUDA device; the power flow has no CPU fallback")
    lib = _lib.load()
    p_mw, q_mvar = torch.as_tensor(p_mw), torch.as_tensor(q_mvar)
    device = p_mw.device if p_mw.is_cuda else torch.device("cuda")
    f64 = dict(dtype=torch.float64, device=device)
    p_in, q_in = p_mw.to(**f64).contiguous(), q_mvar.to(**f64).contiguous()
    N = int(np.asarray(grid["bus_param"]).shape[0])
    if p_in.dim() != 2 or p_in.shape[1] != N or q_in.shape != p_in.shape:
        raise ValueError(f"powerflow.solve: p_mw and q_mvar must be [S, {N}]")
    if max_iter < 0 or not tol_mva > 0:
        raise ValueError("powerflow.solve: max_iter >= 0 and tol_mva > 0")
    S = p_in.shape[0]
    vs = torch.as_tensor(v_slack, **f64).expand(S).contiguous()
    sym, _dev, topo = _topology(grid, device)
    E = sym["edge_ft"].shape[0]
    if chunk is None:
        per = lib.dss2_powerflow_workspace_bytes(ctypes.byref(topo), 1)
        chunk = max(1, min(S, WORKSPACE_BUDGET // per))
    chunk = max(1, min(int(chunk), S))
    ws = torch.empty(lib.dss2_powerflow_workspace_bytes(ctypes.byref(topo), chunk), dtype=torch.uint8, device=device)
    out = {"vm_pu": torch.empty(S, N, **f64), "va_rad": torch.empty(S, N, **f64), "p_mw": p_in.clone(), "q_mvar": q_in.clone()}
    for k in ("p_from", "q_from", "p_to", "q_to"):
        out[k] = torch.empty(S, E, **f64)
    out["iterations"] = torch.empty(S, dtype=torch.int32, device=device)
    out["converged"] = torch.empty(S, dtype=torch.bool, device=device)
    out["max_mismatch_mva"] = torch.empty(S, **f64)
    P = _lib.ptr
    with torch.cuda.device(device):
        _lib.check(lib.dss2_powerflow(ctypes.byref(topo), S, P(p_in), P(q_in), P(vs), float(tol_mva), int(max_iter), P(out["vm_pu"]),
                                      P(out["va_rad"]), P(out["p_mw"]), P(out["q_mvar"]), P(out["p_from"]), P(out["q_from"]), P(out["p_to"]),
                                      P(out["q_to"]), P(out["iterations"]), P(out["converged"]), P(out["max_mismatch_mva"]), P(ws), ws.numel(),
                                      chunk, _lib.stream()), "dss2_powerflow")
    return out


def injections(grid, vm_pu, va_rad):
    """Load-positive bus injections p_mw, q_mvar [S,N] that the pi-model gives at the state (vm_pu, va_rad) [S,N]: minus the sum of the
    closed branches' flows leaving each bus (synth.branch_flows, data.py:428-429).  Declared zero-injection buses are not zeroed."""
    vm, va = torch.as_tensor(vm_pu, dtype=torch.float64), torch.as_tensor(va_rad, dtype=torch.float64)
    dev = vm.device
    ep = np.asarray(grid["edge_param"], dtype=np.float64)
    ce = torch.as_tensor(ep[ep[:, 6] == 1.0], dtype=torch.float64, device=dev)
    frm, to = ce[:, 0].long(), ce[:, 1].long()
    v_lv = float(np.asarray(grid["bus_param"])[:, 0].min())
    p_f, q_f, p_t, q_t = branch_flows(vm, va, frm, to, ce[:, 2], ce[:, 3], ce[:, 4], ce[:, 5], v_lv)
    p, q = torch.zeros_like(vm), torch.zeros_like(vm)
    p.index_add_(1, to, -p_t)
    p.index_add_(1, frm, -p_f)
    q.index_add_(1, to, -q_t)
    q.index_add_(1, frm, -q_f)
    return p, q


def solved_scenarios(grid, p_mw, q_mvar, **solve_kw):
    """solve() in the pickle layout of synth.sample_scenarios, column for column: nodes [S,N,7] (NODE_COLS), edges [S,E_all,11]
    (EDGE_COLS; open edges carry zero flow), labels [S,N,2] = (vm_pu, va_rad), fp64 on the device.  Raises Dss2Error, with the count,
    when a scenario did not converge (this reads one flag count back to the host)."""
    r = solve(grid, p_mw, q_mvar, **solve_kw)
    bad = int((~r["converged"]).sum())
    if bad:
        raise _lib.Dss2Error(f"powerflow: {bad} of {r['converged'].numel()} scenarios did not converge")
    dev = r["vm_pu"].device
    S, N = r["vm_pu"].shape
    bus = torch.as_tensor(np.asarray(grid["bus_param"], dtype=np.float64), device=dev)
    edge = torch.as_tensor(np.asarray(grid["edge_param"], dtype=np.float64), device=dev)
    nodes = torch.cat([bus.unsqueeze(0).expand(S, N, 3), r["vm_pu"].unsqueeze(-1), r["va_rad"].unsqueeze(-1),
                       r["p_mw"].unsqueeze(-1), r["q_mvar"].unsqueeze(-1)], dim=-1)
    e_all = edge.shape[0]
    flows = torch.zeros(S, e_all, 2, dtype=torch.float64, device=dev)
    cidx = torch.as_tensor(np.nonzero(np.asarray(grid["edge_param"])[:, 6] == 1.0)[0], device=dev)
    flows[:, cidx, 0] = r["p_from"]
    flows[:, cidx, 1] = r["q_from"]
    edges = torch.cat([edge.unsqueeze(0).expand(S, e_all, 9), flows], dim=-1)
    labels = torch.stack([r["vm_pu"], r["va_rad"]], dim=-1)
    return nodes, edges, labels
