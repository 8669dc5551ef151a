"""Classical weighted-least-squares state estimation on the device: the estimator the reference runs beside DSS2 (case_study.py:1226-1357,
pandapower's WLS estimator) on the noisy measurements the GNN learns from, so that a trained model can be compared with it on the same
batches, in accuracy and in time.

For one scenario with N buses and E closed edges the estimator minimises, over (V, theta) with theta_slack = 0,

    J_s(V, th) = w_v  sum_n [R_n0 (Z_n0 - V_n)^2 + R_n1 (Z_n1 - th_n)^2] + w_p sum_n [R_n2 (Z_n2 - p_n)^2 + R_n3 (Z_n3 - q_n)^2]
               + w_pf sum_e [R'_e0 (Z'_e0 - P_f,e)^2 + R'_e1 (Z'_e1 - Q_f,e)^2]

with every term defined as the loss defines it (`gsp_wls_edge`, data.py:393-459): Z, R, Z', R' are the de-normalised, masked
measurements and weights (data.py:397-409; a normalised value of exactly 0 is absent); the slack is x column 9 (data.py:412-413); the
injections are load-positive, p_n = -sum_{to=n} P_t - sum_{from=n} P_f (data.py:428-429); the flows are the pi-model of data.py:370-376
(phase shift ignored) with c = V_lv^2, V_lv = min vn_kv (x column 8), and G, B, Gs, Bs from edge_attr columns 6-9.  All arithmetic is
fp64 on the fp32 inputs promoted exactly.

Two weightings share one code path:
  reg_coefs=None   classical WLS, w_v = w_p = w_pf = 1: every measurement weighted by its own R = 1 / sigma^2;
  reg_coefs=dict   the loss's data term, w_v = lam_v / N, w_p = lam_p / N, w_pf = lam_pf / E.  For a batch of one topology the sum of
                   J_s over the batch divided by B is gsp_wls_edge with lam_reg = 0, so the estimate minimises what the GNN is trained
                   on.  lam_reg, mu_v and mu_theta are ignored: the penalties are squared batch means and cannot be split per scenario.

Gauss-Newton from a flat start in csrc/estimate.cu, one thread per scenario; the gain matrix H^T W H is held as 2x2 (theta, V) blocks
per pair of buses that share a measurement (neighbours, and buses with a common neighbour, through the injections) and factorised by the
power flow's block LU in an elimination order chosen here once per topology.  Out of scope: PV buses, phase shifts, open-line charging,
bad-data detection and robust (LAV, Huber) estimators.
"""
import ctypes

import numpy as np
import torch

from . import _lib
from .ops import stage_rows
from .powerflow import block_elimination
from .synth import _bfs_tree

# bytes of per-chunk workspace wls_estimate aims for: the chunk is the largest scenario count that fits (profiles/r3e_wls_estimate.json
# times this 1 GiB chunk against an L2-sized one)
WORKSPACE_BUDGET = 1 << 30


def symbolic(edge_ft, slack_flags):
    """Host analysis of one topology: `edge_ft` [E,2] local (from, to) of the closed edges, `slack_flags` [N] (x column 9).

    Returns a dict of numpy arrays (int32 index lists) and counts: the block_elimination() lists (bus, pos, blk_ptr, blk_col, diag,
    upd_ptr, upd, fill) of the gain matrix's pattern, whose graph joins every two buses that share a measurement, and
      inc_ptr/inc       per bus its incident edges as (edge, end 0 = from / 1 = to, support slot of the other end)
      sup_ptr/sup_bus   per bus its support {i} u nbr(i): slot 0 = the bus, then the neighbours in incidence order; sup_pos = positions
      pair_ptr/pair_blk per bus the block of every (slot a, slot b) of its support, row-major
      edge_blk [E,4]    blocks (ii, ij, ji, jj) of every edge
    Raises ValueError for a slack count other than 1, a self loop or a grid that is not connected."""
    edge_ft = np.asarray(edge_ft, dtype=np.int64).reshape(-1, 2)
    slack_flags = np.asarray(slack_flags)
    N, E = slack_flags.shape[0], edge_ft.shape[0]
    slacks = np.nonzero(slack_flags == 1)[0]
    if slacks.size != 1:
        raise ValueError(f"estimation: the grid has {slacks.size} slack buses; one is supported")
    slack = int(slacks[0])
    if E == 0 or edge_ft.min() < 0 or edge_ft.max() >= N:
        raise ValueError("estimation: edge list out of range")
    if (edge_ft[:, 0] == edge_ft[:, 1]).any():
        raise ValueError("estimation: self loops are not supported")
    _bfs_tree(N, edge_ft[:, 0], edge_ft[:, 1], slack)   # raises ValueError: not connected through the closed edges

    inc = [[] for _ in range(N)]
    sup = [[i] for i in range(N)]
    slot = [{i: 0} for i in range(N)]
    for e, (f, t) in enumerate(edge_ft.tolist()):
        for end, (me, other) in enumerate(((f, t), (t, f))):
            if other not in slot[me]:
                slot[me][other] = len(sup[me])
                sup[me].append(other)
            inc[me].append((e, end, slot[me][other]))
    # gain-matrix graph: every two buses of one support share that bus's injection measurements (edges lie inside supports)
    adj = [set() for _ in range(N)]
    for s in sup:
        for a in s:
            adj[a].update(b for b in s if b != a)
    el = block_elimination(adj, list(range(N)))
    pos, where = el["pos"], el["where"]

    def blk(a, b):
        return where[int(pos[a])][int(pos[b])]

    inc_ptr = np.zeros(N + 1, dtype=np.int32)
    inc_ptr[1:] = np.cumsum([len(r) for r in inc])
    sup_ptr = np.zeros(N + 1, dtype=np.int32)
    sup_ptr[1:] = np.cumsum([len(s) for s in sup])
    pair_ptr = np.zeros(N + 1, dtype=np.int32)
    pair_ptr[1:] = np.cumsum([len(s) ** 2 for s in sup])
    sup_bus = np.array([b for s in sup for b in s], dtype=np.int32)
    out = dict(el)
    del out["rows"], out["where"]
    out.update({
        "num_buses": N, "num_edges": E, "slack": slack, "edge_ft": edge_ft.astype(np.int32),
        "inc_ptr": inc_ptr, "inc": np.array([z for r in inc for z in r], dtype=np.int32).reshape(-1, 3),
        "sup_ptr": sup_ptr, "sup_bus": sup_bus, "sup_pos": pos[sup_bus].astype(np.int32),
        "pair_ptr": pair_ptr, "pair_blk": np.array([blk(a, b) for s in sup for a in s for b in s], dtype=np.int32),
        "edge_blk": np.array([[blk(f, f), blk(f, t), blk(t, f), blk(t, t)] for f, t in edge_ft.tolist()], dtype=np.int32),
        "max_support": max(len(s) for s in sup)})
    return out


_DEV_KEYS = ("edge_ft", "inc_ptr", "inc", "sup_ptr", "sup_pos", "pair_ptr", "pair_blk", "edge_blk", "bus", "blk_ptr", "blk_col", "diag",
             "upd_ptr", "upd")
_CACHE = {}


def _se_topology(sym, dev=None):
    ptrs = [None if dev is None else dev[k].data_ptr() for k in _DEV_KEYS]
    return _lib.SeTopology(sym["num_buses"], sym["num_edges"], sym["slack"], sym["blk_col"].size, sym["upd"].shape[0], sym["pair_blk"].size,
                           sym["max_support"], *ptrs)


def _topology(edge_ft, slack_flags, device):
    """symbolic() uploaded once per (local edge list, slack flags, device): the analysis, the device arrays and the struct."""
    edge_ft = np.ascontiguousarray(edge_ft, dtype=np.int64)
    slack_flags = np.ascontiguousarray(slack_flags, dtype=np.int64)
    key = (edge_ft.tobytes(), slack_flags.tobytes(), str(device))
    hit = _CACHE.get(key)
    if hit is None:
        sym = symbolic(edge_ft, slack_flags)
        dev = {k: torch.as_tensor(np.ascontiguousarray(sym[k], dtype=np.int32), device=device) for k in _DEV_KEYS}
        hit = _CACHE[key] = (sym, dev, _se_topology(sym, dev))
    return hit


def workspace_bytes(sym, chunk):
    """Device workspace of an estimate of the topology `sym` (symbolic()) that runs `chunk` scenarios per launch."""
    return int(_lib.load(require_cuda=False).dss2_wls_estimate_workspace_bytes(ctypes.byref(_se_topology(sym)), int(chunk)))


def wls_estimate(x, edge_index, edge_attr, ptr, x_mean, x_std, edge_mean, edge_std, reg_coefs=None, tol=1e-8, max_iter=50, chunk=None):
    """WLS state estimate of every scenario of a PyG-ordered batch of one topology (`pack_batch(store, ids)`, the script's DataLoader
    batches): x [Nt,11], edge_index [2,Et], edge_attr [Et,13], ptr [B+1] and the dataset statistics, as gsp_wls_edge takes them.

    reg_coefs: None = classical WLS; a dict = the loss's data term (see the module docstring).  tol: stop when max |dx| <= tol (pu and
    rad).  max_iter: most Gauss-Newton updates.  chunk: scenarios per kernel launch (default: as many as fit WORKSPACE_BUDGET); results do
    not depend on it.  The defaults are chosen from measurements, not tuned: the fp64 right-hand side leaves a rounding floor under the
    step of up to 1.7e-9 on the golden CIGRE-14 scenarios (tol = 1e-10 left 2 of 128 unconverged, 1e-8 none), and max_iter = 50 covers
    the slow tail (profiles/r3e_wls_estimate.json: Oberrhein mostly 5-6 updates, the 10 k-bus feeder 15-33, the golden scenarios in the
    loss weighting up to 36).

    Returns a dict on x's device: vm_pu, va_rad [Nt] f64; output [Nt,2] f32 = ((V - x_mean0) / x_std0, theta), the model's output
    convention, for evaluate_batch / gsp_wls_edge; objective [B] f64 = J_s at the estimate; iterations [B] int32 (updates applied);
    converged [B] bool; max_step [B] f64 (the last max |dx|).  A scenario whose gain matrix is singular, whose values turn non-finite, or
    that does not converge in max_iter updates has converged False; the others are unaffected.

    The topology (graph 0's local edge list and slack) is analysed on the host and cached; every graph of the batch is checked on the
    device to have the same N, E, edge list and slack.  That check costs one host synchronisation per call, so the estimator cannot be
    captured in a CUDA graph.  Raises ValueError on mixed topologies, a slack count other than 1 or a grid that is not connected."""
    lib = _lib.load()
    out_device = x.device
    xg, xs = stage_rows(x)
    eg, es = stage_rows(edge_attr)
    if xg.size(1) < 11 or eg.size(1) < 13:
        raise ValueError("wls_estimate needs the full x [Nt,11] and edge_attr [Et,13] tensors of the batch")
    dev = xg.device
    ei = edge_index.to(dev).long()
    pt = torch.as_tensor(ptr).to(dev).long()
    B, Nt, Et = pt.numel() - 1, xg.size(0), eg.size(0)
    if B < 1 or Nt % B or Et % B or ei.dim() != 2 or ei.size(0) != 2 or ei.size(1) != Et:
        raise ValueError("wls_estimate: the batch's graphs do not share one topology (bus or edge counts differ)")
    N, E = Nt // B, Et // B
    if E == 0:
        raise ValueError("wls_estimate: the graphs have no edges")
    reg = reg_coefs is not None
    w_v, w_p, w_pf = ((float(reg_coefs["lam_v"]) / N, float(reg_coefs["lam_p"]) / N, float(reg_coefs["lam_pf"]) / E) if reg else (1.0, 1.0, 1.0))
    if max_iter < 0 or not tol > 0:
        raise ValueError("wls_estimate: max_iter >= 0 and tol > 0")
    with torch.cuda.device(dev):
        # one copy to the host: whether every graph matches graph 0, then graph 0's local edge list and slack flags
        local = ei.reshape(2, B, E) - pt[:-1].view(1, B, 1)
        slack = xg[:, 9].view(B, N)
        ok = ((pt == torch.arange(B + 1, device=dev) * N).all() & (local == local[:, :1]).all() & (slack == slack[:1]).all())
        head = torch.cat([ok.view(1).long(), local[:, 0].reshape(-1), slack[0].long(), (slack[0] != slack[0].round()).any().view(1).long()])
        h = head.cpu().numpy()
        if not h[0]:
            raise ValueError("wls_estimate: the batch's graphs do not share one topology (edge lists, slack flags or ptr differ)")
        if h[-1]:
            raise ValueError("wls_estimate: the slack flags (x column 9) must be 0 or 1")
        sym, _dev, topo = _topology(h[1:1 + 2 * E].reshape(2, E).T, h[1 + 2 * E:1 + 2 * E + N], dev)
        stats = torch.cat([torch.as_tensor(t).float().reshape(-1).to(dev) for t in (x_mean, x_std, edge_mean, edge_std)]).contiguous()
        if stats.numel() != 28:
            raise ValueError("wls_estimate: x_mean, x_std [8] and edge_mean, edge_std [6]")
        if chunk is None:
            chunk = max(1, min(B, WORKSPACE_BUDGET // lib.dss2_wls_estimate_workspace_bytes(ctypes.byref(topo), 1)))
        chunk = max(1, min(int(chunk), B))
        ws = torch.empty(lib.dss2_wls_estimate_workspace_bytes(ctypes.byref(topo), chunk), dtype=torch.uint8, device=dev)
        f64 = dict(dtype=torch.float64, device=dev)
        res = {"vm_pu": torch.empty(Nt, **f64), "va_rad": torch.empty(Nt, **f64), "output": torch.empty(Nt, 2, dtype=torch.float32, device=dev),
               "objective": torch.empty(B, **f64), "iterations": torch.empty(B, dtype=torch.int32, device=dev),
               "converged": torch.empty(B, dtype=torch.bool, device=dev), "max_step": torch.empty(B, **f64)}
        P = _lib.ptr
        _lib.check(lib.dss2_wls_estimate(ctypes.byref(topo), B, P(xg), xs, P(eg), es, P(stats), w_v, w_p, w_pf, float(tol), int(max_iter),
                                         P(res["vm_pu"]), P(res["va_rad"]), P(res["output"]), P(res["objective"]), P(res["iterations"]),
                                         P(res["converged"]), P(res["max_step"]), P(ws), ws.numel(), chunk, _lib.stream()),
                   "dss2_wls_estimate")
    if out_device.type != "cuda":
        res = {k: v.to(out_device) for k, v in res.items()}
    return res
