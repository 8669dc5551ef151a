"""Batched AC power flow (dss2.powerflow, csrc/powerflow.cu) against the pandapower-solved CIGRE-14 scenarios, the synthetic states of
synth.sample_scenarios and the dense fp64 Newton-Raphson of tests/powerflow_reference.py.

Pandapower's labels satisfy the reference's closed-edge pi-model to 1e-8 MW / 1e-10 MVAr at every bus except the from-ends of the open
edges, where pandapower also charges the lines that are open at one end (a few 1e-3 MVAr the model does not contain).  So the golden
recipe takes pandapower's injections everywhere except the Q of those buses, which is the model's Q at the labels.  sample_scenarios
reports declared zero-injection buses as exactly zero although its random state draws power there, so its recipe takes the model's
injections at the sampled state (dss2.powerflow.injections; equal to the scenario's own columns at every other bus).
"""
import numpy as np
import pytest
import torch

from conftest import REG_COEFS, load_golden

import powerflow_reference as ref
from dss2 import powerflow, synth

GRIDS = ("cigre14", "cigre14_reswitched", "cigre14_all_closed", "ober_sub")


def load(case):
    """A grid of synth.load_grid, the 10 010-bus feeder (ober_sub_x143), or CIGRE-14 with all three switches closed
    (cigre14_all_closed).  The re-switched grid's one loop runs through the slack, so its reduced system is radial; with all switches
    closed two loops avoid the slack and the elimination has fill."""
    if case == "ober_sub_x143":
        return synth.replicate_feeder(synth.load_grid("ober_sub"), 143)
    if case == "cigre14_all_closed":
        grid = synth.load_grid("cigre14")
        ep = grid["edge_param"].copy()
        ep[:, 6] = 1.0
        return dict(grid, name=case, edge_param=ep)
    return synth.load_grid(case)


def golden_recipe():
    """grid, p_mw, q_mvar [128,N] and labels [128,N,2] of the pandapower-solved CIGRE-14 scenarios (see the module docstring)."""
    fx = load_golden("cigre14_scenarios.npz")
    grid = synth.load_grid("cigre14")
    assert np.array_equal(fx["nodes"][0, :, :3], grid["bus_param"]) and np.array_equal(fx["edges"][0, :, :9], grid["edge_param"])
    labels = fx["labels"]
    p, q = fx["nodes"][:, :, 5].copy(), fx["nodes"][:, :, 6].copy()
    open_from = np.unique(grid["edge_param"][grid["edge_param"][:, 6] != 1.0, 0].astype(np.int64))
    _, q_model = powerflow.injections(grid, torch.from_numpy(labels[:, :, 0]), torch.from_numpy(labels[:, :, 1]))
    q[:, open_from] = q_model.numpy()[:, open_from]
    return grid, p, q, labels


def synthetic_recipe(grid, S, seed=5, device="cpu"):
    """p_mw, q_mvar and labels of S synth.sample_scenarios states (the model's injections at the state)."""
    _, _, labels = synth.sample_scenarios(grid, S, seed=seed, device=device)
    p, q = powerflow.injections(grid, labels[..., 0], labels[..., 1])
    return p, q, labels


def lu_solve_like_the_kernel(sym, A, b):
    """The kernel's row-wise block LU and substitutions on the symbolic lists, in numpy: A [blocks,2,2], b [n,2]."""
    A = A.copy()
    n = sym["diag"].size
    for k in range(n):
        for p in range(sym["blk_ptr"][k], sym["diag"][k]):
            A[p] = A[p] @ A[sym["diag"][sym["blk_col"][p]]]
            for dst, src in sym["upd"][sym["upd_ptr"][p]:sym["upd_ptr"][p + 1]]:
                A[dst] -= A[p] @ A[src]
        A[sym["diag"][k]] = np.linalg.inv(A[sym["diag"][k]])
    y = b.copy()
    for k in range(n):
        for p in range(sym["blk_ptr"][k], sym["diag"][k]):
            y[k] -= A[p] @ y[sym["blk_col"][p]]
    for k in range(n - 1, -1, -1):
        for p in range(sym["diag"][k] + 1, sym["blk_ptr"][k + 1]):
            y[k] -= A[p] @ y[sym["blk_col"][p]]
        y[k] = A[sym["diag"][k]] @ y[k]
    return y


# ---------------------------------------------------------------------------------------------------------------------------------
# CPU
# ---------------------------------------------------------------------------------------------------------------------------------
def test_reference_returns_pandapower_labels():
    grid, p, q, labels = golden_recipe()
    vm, va, its, conv, _ = ref.powerflow_nr(grid["bus_param"], grid["edge_param"], p, q, labels[:, 0, 0])
    assert conv.all()
    assert np.abs(vm - labels[:, :, 0]).max() <= 1e-9
    assert np.abs(va - labels[:, :, 1]).max() <= 1e-9


@pytest.mark.parametrize("case", GRIDS)
def test_reference_recovers_synthetic_states(case):
    grid = load(case)
    p, q, labels = synthetic_recipe(grid, 12)
    vm, va, _, conv, _ = ref.powerflow_nr(grid["bus_param"], grid["edge_param"], p.numpy(), q.numpy(), 1.03)
    assert conv.all()
    assert np.abs(vm - labels[..., 0].numpy()).max() <= 1e-9
    assert np.abs(va - labels[..., 1].numpy()).max() <= 1e-9


@pytest.mark.parametrize("case", ["cigre14", "cigre14_reswitched", "ober_sub", "ober_sub_x143"])
def test_symbolic_radial_grids_have_no_fill(case):
    grid = load(case)
    sym = powerflow.symbolic(grid)
    n = grid["bus_param"].shape[0] - 1
    assert sym["fill"] == 0 and (sym["blk_y"] >= 0).all()
    assert sorted(sym["bus"].tolist()) == [i for i in range(n + 1) if i != sym["slack"]]
    # radial: each bus has one later neighbour, so one update per lower block (the parent's diagonal)
    assert sym["upd"].shape[0] == (sym["blk_col"].size - n) // 2


def test_symbolic_meshed_grid_has_fill_and_a_valid_elimination():
    sym = powerflow.symbolic(load("cigre14_all_closed"))
    assert sym["fill"] > 0 and (sym["blk_y"] < 0).sum() == 2 * sym["fill"]
    n = sym["diag"].size
    rng = np.random.default_rng(0)
    A = rng.standard_normal((sym["blk_col"].size, 2, 2))
    A[sym["blk_y"] < 0] = 0.0                      # fill blocks start as zeros, as in the kernel's assembly
    A[sym["diag"]] += 20.0 * np.eye(2)
    dense = np.zeros((2 * n, 2 * n))
    for k in range(n):
        for p in range(sym["blk_ptr"][k], sym["blk_ptr"][k + 1]):
            m = sym["blk_col"][p]
            dense[2 * k:2 * k + 2, 2 * m:2 * m + 2] = A[p]
    b = rng.standard_normal((n, 2))
    x = lu_solve_like_the_kernel(sym, A, b)
    assert np.abs(x.reshape(-1) - np.linalg.solve(dense, b.reshape(-1))).max() <= 1e-12


def test_symbolic_rejects_isolated_bus_and_two_slacks():
    grid = synth.load_grid("cigre14")
    ep = grid["edge_param"].copy()
    bus = 5
    ep[(ep[:, 0] == bus) | (ep[:, 1] == bus), 6] = 0.0
    with pytest.raises(ValueError, match="not connected"):
        powerflow.symbolic(dict(grid, edge_param=ep))
    bp = grid["bus_param"].copy()
    bp[3, 1] = 1.0
    with pytest.raises(ValueError, match="2 slack buses"):
        powerflow.symbolic(dict(grid, bus_param=bp))


# ---------------------------------------------------------------------------------------------------------------------------------
# GPU
# ---------------------------------------------------------------------------------------------------------------------------------
def _cuda(*ts):
    return [torch.as_tensor(t, dtype=torch.float64).cuda() for t in ts]


@pytest.mark.gpu
def test_solve_returns_pandapower_labels():
    grid, p, q, labels = golden_recipe()
    r = powerflow.solve(grid, *_cuda(p, q), v_slack=torch.as_tensor(labels[:, 0, 0]).cuda())
    _, _, its, _, _ = ref.powerflow_nr(grid["bus_param"], grid["edge_param"], p, q, labels[:, 0, 0])
    assert bool(r["converged"].all())
    assert np.array_equal(r["iterations"].cpu().numpy(), its)
    assert float((r["vm_pu"].cpu() - torch.from_numpy(labels[:, :, 0])).abs().max()) <= 1e-9
    assert float((r["va_rad"].cpu() - torch.from_numpy(labels[:, :, 1])).abs().max()) <= 1e-9
    assert float(r["max_mismatch_mva"].max()) <= 1e-8


@pytest.mark.gpu
@pytest.mark.parametrize("case,S", [("cigre14", 64), ("cigre14_reswitched", 64), ("cigre14_all_closed", 64), ("ober_sub", 256),
                                    ("ober_sub_x143", 4)])
def test_solve_recovers_synthetic_states(case, S):
    grid = load(case)
    p, q, labels = synthetic_recipe(grid, S, device="cuda")
    r = powerflow.solve(grid, p, q)
    assert bool(r["converged"].all())
    assert float((r["vm_pu"] - labels[..., 0]).abs().max()) <= 1e-9
    assert float((r["va_rad"] - labels[..., 1]).abs().max()) <= 1e-9
    if case != "ober_sub_x143":
        _, _, its, _, _ = ref.powerflow_nr(grid["bus_param"], grid["edge_param"], p[:16].cpu().numpy(), q[:16].cpu().numpy(), 1.03)
        assert np.array_equal(r["iterations"][:16].cpu().numpy(), its)


@pytest.mark.gpu
@pytest.mark.parametrize("case", GRIDS)
def test_flows_slack_and_layout_match_branch_flows(case):
    grid = load(case)
    p, q, _ = synthetic_recipe(grid, 32, device="cuda")
    r = powerflow.solve(grid, p, q)
    closed = grid["edge_param"][:, 6] == 1.0
    ce = torch.as_tensor(grid["edge_param"][closed], device="cuda")
    flows = synth.branch_flows(r["vm_pu"], r["va_rad"], ce[:, 0].long(), ce[:, 1].long(), ce[:, 2], ce[:, 3], ce[:, 4], ce[:, 5],
                               float(grid["bus_param"][:, 0].min()))
    for name, ref in zip(("p_from", "q_from", "p_to", "q_to"), flows):
        assert float((r[name] - ref).abs().max()) <= 1e-12 * float(ref.abs().max()), name
    # slack injection = minus the flows leaving the slack; every other entry is the input
    p_ref, q_ref = powerflow.injections(grid, r["vm_pu"], r["va_rad"])
    sl = int(np.nonzero(grid["bus_param"][:, 1] == 1.0)[0][0])
    for out, ref, given in ((r["p_mw"], p_ref, p), (r["q_mvar"], q_ref, q)):
        assert float((out[:, sl] - ref[:, sl]).abs().max()) <= 1e-12 * float(ref[:, sl].abs().max())
        keep = [i for i in range(p.shape[1]) if i != sl]
        assert torch.equal(out[:, keep], given[:, keep])
    # solved_scenarios: the layout of sample_scenarios column for column
    nodes, edges, labels = powerflow.solved_scenarios(grid, p, q)
    n_ref, e_ref, l_ref = synth.sample_scenarios(grid, 32, seed=5, device="cuda")
    assert nodes.shape == n_ref.shape and edges.shape == e_ref.shape and labels.shape == l_ref.shape
    assert nodes.dtype == edges.dtype == labels.dtype == torch.float64
    assert torch.equal(nodes[..., :3], n_ref[..., :3]) and torch.equal(edges[..., :9], e_ref[..., :9])
    zi = grid["bus_param"][:, 2] == 1.0
    nz = torch.as_tensor(~zi, device="cuda")
    assert float((nodes[..., 3:5] - n_ref[..., 3:5]).abs().max()) <= 1e-9
    assert float((nodes[:, nz, 5:7] - n_ref[:, nz, 5:7]).abs().max()) <= 1e-9 * float(n_ref[..., 5:7].abs().max())
    assert float((edges[..., 9:] - e_ref[..., 9:]).abs().max()) <= 1e-9 * float(e_ref[..., 9:].abs().max())
    assert torch.equal(edges[:, torch.as_tensor(~closed, device="cuda"), 9:], e_ref[:, torch.as_tensor(~closed, device="cuda"), 9:])
    assert torch.equal(labels, torch.stack([r["vm_pu"], r["va_rad"]], -1))


@pytest.mark.gpu
def test_failures_are_reported_per_scenario():
    grid, p, q, labels = golden_recipe()
    p, q = _cuda(p[:24], q[:24])
    bad = torch.zeros(24, dtype=torch.bool, device="cuda")
    bad[[1, 7, 8, 20]] = True
    scale = torch.where(bad, 100.0, 1.0).double()[:, None]
    r = powerflow.solve(grid, p * scale, q * scale, max_iter=10)
    assert torch.equal(r["converged"], ~bad)
    assert bool((r["iterations"][bad] == 10).all())
    alone = powerflow.solve(grid, p[~bad], q[~bad])
    for k in ("vm_pu", "va_rad", "p_mw", "q_mvar", "p_from", "q_from", "p_to", "q_to", "iterations", "converged", "max_mismatch_mva"):
        assert torch.equal(r[k][~bad], alone[k]), k
    with pytest.raises(powerflow._lib.Dss2Error, match="4 of 24 scenarios did not converge"):
        powerflow.solved_scenarios(grid, p * scale, q * scale)


@pytest.mark.gpu
def test_deterministic_and_independent_of_chunking():
    grid = synth.load_grid("ober_sub")
    p, q, _ = synthetic_recipe(grid, 1000, seed=11, device="cuda")
    a, b = powerflow.solve(grid, p, q), powerflow.solve(grid, p, q)
    c = powerflow.solve(grid, p, q, chunk=96)
    parts = [powerflow.solve(grid, p[i:i + 300], q[i:i + 300]) for i in range(0, 1000, 300)]
    for k in a:
        assert torch.equal(a[k], b[k]), k
        assert torch.equal(a[k], c[k]), k
        assert torch.equal(a[k], torch.cat([d[k] for d in parts])), k


@pytest.mark.gpu
def test_solved_scenarios_train_end_to_end():
    from dss2 import dataset
    from dss2.trainer import GraphedTrainer
    fx = load_golden("cigre14_scenarios.npz")
    grid = synth.load_grid("cigre14")
    nodes, edges, labels = powerflow.solved_scenarios(grid, *_cuda(fx["nodes"][:, :, 5], fx["nodes"][:, :, 6]))
    S, N, E = nodes.shape[0], nodes.shape[1], int((grid["edge_param"][:, 6] == 1.0).sum())
    gen = torch.Generator(device="cuda").manual_seed(0)
    zn = torch.randn(S, N, 4, generator=gen, dtype=torch.float64, device="cuda")
    ze = torch.randn(S, E, 2, generator=gen, dtype=torch.float64, device="cuda")
    store = dataset.build_scenario_store(nodes, edges, labels, grid["noise_param"], grid["meas_v"], grid["meas_pflow"], zn, ze, device="cuda")
    tr = GraphedTrainer(store, 32, reg_coefs=REG_COEFS, lr=3e-3, seed=0).capture()
    losses = []
    for step in range(30):
        ids = torch.arange(32 * step, 32 * step + 32, device="cuda") % S
        losses.append(float(tr.step(ids)))
    assert all(np.isfinite(losses))
    assert losses[-1] < losses[0]
