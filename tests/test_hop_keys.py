"""Swizzle keys of the TAG layer kernels' plain level tiles (DSS2_HOP_KEYS_* in dss2_b200.h, hop_keys_tile in csrc/graph.cu).

The keys only move bytes inside shared memory and inside the spilled hop levels, so every output must be bit-identical between the
`identity` and `color` policies.  CPU: the host model of the key assignment.  GPU: the device keys against that model, then the layer
kernels, the weight-gradient passes reading the spilled levels, training steps and an evaluator epoch, bit for bit across policies."""
import numpy as np
import pytest
import torch

from dss2 import _lib, graph, synth


def _grid_batch(case, nb):
    """(edge_index [2, E], ptr [nb + 1]) of nb copies of a repository grid, numpy."""
    st = synth.synthetic_store(synth.load_grid(case), 1, device="cpu")
    ei, n = st.edge_index.numpy(), st.max_nodes
    return np.concatenate([ei + b * n for b in range(nb)], axis=1), np.arange(nb + 1) * n


# ---------------------------------------------------------------------------------------------------------------- CPU


def test_identity_policy_is_row_and_7():
    ci, tp = graph.host_ell(*_grid_batch("ober_sub", 37))
    keys = graph.host_hop_keys(ci, tp, "identity")
    assert np.array_equal(keys, (np.arange(ci.shape[0]) & 7).astype(np.uint8))


@pytest.mark.parametrize("case", ["ober_sub", "cigre14", "cigre14_reswitched"])
def test_color_keys_in_range_deterministic_and_fewer_gather_wavefronts(case):
    ci, tp = graph.host_ell(*_grid_batch(case, 64))
    keys = graph.host_hop_keys(ci, tp, "color")
    assert keys.max() <= 7
    assert np.array_equal(keys, graph.host_hop_keys(ci, tp, "color"))
    ident = graph.hop_wavefronts(ci, tp, graph.host_hop_keys(ci, tp, "identity"))
    col = graph.hop_wavefronts(ci, tp, keys)
    assert ident["store"][0] == ident["store"][1]          # identity: consecutive rows never share banks
    assert col["gather"][0] < ident["gather"][0] and col["gather"][0] <= 1.15 * col["gather"][1]


def test_host_keys_reject_oversized_tiles_and_unknown_policies():
    ci, tp = graph.host_ell(*_grid_batch("cigre14", 40))
    with pytest.raises(_lib.Dss2Error):
        graph.host_hop_keys(ci, np.array([0, ci.shape[0]]), "color")     # 600 rows in one tile
    lib = _lib.load(require_cuda=False)
    keys = np.zeros(ci.shape[0], dtype=np.uint8)
    tp = np.ascontiguousarray(tp, dtype=np.int64)
    assert lib.dss2_hop_keys_host(ci.ctypes.data, tp.ctypes.data, len(tp) - 1, 7, keys.ctypes.data) != 0


def test_saturated_degree_keeps_keys_valid():
    # a hub with more entries than the ELL degree field holds: the degree saturates, the keys stay in range
    hub = _lib.ELL_DEG_MASK + 10
    ei = np.stack([np.r_[np.zeros(hub, np.int64), np.arange(1, 6)], np.r_[np.ones(hub, np.int64), np.arange(2, 7)]])
    ci, tp = graph.host_ell(ei, np.array([0, 7]))
    assert ci[1, 1] == _lib.ELL_DEG_MASK
    assert graph.host_hop_keys(ci, tp, "color").max() <= 7


# ---------------------------------------------------------------------------------------------------------------- GPU


def _graphs():
    """name -> (edge_index int64 [2, E] cuda, ptr cuda, tile_cap)."""
    rng = np.random.default_rng(5)
    out = {}
    out["bench"] = _grid_batch("ober_sub", 48) + (256,)
    sizes = rng.integers(2, 71, size=30)             # ragged: random trees
    eis, ptr = [], [0]
    for n in sizes:
        par = np.array([rng.integers(0, i) for i in range(1, n)])
        eis.append(np.stack([par, np.arange(1, n)]) + ptr[-1])
        ptr.append(ptr[-1] + n)
    out["ragged"] = (np.concatenate(eis, axis=1), np.array(ptr), 256)
    hubs, ptr = [], [0]                              # stars with 5..40 leaves (hub rows) and parallel lines
    for leaves in (5, 9, 40, 17):
        hubs.append(np.stack([np.zeros(leaves, np.int64), np.arange(1, leaves + 1)]) + ptr[-1])
        hubs.append(np.array([[0, 0], [1, 1]]) + ptr[-1])
        ptr.append(ptr[-1] + leaves + 1)
    out["hubs"] = (np.concatenate(hubs, axis=1), np.array(ptr), 256)
    ei, ptr = _grid_batch("cigre14", 1)              # input self loops on every fourth bus (edges stay graph-major)
    one = np.concatenate([ei, np.stack([np.arange(0, ptr[-1], 4)] * 2)], axis=1)
    out["self_loops"] = (np.concatenate([one + b * ptr[-1] for b in range(40)], axis=1), np.arange(41) * ptr[-1], 256)
    out["rw4"] = _grid_batch("ober_sub", 21)[:2] + (128,)
    return {k: (torch.from_numpy(np.ascontiguousarray(e)).long().cuda(), torch.from_numpy(p).long().cuda(), c) for k, (e, p, c) in out.items()}


def _build(ei, ptr, cap, policy):
    return graph.BatchGraph(ei, int(ptr[-1]), ptr=ptr, undirect=1, tile_cap=cap, hop_keys=policy)


@pytest.mark.gpu
def test_device_keys_equal_the_host_model():
    for name, (ei, ptr, cap) in _graphs().items():
        ci, tp = graph.host_ell(ei.cpu().numpy(), ptr.cpu().numpy(), cap)
        for policy in ("identity", "color"):
            g = _build(ei, ptr, cap, policy)
            assert g.c.num_tiles == len(tp) - 1 and g.c.hop_keys == _lib.HOP_KEYS[policy], name
            arr = g.arrays()
            keys = arr["hop_key"].cpu().numpy()
            assert np.array_equal(keys, graph.host_hop_keys(ci, tp, policy)), (name, policy)
            word = arr["ell_ci"].cpu().numpy().view(np.uint32).reshape(-1, 2)
            assert np.array_equal(word[:, 0], ci[:, 0]) and np.array_equal(word[:, 1] & _lib.ELL_DEG_MASK, ci[:, 1]), name
            up = word[:, 1] >> _lib.ELL_KEY_SHIFT
            assert np.array_equal(up & 7, keys), name
            n0 = np.repeat(tp[:-1], np.diff(tp))
            for d in range(4):
                act = np.minimum(ci[:, 1], 4) > d
                src = n0 + ((ci[:, 0] >> (8 * d)) & 0xff)
                assert np.array_equal((up[act] >> (3 + 3 * d)) & 7, keys[src[act]]), (name, d)


def _layer_outputs(g, cout, act, seed):
    """Forward, backward-to-input, and both weight-gradient passes (reading the spilled levels) of one K = 2 layer on graph g."""
    lib, P = _lib.load(), _lib.ptr
    K, nt = 2, g.num_nodes
    gen = torch.Generator(device="cuda").manual_seed(seed)
    x = torch.randn(nt, 32, device="cuda", generator=gen)
    w = torch.randn(K + 1, cout, 32, device="cuda", generator=gen) / 6.0
    bias = torch.randn(cout, device="cuda", generator=gen)
    gy = torch.randn(nt, cout, device="cuda", generator=gen)
    y = torch.full((nt, cout), float("nan"), device="cuda")
    bits = torch.zeros(nt, dtype=torch.int32, device="cuda")
    _lib.check(lib.dss2_tag_fwd_tc2(g.ref, P(x), P(w), P(bias), cout, K, act, 0.0, 0, None, 0, None, None, 0, P(y), P(bits) if act else None,
                                    _lib.stream()), "fwd")
    ws = torch.empty(lib.dss2_tag_bwd_tc2_workspace_bytes(nt, K), dtype=torch.uint8, device="cuda")
    gx = torch.full((nt, 32), float("nan"), device="cuda")
    abits = bits if act else None
    _lib.check(lib.dss2_tag_bwd_tc2_gx(g.ref, P(w), cout, K, act, 0.3, P(abits), P(gy), P(gx), P(ws), ws.numel(), _lib.stream()), "gx")
    npart, nw = lib.dss2_num_partials(), (K + 1) * cout * 32
    out = {"y": y, "bits": bits, "gx": gx}
    for name, fn in (("gw", lib.dss2_tag_bwd_tc2_gw), ("gw_ffma", lib.dss2_tag_gw_ffma)):
        part = torch.zeros(npart, nw + 8 + 32, device="cuda")
        _lib.check(fn(nt, P(x), cout, K, act, 0.3, P(abits), P(gy), P(part), nw + 40, nw + 8, P(ws), ws.numel(), _lib.stream()), name)
        out[name] = part
    torch.cuda.synchronize()
    return out


@pytest.mark.gpu
@pytest.mark.parametrize("cout,act", [(32, 1), (32, 0), (16, 0), (8, 0), (2, 0)])
def test_layer_kernels_bit_identical_across_policies(cout, act):
    for name, (ei, ptr, cap) in _graphs().items():
        res = {}
        for policy in ("identity", "color"):
            res[policy] = _layer_outputs(_build(ei, ptr, cap, policy), cout, act, seed=cout + 100 * act)
        for k, v in res["identity"].items():
            assert torch.isfinite(v.float()).all() or k == "bits", (name, k)
            assert torch.equal(v.view(torch.int32), res["color"][k].view(torch.int32)), (name, cout, act, k)


@pytest.mark.gpu
def test_training_steps_and_evaluator_epoch_bit_identical_across_policies(monkeypatch):
    from dss2.evaluator import GraphedEvaluator
    from dss2.trainer import GraphedTrainer, default_spec
    nb = 6
    got = {}
    for policy in ("identity", "color"):
        monkeypatch.setenv("DSS2_HOP_KEYS", policy)
        store = synth.synthetic_store(synth.load_grid("ober_sub"), 4 * nb, seed=5, device="cuda")
        tr = GraphedTrainer(store, nb, spec=default_spec(p_drop=0.3), seed=1).capture()
        assert tr.graph.hop_keys == policy
        losses = [tr.step(torch.arange(s, s + nb, device="cuda") % store.num_scenarios).clone() for s in range(4)]
        ev = GraphedEvaluator(store, nb, trainer=tr)
        for s in range(0, 3 * nb, nb):
            ev.evaluate(torch.arange(s, s + nb, device="cuda"))
        got[policy] = (torch.stack(losses), {k: v.clone() for k, v in tr.state_dict().items()}, ev.metrics(reset=True))
    a, b = got["identity"], got["color"]
    assert torch.equal(a[0], b[0])
    assert a[1].keys() == b[1].keys() and all(torch.equal(a[1][k], b[1][k]) for k in a[1])
    assert all(x == y or (x != x and y != y) for x, y in zip(a[2].values(), b[2].values()))
