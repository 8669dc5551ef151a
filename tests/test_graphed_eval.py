"""GraphedEvaluator (dss2/evaluator.py): the captured validation / inference pass of the throughput tier against the drop-in path
(networks module in eval() under no_grad -> metrics.evaluate_batch / data.get_pflow), bit for bit, and the device finaliser of
dss2_eval_metrics_acc against the script's formulas evaluated in Python on the kernel's own sums."""
import math

import pytest
import torch

pytestmark = pytest.mark.gpu

B = 8          # graphs per batch; the validation set is 2 B + R scenarios, so its last batch is partial
R = 3


def _store(case, n, seed):
    from dss2 import synth
    return synth.synthetic_store(synth.load_grid(case), n, seed=seed, device="cuda")


def _trainer(network, store, p_drop=0.0, seed=0, gat_dropout=0.0):
    from dss2.trainer import GraphedTrainer, default_spec
    spec = None
    if network == "skippfn":
        spec = default_spec(p_drop=p_drop)
    elif network == "gat" and gat_dropout:
        from dss2.gat import GATSpec
        spec = GATSpec(dim_feat=8, dim_dense=32, dim_out=2, num_layers=8, edge_dim=6, dropout=gat_dropout)
    return GraphedTrainer(store, B, spec=spec, seed=seed, network=network).capture()


def _module(network, spec, sd):
    """The drop-in module with the trainer's parameters, in eval() (the script's validation loop)."""
    import networks
    if network == "skippfn":
        m = networks.SkipPFN(spec.fn, spec.fe, spec.dim_out, spec.hid, spec.n_layers, spec.K, spec.p_drop, spec.L)
    elif network == "gat":
        m = networks.GAT_DSSE(dim_feat=8, dim_dense=32, dim_out=2, heads=1, num_layers=spec.num_layers, edge_dim=6, dropout=spec.dropout)
    else:
        m = networks.GINE_DSSE(dim_feat=8, dim_dense=32, dim_out=2, num_layers=spec.num_layers, edge_dim=6)
    msd = m.state_dict()
    m.load_state_dict({k: (sd[k].reshape(v.shape).cpu() if k in sd else v) for k, v in msd.items()}, strict=True)
    return m.cuda().eval()


def _batches(lo, n_val):
    ids = torch.arange(lo, lo + n_val, device="cuda")
    return [ids[i:i + B] for i in range(0, n_val, B)]


def _dropin(model, store, sel):
    from dss2 import batching
    pb = batching.pack_batch(store, sel)
    with torch.no_grad():
        out = model(pb.x[:, :8], pb.edge_index, pb.edge_attr[:, :6])
    return pb, out


def _dropin_epoch(model, store, batches):
    """The script's aggregation: sequential Python sum of the per-batch values, divided by the number of batches."""
    from dss2 import metrics
    tot = None
    for sel in batches:
        pb, out = _dropin(model, store, sel)
        m = metrics.evaluate_batch(out, pb.y, pb.x, pb.edge_index, pb.edge_attr, store.x_mean, store.x_std)
        tot = dict(m) if tot is None else {k: tot[k] + m[k] for k in tot}
    return {k: v / len(batches) for k, v in tot.items()}


def _same(got, want):
    for k, w in want.items():
        g = got[k]
        assert g == w or (math.isnan(g) and math.isnan(w)), (k, g, w)


def _train(tr, store, steps=3):
    for s in range(steps):
        tr.step(torch.arange(s, s + B, device="cuda") % store.num_scenarios)


def _epoch(ev, batches):
    for sel in batches:
        ev.evaluate(sel)
    return ev.metrics(reset=True)


@pytest.fixture
def tiny_tiles(monkeypatch):
    """A tile cap below the grid size: every kernel takes its large-graph path (global scratch, one launch per phase)."""
    from dss2 import graph, ops
    monkeypatch.setenv("DSS2_TILE_CAP", "8")
    ei = torch.tensor([[i for i in range(11)], [i + 1 for i in range(11)]], device="cuda")
    assert graph.BatchGraph(ei, 12, tile_cap=ops.tile_cap()).c.num_tiles == 0
    yield


def _check_against_dropin(network, train_case="ober_sub", val_case=None):
    """Trainer on `train_case`, evaluator on 2 B + R held-out scenarios (of `val_case`'s own store when given): epoch metrics, inference
    output and branch flows equal the drop-in path; replay equals eager launches; a second epoch repeats; an evaluator built from the
    state_dict equals the one on the trainer."""
    import data
    from dss2.evaluator import GraphedEvaluator
    store = _store(train_case, 4 * B, seed=5)
    tr = _trainer(network, store)
    _train(tr, store)
    if val_case is None:
        val, batches = store, _batches(B, 2 * B + R)
    else:
        val, batches = _store(val_case, 2 * B + R, seed=21), _batches(0, 2 * B + R)
    ev = GraphedEvaluator(val, B, trainer=tr)
    got = _epoch(ev, batches)
    assert got["batches"] == len(batches) == 3
    model = _module(network, tr.spec, tr.state_dict())
    _same(got, _dropin_epoch(model, val, batches))
    # a second epoch after the reset gives the same dict
    _same(_epoch(ev, batches), got)
    # inference on the partial batch: the output, and get_pflow of the estimate built with torch ops (bench.py's inference step)
    sel = batches[-1]
    out, pflow = ev.infer(sel)
    pb, want = _dropin(model, val, sel)
    assert torch.equal(out, want)
    xs, xm = val.x_std.cuda(), val.x_mean.cuda()
    est = torch.cat([want[:, 0:1] * xs[:1] + xm[:1], want[:, 1:] * (1. - pb.x[:, 9:10])], 1)
    ref = data.get_pflow(est, pb.edge_index, node_param=pb.x[:, 8:], edge_param=pb.edge_attr[:, 6:])
    assert len(pflow) == 8 and all(torch.equal(a, b) for a, b in zip(pflow, ref))
    # graph replay == eager launches; an evaluator from the reference's parameter names == the one reading the trainer's buffer
    eager = GraphedEvaluator(val, B, trainer=tr, use_cuda_graph=False)
    _same(_epoch(eager, batches), got)
    assert torch.equal(eager.infer(sel)[0], out)
    from_sd = GraphedEvaluator(val, B, network=network, spec=tr.spec, state_dict=tr.state_dict())
    _same(_epoch(from_sd, batches), got)
    assert torch.equal(from_sd.infer(sel)[0], out)


@pytest.mark.parametrize("network", ["skippfn", "gat", "gine"])
def test_evaluator_equals_dropin_path(network):
    _check_against_dropin(network)


def test_evaluator_on_another_store_reswitched_grid():
    """Trained on CIGRE-14, evaluated on the re-switched (meshed, other edge list) CIGRE-14: the evaluator builds its own structure."""
    _check_against_dropin("skippfn", train_case="cigre14", val_case="cigre14_reswitched")


def test_evaluator_large_graph_path(tiny_tiles):
    _check_against_dropin("skippfn")


def test_training_is_unaffected_by_interleaved_evaluation():
    """Two trainers, same seed, SkipPFN with dropout: one runs captured evaluate / infer calls between its steps.  Loss trajectory,
    parameters, optimizer state and step counter stay identical."""
    from dss2.evaluator import GraphedEvaluator
    store = _store("ober_sub", 4 * B, seed=5)
    a = _trainer("skippfn", store, p_drop=0.3)
    b = _trainer("skippfn", store, p_drop=0.3)
    ev = GraphedEvaluator(store, B, trainer=b)
    batches = _batches(B, 2 * B + R)
    la, lb = [], []
    for s in range(5):
        ids = torch.arange(s, s + B, device="cuda") % store.num_scenarios
        la.append(a.step(ids).clone())
        lb.append(b.step(ids).clone())
        ev.evaluate(batches[s % 3])
        ev.infer(batches[(s + 1) % 3])
    assert ev.metrics()["batches"] == 5
    assert all(torch.equal(x, y) for x, y in zip(la, lb))
    for name in ("flat", "exp_avg", "exp_inf", "step_state"):
        assert torch.equal(getattr(a, name), getattr(b, name)), name


def test_multi_head_gat_evaluation_leaves_trainer_parameters_untouched():
    """GAT_DSSE with heads > 1: the runner's forward rewrites the constant blocks at the tail of the parameter buffer it reads.  The
    evaluator reads a private copy of the trainer's buffer, so its bytes - tail included, which the trainer's Adamax updates - stay
    as they are, and the result equals an evaluator that owns its parameters.  (A stand-in carries the three things the evaluator reads
    from a trainer: network, spec and flat.)"""
    import types
    from dss2.evaluator import GraphedEvaluator
    from dss2.gat import GATSpec
    store = _store("ober_sub", 2 * B + R, seed=5)
    spec = GATSpec(dim_feat=8, dim_dense=32, dim_out=2, num_layers=4, edge_dim=6, heads=2)
    table, size = spec.layout()
    g = torch.Generator(device="cuda").manual_seed(11)
    flat = torch.randn(size, device="cuda", generator=g) * 0.2
    sd = {k: flat[o:o + n].clone() for k, (o, n) in table.items() if not k.startswith("_")}
    tr = types.SimpleNamespace(network="gat", spec=spec, flat=flat)
    before = flat.clone()
    ev = GraphedEvaluator(store, B, trainer=tr)
    own = GraphedEvaluator(store, B, network="gat", spec=spec, state_dict=sd)
    batches = _batches(0, 2 * B + R)
    _same(_epoch(ev, batches), _epoch(own, batches))
    assert torch.equal(ev.infer(batches[-1])[0], own.infer(batches[-1])[0])
    assert torch.equal(flat, before)
    # the copy is refreshed on every call: a parameter update of the trainer shows in the next evaluation
    flat[table["model.module_0.lin_l.weight"][0]] += 1.0
    assert not torch.equal(ev.infer(batches[0])[0], own.infer(batches[0])[0])


def test_eval_mode_dropout_semantics():
    """SkipPFN keeps its dropout on in eval(): two inferences of the same batch differ, and both differ from p = 0.  GAT_DSSE's attention
    dropout is off in eval(): deterministic, equal to the model without dropout."""
    from dss2.evaluator import GraphedEvaluator
    from dss2.gat import GATSpec
    from dss2.trainer import default_spec
    store = _store("ober_sub", 2 * B, seed=5)
    tr = _trainer("skippfn", store, p_drop=0.3)
    sd = tr.state_dict()
    sel = torch.arange(B, device="cuda")
    ev = GraphedEvaluator(store, B, trainer=tr)
    o1 = ev.infer(sel)[0].clone()
    o2 = ev.infer(sel)[0].clone()
    o0 = GraphedEvaluator(store, B, network="skippfn", spec=default_spec(p_drop=0.0), state_dict=sd).infer(sel)[0]
    assert not torch.equal(o1, o2) and not torch.equal(o1, o0) and not torch.equal(o2, o0)
    tg = _trainer("gat", store, gat_dropout=0.3)
    gsd = tg.state_dict()
    eg = GraphedEvaluator(store, B, trainer=tg)
    g1 = eg.infer(sel)[0].clone()
    g2 = eg.infer(sel)[0].clone()
    spec0 = GATSpec(dim_feat=8, dim_dense=32, dim_out=2, num_layers=8, edge_dim=6, dropout=0.0)
    g0 = GraphedEvaluator(store, B, network="gat", spec=spec0, state_dict=gsd).infer(sel)[0]
    assert torch.equal(g1, g2) and torch.equal(g1, g0)


def test_no_host_synchronisation_after_capture_and_length_limits():
    from dss2 import _lib
    from dss2.evaluator import GraphedEvaluator
    store = _store("ober_sub", 4 * B, seed=5)
    tr = _trainer("skippfn", store, p_drop=0.3)
    ev = GraphedEvaluator(store, B, trainer=tr)
    batches = _batches(B, 2 * B + R)
    for sel in batches:          # first call per length: warm-up + capture
        ev.evaluate(sel)
        ev.infer(sel)
    ev.metrics()
    torch.cuda.synchronize()
    torch.cuda.set_sync_debug_mode("error")
    try:
        for sel in batches:
            ev.evaluate(sel)
            ev.infer(sel)
            tr.step(batches[0])
    finally:
        torch.cuda.set_sync_debug_mode(0)
    assert ev.metrics()["batches"] == 3
    for bad in (batches[0][:0], torch.arange(B + 1, device="cuda")):
        with pytest.raises(_lib.Dss2Error):
            ev.evaluate(bad)
        with pytest.raises(_lib.Dss2Error):
            ev.infer(bad)


# ---------------------------------------------------------------------------------------------- the device finaliser
def _python_formulas(s, n):
    """The script's per-batch metrics from the 19 sums of dss2_eval_metrics, in Python (fp64) - what the device finaliser reproduces."""
    def std(sx, sxx):
        return math.sqrt(max((sxx - sx * sx / n) / (n - 1.0), 0.0)) if n > 1 else float("nan")

    def ratio(a, b):
        return a / b if b != 0.0 else float("nan")

    sqrt = math.sqrt
    return [sqrt(s[0] / n), s[1] / n, sqrt(s[2] / n), s[3] / n, sqrt(ratio(s[13], s[12])), ratio(s[14], s[12]),
            sqrt(ratio(s[16], s[15])), ratio(s[17], s[15]), 100.0 * ratio(std(s[4], s[5]), std(s[8], s[9])),
            100.0 * ratio(std(s[6], s[7]), std(s[10], s[11]))]


def _bits_equal(got, want, what):
    for k, (g, w) in enumerate(zip(got, want)):
        assert g == w or (math.isnan(g) and math.isnan(w)), (what, k, g, w)


@pytest.mark.parametrize("case", ["ober_sub", "cigre14", "cigre14_reswitched"])
def test_device_finaliser_is_bit_exact(case):
    """dss2_eval_metrics_acc adds exactly the values the Python formulas give on dss2_eval_metrics' sums.  Every run is compared on its
    own (accumulator zeroed before it), so a NaN of one run cannot hide another run's value: full batches, where all ten metrics are
    finite (every grid has lines and a transformer), NaN exactly where a count is zero (no branch) or a std has a single bus.  Then the
    batch-after-batch accumulation of finite runs against the sequential Python sum."""
    from dss2 import _lib, batching
    lib = _lib.load()
    store = _store(case, 6, seed=3)
    ws = torch.zeros(lib.dss2_eval_workspace_bytes(), dtype=torch.uint8, device="cuda")
    g = torch.Generator(device="cuda").manual_seed(7)

    def run(sel, kind, acc):
        pb = batching.pack_batch(store, sel)
        nt, et = pb.x.size(0), pb.edge_index.size(1)
        if kind == "no_branch":
            et = 0
        elif kind == "one_bus":
            nt, et = 1, 0
        out = torch.randn(pb.x.size(0), 2, device="cuda", generator=g) * 0.05
        args = lambda dst: (_lib.ptr(pb.edge_index), nt, et, _lib.ptr(pb.x), 11, _lib.ptr(pb.edge_attr), 13, _lib.ptr(out), 2, _lib.ptr(pb.y), 2,
                            float(store.x_mean[0]), float(store.x_std[0]), _lib.ptr(pb.vminmax), _lib.ptr(dst), _lib.ptr(ws), ws.numel(),
                            _lib.stream())
        sums = torch.zeros(19, dtype=torch.float64, device="cuda")
        _lib.check(lib.dss2_eval_metrics(*args(sums)), "dss2_eval_metrics")
        _lib.check(lib.dss2_eval_metrics_acc(*args(acc)), "dss2_eval_metrics_acc")
        return _python_formulas(sums.cpu().tolist(), float(nt))

    nan_keys = {"full": set(), "no_branch": {4, 5, 6, 7}, "one_bus": {4, 5, 6, 7, 8, 9}}
    for sel, kind in [([0, 1, 2], "full"), ([3, 4, 5], "full"), ([0, 1, 2], "no_branch"), ([5], "one_bus")]:
        acc = torch.zeros(11, dtype=torch.float64, device="cuda")
        want = run(sel, kind, acc)
        got = acc.cpu().tolist()
        assert got[10] == 1.0
        assert {k for k in range(10) if math.isnan(want[k])} == nan_keys[kind], (kind, want)
        _bits_equal(got[:10], want, kind)
    # sequential accumulation over finite batches
    acc = torch.zeros(11, dtype=torch.float64, device="cuda")
    want = [0.0] * 10
    for sel in ([0, 1, 2], [3, 4, 5], [1, 4], [2, 3, 5, 0]):
        want = [w + v for w, v in zip(want, run(sel, "full", acc))]
    got = acc.cpu().tolist()
    assert got[10] == 4.0 and all(math.isfinite(w) for w in want), want
    assert got[:10] == want, (got, want)
