"""Runs the TEXT of the reference's training script (dss2_run.py) - only `epochs=600` -> `epochs=2` changed - once over the drop-in
modules of this repo (GPU kernels behind CPU tensors, exactly what a user switching over would do) and once over the reference's own
modules (verbatim copies in the git-ignored oracle/_ref, CPU), and compares what the script itself records: the per-epoch training
loss and every per-epoch validation metric (dss2_run.py:147,211-236).

Everything the script imports that this image lacks is supplied FROM tests/: `pandapower` (imported, never used), `torchmetrics`
(MeanAbsoluteError), and `torch_geometric` = oracle/pyg_shim on sys.path - which also makes `data.data_from_pickles` hand out
`torch_geometric.data.Data` objects that the script's own `torch_geometric.loader.DataLoader` collates (the route a real PyG install
takes).  The script draws its model from the global torch RNG; so that both runs start from the same weights and see the same
shuffles, `networks.GAT_DSSE` is wrapped (test infrastructure, the script text is untouched) to load one fixed state_dict and reseed.
"""
import importlib.util
import os
import pickle
import random
import sys
import types

import numpy as np
import pytest
import torch

from conftest import GOLDEN, PKG, ROOT

import dss2_oracle as orc

REF_DIR = os.path.join(ROOT, "oracle", "_ref")
SHIM = os.path.join(ROOT, "oracle", "pyg_shim")


def _script_text():
    path = os.path.join(REF_DIR, "dss2_run.py")
    if not os.path.exists(path):
        pytest.skip("the reference's dss2_run.py is not in oracle/_ref (build with DSS2_REFERENCE=<reference checkout>)")
    text = open(path).read()
    assert "epochs=600" in text
    return text.replace("epochs=600", "epochs=2"), path


def _write_pickles(root):
    """data/cigre14/{nodes,edges,labels,noise_param} in the reference's pickle layout from the 128-scenario fixture."""
    import pandas as pd
    sys.path.insert(0, PKG)
    from dss2 import synth
    fx = np.load(os.path.join(GOLDEN, "cigre14_scenarios.npz"), allow_pickle=False)
    folder = os.path.join(root, "data", "cigre14")
    os.makedirs(folder, exist_ok=True)
    nodes = [pd.DataFrame(a, columns=[str(c) for c in fx["node_cols"]]) for a in fx["nodes"]]
    edges = [pd.DataFrame(a, columns=[str(c) for c in fx["edge_cols"]]) for a in fx["edges"]]
    labels = [pd.DataFrame(a, columns=["vm_pu", "va_rad"]) for a in fx["labels"]]
    noise = pd.DataFrame([synth.load_grid("cigre14")["noise_param"]], index=["def_value"],
                         columns=["p_noise", "v_noise", "i_noise", "pm_noise", "sgen_noise", "zero_inj_coef"])
    for name, obj in (("nodes", nodes), ("edges", edges), ("labels", labels), ("noise_param", noise)):
        with open(os.path.join(folder, name), "wb") as fh:
            pickle.dump(obj, fh)


def _stub_modules():
    pp = types.ModuleType("pandapower")
    tm = types.ModuleType("torchmetrics")
    reg = types.ModuleType("torchmetrics.regression")

    class MeanAbsoluteError:          # torchmetrics.regression.MeanAbsoluteError as the script uses it (dss2_run.py:189-191)
        def __call__(self, pred, target):
            return (pred - target).abs().mean()

    reg.MeanAbsoluteError = MeanAbsoluteError
    tm.regression = reg
    return {"pandapower": pp, "torchmetrics": tm, "torchmetrics.regression": reg}


def _load(name, path):
    spec = importlib.util.spec_from_file_location(name, path)
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def _run(text, origin, modules, workdir, sd0):
    """exec the script with `modules` = {'networks','data','loadsampling'} installed under those names."""
    net = modules["networks"]
    wrapped = types.ModuleType("networks")
    wrapped.__dict__.update({k: v for k, v in net.__dict__.items() if not k.startswith("__")})
    real = net.GAT_DSSE

    def GAT_DSSE(*a, **kw):
        m = real(*a, **kw)
        m.load_state_dict(sd0, strict=True)
        torch.manual_seed(3)          # the loaders' shuffles follow from here in both runs
        return m

    wrapped.GAT_DSSE = GAT_DSSE
    installed = dict(_stub_modules(), networks=wrapped, data=modules["data"], loadsampling=modules["loadsampling"])
    saved = {k: sys.modules.get(k) for k in installed}
    cwd = os.getcwd()
    random.seed(1)
    np.random.seed(0)
    torch.manual_seed(2)
    ns = {"__name__": "__dss2_run__"}
    try:
        sys.modules.update(installed)
        os.chdir(workdir)
        exec(compile(text, origin, "exec"), ns)
    finally:
        os.chdir(cwd)
        for k, v in saved.items():
            if v is None:
                sys.modules.pop(k, None)
            else:
                sys.modules[k] = v
    return ns


LISTS = ("train_list", "rmse_v_list", "mae_v_list", "rmse_th_list", "mae_th_list", "rmse_loading_list", "mae_loading_list",
         "rmse_loading_trafos_list", "mae_loading_trafos_list", "prop_std_v_list", "prop_std_th_list")


@pytest.mark.gpu
def test_reference_script_text_runs_on_the_drop_in_modules(tmp_path):
    text, origin = _script_text()
    if not os.path.exists(os.path.join(REF_DIR, "networks.py")):
        pytest.skip("oracle/_ref is empty: no reference modules to compare with")
    if SHIM not in sys.path:
        sys.path.insert(0, SHIM)
    _write_pickles(str(tmp_path))
    sd0 = orc.init_gat_state_dict(num_layers=8, seed=12)
    import data as our_data
    import loadsampling as our_ls
    import networks as our_net
    ours = _run(text, origin, {"networks": our_net, "data": our_data, "loadsampling": our_ls}, str(tmp_path), sd0)
    assert type(ours["dataset"][0]).__module__.startswith("torch_geometric"), "data_from_pickles must hand out torch_geometric Data objects"
    ck = torch.load(os.path.join(str(tmp_path), "gat.pt"), weights_only=False)            # dss2_run.py:240-247, written by OUR run
    ref_mods = {n: _load(f"_dss2_script_ref_{n}", os.path.join(REF_DIR, f"{n}.py")) for n in ("networks", "data", "loadsampling")}
    theirs = _run(text, origin, ref_mods, str(tmp_path), sd0)
    for name in LISTS:
        print(f"{name:26s} ours {ours[name]}  reference {theirs[name]}")
    print("stats ours", [t.tolist() for t in (ours["x_mean"], ours["x_std"], ours["pflow_mean"], ours["pflow_std"])])
    print("stats ref ", [t.tolist() for t in (theirs["x_mean"], theirs["x_std"], theirs["pflow_mean"], theirs["pflow_std"])])
    d0, r0 = ours["dataset"][0], theirs["dataset"][0]
    print("graph0 equal:", torch.equal(d0.x, r0.x), torch.equal(d0.edge_attr, r0.edge_attr), torch.equal(d0.edge_index, r0.edge_index), torch.equal(d0.y, r0.y))
    assert len(ours["train_list"]) == 2 and len(theirs["train_list"]) == 2
    # two epochs = four Adamax steps from identical weights, batches and shuffles.  Adamax divides by a running max of |grad|, so fp32
    # rounding differences in near-zero gradient entries become +-lr parameter differences: 1e-3-level drift after a few steps is
    # what two correct fp32 implementations show (tests/test_gpu_parity.py::test_dss2_run_flow_with_default_gat_model measures it)
    for name in LISTS:
        a, b = np.asarray(ours[name]), np.asarray(theirs[name])
        assert a.shape == b.shape == (2,), name
        assert np.allclose(a, b, rtol=2e-2, atol=1e-7), (name, a, b)
    assert abs(ours["train_list"][0] - theirs["train_list"][0]) <= 2e-3 * abs(theirs["train_list"][0]), (ours["train_list"], theirs["train_list"])
    # checkpoints interchange: the script's own torch.save of OUR model loads into the reference's model
    ref_model = ref_mods["networks"].GAT_DSSE(dim_feat=8, dim_dense=32, dim_out=2, heads=1, num_layers=8, edge_dim=6)
    ref_model.load_state_dict(ck["model_state_dict"], strict=True)
