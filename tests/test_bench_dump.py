"""bench.py --dump-outputs: what the last timed step computed, written as .npy files for comparing two builds output for output."""
import hashlib
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from conftest import ROOT

import bench


def test_dump_outputs_dtypes_and_seeded_sample(tmp_path, monkeypatch):
    monkeypatch.setattr(bench, "DUMP_BUDGET", 4000)
    big = torch.randn(1000, 2)
    arrays = {"big": big, "small": torch.arange(5, dtype=torch.int32), "loss": torch.tensor(2.5, dtype=torch.float64)}
    bench.dump_outputs(str(tmp_path / "a"), arrays)
    bench.dump_outputs(str(tmp_path / "b"), arrays)
    got = {n: np.load(tmp_path / "a" / f"{n}.npy") for n in arrays}
    assert got["loss"].dtype == np.float64 and got["loss"] == 2.5
    assert got["small"].dtype == np.float32 and got["small"].tolist() == [0, 1, 2, 3, 4]
    # over budget: the large array keeps a seeded sample of its rows, in order, the same in every run
    assert sum(a.nbytes for a in got.values()) <= 4000 and 0 < got["big"].shape[0] < 1000 and got["big"].shape[1] == 2
    rows = [int(np.flatnonzero((big.numpy() == r).all(1))[0]) for r in got["big"]]
    assert rows == sorted(rows)
    assert all(np.array_equal(got[n], np.load(tmp_path / "b" / f"{n}.npy")) for n in arrays)


def _bench(tmp_path, *args):
    """bench.py on the cigre14 config with --dump-outputs: (its JSON line, {name: array} of the dump)."""
    out = tmp_path / "dump"
    run = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--config", "cigre14", "--warmup", "3", "--no-e2e",
                          "--no-cpu-baseline", "--dump-outputs", str(out), *args], capture_output=True, text=True, cwd=str(tmp_path), timeout=600)
    assert run.returncode == 0, run.stderr[-2000:]
    return json.loads(run.stdout.strip().splitlines()[-1]), {f[:-len(".npy")]: np.load(out / f) for f in sorted(os.listdir(out))}


def _num_parameters(network):
    import networks
    if network == "gat":
        model = networks.GAT_DSSE(dim_feat=8, dim_dense=32, dim_out=2, heads=1, num_layers=8, edge_dim=6)
    else:
        model = networks.SkipPFN(dim_featn=8, dim_feate=6, dim_out=2, dim_hid=32, n_gnn_layers=8, K=2, dropout_rate=0.3, L=5)
    return sum(p.numel() for p in model.parameters())


@pytest.mark.gpu
@pytest.mark.parametrize("network", ["skippfn", "gat"])
def test_bench_dumps_the_last_timed_training_step(tmp_path, network):
    steps = 3
    line, dump = _bench(tmp_path, "--network", network, "--steps", str(steps))
    assert sorted(dump) == ["loss", "loss_per_step", "parameters"] and all(a.dtype == np.float32 for a in dump.values())
    assert line["steps"] == steps and dump["loss_per_step"].shape == (steps,)
    assert hashlib.sha256(dump["loss_per_step"].tobytes()).hexdigest()[:16] == line["loss_trajectory_sha256_16"]
    assert dump["loss"].shape == () and float(dump["loss"]) == line["final_loss"] == float(dump["loss_per_step"][-1])
    assert dump["parameters"].shape == (_num_parameters(network),) and np.isfinite(dump["parameters"]).all()


@pytest.mark.gpu
def test_bench_dumps_the_last_timed_inference_step(tmp_path):
    line, dump = _bench(tmp_path, "--mode", "infer", "--steps", "2")
    cfg = line["config"]
    assert sorted(dump) == ["output", "pflow"] and all(a.dtype == np.float32 for a in dump.values())
    assert dump["output"].shape == (cfg["nodes_per_step_per_gpu"], 2)
    assert dump["pflow"].shape == (cfg["edges_per_step_per_gpu"], 8) and np.isfinite(dump["pflow"]).all()
