"""train_models(seeds=[...]) trains every seed as one model batch; each seed's checkpoints (parameters and optimizer state) and
metrics must equal bit for bit what train_model(seed=s) writes for it."""
import json
import os

import numpy as np
import pytest
import torch

from ms_hgnn import morphology as M
from test_com_grf_metrics import _stats_dir

pytestmark = pytest.mark.gpu
DEV = torch.device("cuda:0") if torch.cuda.is_available() else None


def _same_runs(path_a, path_b):
    names_a = sorted(c for c in os.listdir(path_a) if c.endswith(".ckpt"))
    assert names_a == sorted(c for c in os.listdir(path_b) if c.endswith(".ckpt")) and names_a
    for c in names_a:
        a = torch.load(os.path.join(path_a, c), weights_only=False)
        b = torch.load(os.path.join(path_b, c), weights_only=False)
        assert a["epoch"] == b["epoch"] and a["global_step"] == b["global_step"]
        assert a["state_dict"].keys() == b["state_dict"].keys()
        for k in a["state_dict"]:
            assert torch.equal(a["state_dict"][k], b["state_dict"][k]), (c, k)
        sa, sb = a["optimizer_states"][0], b["optimizer_states"][0]
        assert sa["param_groups"] == sb["param_groups"] and sa["state"].keys() == sb["state"].keys() and sa["state"]
        for i in sa["state"]:
            for k in ("step", "exp_avg", "exp_avg_sq"):
                assert torch.equal(sa["state"][i][k], sb["state"][i][k]), (c, i, k)
    rows = lambda p: [json.loads(l) for l in open(os.path.join(p, "metrics.jsonl"))]
    assert rows(path_a) == rows(path_b)


def _check(tmp_path, monkeypatch, tr, va, te, kw):
    from ms_hgnn.lightning_py.gnnLightning import train_model, train_models
    monkeypatch.chdir(tmp_path)
    paths = train_models(tr, va, te, seeds=[0, 5], mode="tc", **kw)
    assert len(paths) == 2 and paths[0] != paths[1]
    for seed, p in zip((0, 5), paths):
        _same_runs(p, train_model(tr, va, te, seed=seed, mode="tc", **kw))


def test_train_models_mini_cheetah_contact(tmp_path, monkeypatch):
    import window_oracle as WO
    from ms_hgnn.lightning_py.gnnLightning import WindowSubset
    from ms_hgnn.windows import DeviceSequence, WindowSpec
    mat = WO.synthetic_mat(800, seed=21, dtype=np.float32)
    mat["contacts"] = (mat["qd"][:, [2, 5, 8, 11]] > 0).astype(np.float32)
    ds = DeviceSequence(mat, WindowSpec("heterogeneous_gnn_k4", 150, True), DEV, torch.float32)
    tr, va, te = WindowSubset(ds, torch.arange(0, 400)), WindowSubset(ds, torch.arange(400, 520)), WindowSubset(ds, torch.arange(520, len(ds)))
    kw = dict(normalize=True, testing_mode=True, disable_logger=True, batch_size=64, num_layers=2, optimizer="adam", lr=1e-3,
              hidden_size=16, regression=False, epochs=3, symmetry_mode="MorphSym", group_operator_path=M.cfg_path("mini_cheetah-k4"))
    _check(tmp_path, monkeypatch, tr, va, te, kw)


def test_train_models_com(tmp_path, monkeypatch):
    import window_oracle as WO
    from ms_hgnn.lightning_py.gnnLightning import WindowSubset
    from ms_hgnn.windows import DeviceSequence, WindowSpec
    mat = WO.synthetic_solo_mat(1200, seed=31)
    data = _stats_dir(tmp_path, mat["y_mean"], mat["y_std"])
    ds = DeviceSequence(mat, WindowSpec("heterogeneous_gnn_k4_com", 1, True, dataset="solo12"), DEV, torch.float32)
    tr, va, te = WindowSubset(ds, torch.arange(0, 800)), WindowSubset(ds, torch.arange(800, 1000)), WindowSubset(ds, torch.arange(1000, len(ds)))
    kw = dict(normalize=True, testing_mode=True, disable_logger=True, batch_size=64, num_layers=2, optimizer="adam", lr=1e-3,
              hidden_size=16, epochs=3, data_path=data, symmetry_mode="MorphSym", group_operator_path=M.cfg_path("solo12-k4"))
    _check(tmp_path, monkeypatch, tr, va, te, kw)
