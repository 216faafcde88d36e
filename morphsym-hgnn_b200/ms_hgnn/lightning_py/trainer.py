"""``train_model`` / ``evaluate_model`` re-hosted on the native engine (SURVEY 8f-1).

Drop-in for ``gnnLightning.py:L913-1095`` (``evaluate_model``) and ``L1099-1421`` (``train_model``): same keyword
arguments, same return values, the reference's checkpoint policy (``ModelCheckpoint`` top-7 by ``val_CE_loss`` /
``val_MSE_loss`` plus the 3 latest epochs, file names ``epoch=E-val_CE_loss=0.12345-val_F1_Score_Leg_Avg=0.98765.ckpt``,
``EarlyStopping(patience=10)``, resume from ``ckpt_path``) and a checkpoint layout a Lightning user recognises
(``state_dict`` with the ``model.`` prefix, ``hyper_parameters``, ``epoch``, ``global_step``, ``optimizer_states`` in
``torch.optim.Adam.state_dict()`` form).  Differences, all forced by the environment or by the device-side data path:

* ``lightning.Trainer`` / ``WandbLogger`` are not installed: the epoch loop below plays the trainer; metrics go to
  ``<path_to_save>/metrics.jsonl`` instead of W&B (``disable_logger=False`` still requires ``logger_project_name``).
* datasets are ``WindowSubset``s of a ``DeviceSequence`` (ms_hgnn.windows) instead of ``torch.utils.data.Subset``s of a
  ``FlexibleDataset``: a batch is a tensor of window indices and is collated on the GPU.
* the optimisation step is the fused native step (``FusedTrainer``), not autograd + ``torch.optim``.

Centre-of-mass momentum (the Solo12 formats ``heterogeneous_gnn_{k4,c2,s4}_com``) goes through the same loops with
``COM_HGNN_SYM_Lightning(model_type=<format>, data_path=data_path)``; ``data_path/processed/rss_stats.npz`` supplies the
label standardiser when it exists.  Three choices for COM could not be checked against the reference's own code and follow
the regression branch of these loops: the monitor ``val_MSE_loss``, the checkpoint name ``epoch=E-val_MSE_loss=x.xxxxx.ckpt``
(no second metric: COM logs no ``val_L1_loss``) and ``evaluate_model``'s return tuple ``(pred, labels, mse, rmse, mse_lin,
mse_ang, cos_sim_lin, cos_sim_ang)``, in the order ``COM_Base_Lightning`` computes them.
"""
from __future__ import annotations

import json
import os
import time
from pathlib import Path
from typing import List, Optional

import torch

from .. import _native as N
from ..synthetic import HeteroBatch
from ..train import FusedTrainer

_HGNN_FORMATS = ("heterogeneous_gnn", "heterogeneous_gnn_k4", "heterogeneous_gnn_c2")
_COM_FORMATS = ("heterogeneous_gnn_k4_com", "heterogeneous_gnn_c2_com", "heterogeneous_gnn_s4_com")


class WindowSubset:
    """``torch.utils.data.Subset`` of a device-resident sequence: ``dataset`` + the entries it may draw."""

    def __init__(self, dataset, indices):
        self.dataset = dataset
        self.indices = torch.as_tensor(indices, dtype=torch.int64).reshape(-1)
        if self.indices.numel() and (int(self.indices.min()) < 0 or int(self.indices.max()) >= len(dataset)):
            raise IndexError("subset index out of range")

    def __len__(self) -> int:
        return int(self.indices.numel())


def _loader(subset: WindowSubset, batch_size: int, shuffle: bool, generator: Optional[torch.Generator], limit: Optional[int]):
    """Index batches in DataLoader order (``shuffle`` draws a fresh permutation per epoch; the last batch may be short)."""
    idx = subset.indices
    if shuffle:
        idx = idx[torch.randperm(idx.numel(), generator=generator)]
    chunks = list(torch.split(idx, batch_size))
    return chunks[:limit] if limit is not None else chunks


def _build_module(model_type, hidden_size, num_layers, data_metadata, dummy_batch, optimizer, lr, regression, symmetry_mode,
                  group_operator_path, grf_body_to_world_frame, grf_dimension, data_path):
    from . import gnnLightning as G
    if model_type in _COM_FORMATS:
        from .gnnLightning_com import COM_HGNN_SYM_Lightning
        return COM_HGNN_SYM_Lightning(hidden_channels=hidden_size, num_layers=num_layers, data_metadata=data_metadata,
                                      dummy_batch=dummy_batch, optimizer=optimizer, lr=lr, symmetry_mode=symmetry_mode,
                                      group_operator_path=group_operator_path, model_type=model_type, data_path=data_path)
    if model_type == "heterogeneous_gnn":
        return G.Heterogeneous_GNN_Lightning(hidden_channels=hidden_size, num_layers=num_layers, data_metadata=data_metadata,
                                             dummy_batch=dummy_batch, optimizer=optimizer, lr=lr, regression=regression,
                                             grf_dimension=1)
    if model_type == "heterogeneous_gnn_k4":
        return G.HGNN_K4_Lightning(hidden_channels=hidden_size, num_layers=num_layers, data_metadata=data_metadata,
                                   dummy_batch=dummy_batch, optimizer=optimizer, lr=lr, regression=regression,
                                   symmetry_mode=symmetry_mode, group_operator_path=group_operator_path)
    if model_type == "heterogeneous_gnn_c2":
        if regression:
            return G.HGNN_C2_Lightning_Reg(hidden_channels=hidden_size, num_layers=num_layers, data_metadata=data_metadata,
                                           dummy_batch=dummy_batch, optimizer=optimizer, lr=lr, regression=regression,
                                           symmetry_mode=symmetry_mode, group_operator_path=group_operator_path,
                                           grf_body_to_world_frame=grf_body_to_world_frame, grf_dimension=grf_dimension)
        return G.HGNN_C2_Lightning_Cls(hidden_channels=hidden_size, num_layers=num_layers, data_metadata=data_metadata,
                                       dummy_batch=dummy_batch, optimizer=optimizer, lr=lr, regression=regression,
                                       symmetry_mode=symmetry_mode, group_operator_path=group_operator_path)
    raise ValueError("Invalid model type.")


def _plain_batch(b: HeteroBatch) -> dict:
    """A pickle-friendly copy of a (small) batch for ``hyper_parameters['dummy_batch']``."""
    return {"x": {k: v.detach().cpu() for k, v in b.x_dict.items()},
            "edge_index": {k: v.detach().cpu() for k, v in b.edge_index_dict.items()},
            "y": b.y.detach().cpu(), "batch_size": b.batch_size}


def _adam_state(trainer: FusedTrainer, module) -> dict:
    """The fused optimizer's flat moments in ``torch.optim.Adam.state_dict()`` form (parameter order = named_parameters())."""
    state, off = {}, 0
    params = list(module.parameters())
    if trainer.exp_avg is not None:
        for i, p in enumerate(params):
            n = p.numel()
            state[i] = {"step": torch.tensor(float(trainer.step_count)),
                        "exp_avg": trainer.exp_avg[off:off + n].reshape(p.shape).cpu().clone(),
                        "exp_avg_sq": trainer.exp_avg_sq[off:off + n].reshape(p.shape).cpu().clone()}
            off += n
    return {"state": state, "param_groups": [{"lr": trainer.lr, "betas": tuple(trainer.betas), "eps": trainer.eps,
                                               "weight_decay": trainer.weight_decay, "amsgrad": False,
                                               "params": list(range(len(params)))}]}


def _load_adam_state(trainer: FusedTrainer, module, opt_state: dict, device) -> None:
    st = opt_state.get("state", {})
    if not st:
        return
    n = sum(p.numel() for p in module.parameters())
    trainer.grads = torch.empty(n, dtype=torch.float32, device=device)
    trainer.exp_avg = torch.zeros(n, dtype=torch.float32, device=device)
    trainer.exp_avg_sq = torch.zeros(n, dtype=torch.float32, device=device)
    off = 0
    for i, p in enumerate(module.parameters()):
        k = p.numel()
        if i in st:
            trainer.exp_avg[off:off + k] = st[i]["exp_avg"].reshape(-1).to(device, torch.float32)
            trainer.exp_avg_sq[off:off + k] = st[i]["exp_avg_sq"].reshape(-1).to(device, torch.float32)
            trainer.step_count = int(float(st[i]["step"]))
        off += k


def _save_checkpoint(path: Path, module, trainer: FusedTrainer, epoch: int, global_step: int, dummy: dict, loop_state: dict = None) -> None:
    hp = {k: v for k, v in dict(module.hparams).items() if k not in ("dummy_batch", "activation_fn")}
    hp["dummy_batch"] = dummy
    torch.save({"epoch": epoch, "global_step": global_step, "pytorch-lightning_version": "mshgnn_b200",
                "loop_state": loop_state,       # early-stopping / top-k bookkeeping and the shuffle generator (Lightning keeps them under "callbacks" / "loops")
                "state_dict": {k: v.detach().cpu() for k, v in module.state_dict().items()},
                "optimizer_states": [_adam_state(trainer, module)], "lr_schedulers": [], "hyper_parameters": hp,
                "class": type(module).__name__}, str(path))


def _value(v) -> float:
    return float(v.item()) if torch.is_tensor(v) else float(v)


def _run_epoch(module, dataset, batches, kind: str):
    getattr(module, f"on_{kind}_epoch_start")()
    step = getattr(module, f"{kind}_step")
    with torch.no_grad():
        for bi, idx in enumerate(batches):
            step(dataset.batch(idx), bi)
    getattr(module, f"on_{kind}_epoch_end")()
    return {k: _value(v) for k, v in module.logged.items() if k.startswith(("val_" if kind == "validation" else kind + "_"))}


class _Run:
    """One seed's training run: its module, shuffle generator, checkpoint folder, metrics log and the early-stopping / top-k
    bookkeeping of the reference's callbacks."""

    def __init__(self, train_dataset, model_type, com, data_metadata, seed, batch_size, normalize, hidden_size, num_layers, optimizer, lr,
                 regression, symmetry_mode, group_operator_path, grf_body_to_world_frame, grf_dimension, data_path,
                 disable_logger, logger_project_name, subfoler_name, train_percentage_to_log):
        torch.manual_seed(seed)                                    # seed_everything(seed)
        self.gen = torch.Generator().manual_seed(seed)
        self.ds = ds = train_dataset.dataset
        dummy_idx = _loader(train_dataset, batch_size, True, self.gen, 1)[0]
        dummy_batch = ds.batch(dummy_idx)
        self.module = module = _build_module(model_type, hidden_size, num_layers, data_metadata, dummy_batch, optimizer, lr, regression,
                                             symmetry_mode, group_operator_path, grf_body_to_world_frame, grf_dimension, data_path).to(ds.device)
        module.model.validate_edges = "cached"
        n_params = sum(p.numel() for p in module.model.parameters() if p.requires_grad)

        if not disable_logger:
            if logger_project_name is None:
                raise ValueError("Need to define \"logger_project_name\" if logger is enabled.")
            path_to_save = Path("models", subfoler_name, f"{logger_project_name}-seed{seed}-{time.strftime('%Y%m%d-%H%M%S')}")
        else:
            path_to_save = Path("models", f"{model_type}_run-seed{seed}-{time.strftime('%Y%m%d-%H%M%S')}")
        base, k = path_to_save, 0
        while path_to_save.exists():                               # two runs inside the same second
            k += 1
            path_to_save = Path(str(base) + f"-{k}")
        path_to_save.mkdir(parents=True)
        self.path = path_to_save
        self.log_f = open(path_to_save / "metrics.jsonl", "a")
        self.log_f.write(json.dumps({"config": {"batch_size": batch_size, "normalize": normalize, "num_parameters": n_params, "seed": seed,
                                                "train_percentage": train_percentage_to_log, "model_type": model_type}}) + "\n")
        if regression or com:
            self.monitor, self.second = "val_MSE_loss", "val_L1_loss"
        else:
            self.monitor, self.second = "val_CE_loss", "val_F1_Score_Leg_Avg"
        self.dummy_idx = dummy_idx
        self.saved: List[tuple] = []        # (epoch, monitor value, path)
        self.best_seen, self.bad_epochs = float("inf"), 0
        self.stopped = False

    def start(self):
        self.dummy_plain = _plain_batch(self.ds.batch(self.dummy_idx[:min(20, self.dummy_idx.numel())]))

    def resume(self, resumed) -> None:
        """early stopping, the top-k policy and the shuffle order continue where the run stopped"""
        self.best_seen, self.bad_epochs = float(resumed["best_seen"]), int(resumed["bad_epochs"])
        self.saved = [(int(e), float(v), Path(pth)) for e, v, pth in resumed["saved"] if Path(pth).exists()]
        self.gen.set_state(resumed["generator_state"])

    def end_epoch(self, trainer, val_dataset, batch_size, lim_val, epoch, global_step, loss, early_stopping) -> None:
        """Validation, metrics line, checkpoint and the top-k / early-stopping policy after a training epoch."""
        module, monitor, second = self.module, self.monitor, self.second
        module.eval()
        _run_epoch(module, val_dataset.dataset, _loader(val_dataset, batch_size, False, None, lim_val), "validation")
        logged = {k: _value(v) for k, v in module.logged.items() if k.startswith("val_")}
        logged.update(epoch=epoch, global_step=global_step, train_loss_last_step=_value(loss))
        self.log_f.write(json.dumps(logged) + "\n"); self.log_f.flush()
        name = f"epoch={epoch}-{monitor}={logged[monitor]:.5f}" + (f"-{second}={logged[second]:.5f}" if second in logged else "") + ".ckpt"
        saved = self.saved
        saved.append((epoch, logged[monitor], self.path / name))
        better = logged[monitor] < self.best_seen
        _save_checkpoint(self.path / name, module, trainer, epoch, global_step, self.dummy_plain,
                         {"best_seen": min(self.best_seen, logged[monitor]), "bad_epochs": 0 if better else self.bad_epochs + 1,
                          "saved": [(e, v, str(pth)) for e, v, pth in saved], "generator_state": self.gen.get_state()})
        # ModelCheckpoint(save_top_k=7, mode='min', monitor=monitor) + ModelCheckpoint(save_top_k=3, mode='max', monitor='epoch')
        keep = {s[2] for s in sorted(saved, key=lambda s: s[1])[:7]} | {s[2] for s in sorted(saved, key=lambda s: s[0])[-3:]}
        for s in saved:
            if s[2] not in keep and s[2].exists():
                s[2].unlink()
        self.saved = [s for s in saved if s[2] in keep]
        if logged[monitor] < self.best_seen:
            self.best_seen, self.bad_epochs = logged[monitor], 0
        else:
            self.bad_epochs += 1
        if early_stopping and self.bad_epochs >= 10:                # EarlyStopping(monitor, patience=10, mode='min')
            self.stopped = True

    def finish(self, test_dataset, batch_size, lim_test, disable_test) -> str:
        if not disable_test:
            logged = _run_epoch(self.module, test_dataset.dataset, _loader(test_dataset, batch_size, False, None, lim_test), "test")
            self.log_f.write(json.dumps(logged) + "\n")
        self.log_f.close()
        return str(self.path)


def _check_run_args(train_dataset, val_dataset, test_dataset, disable_test, hidden_size, devices):
    fmts = [train_dataset.dataset.get_data_format(), val_dataset.dataset.get_data_format()]
    if not disable_test:
        fmts.append(test_dataset.dataset.get_data_format())
    if len(set(fmts)) != 1:
        raise ValueError("Data formats of datasets don't match")
    model_type = fmts[0]
    if model_type not in _HGNN_FORMATS + _COM_FORMATS:
        raise ValueError("Invalid model type.")
    if not 1 <= hidden_size <= 128:
        # narrower models run zero-padded on the 128-channel kernels; wider ones have no kernels
        raise ValueError(f"hidden_size={hidden_size}: the B200-native path supports hidden_size 1..128")
    if devices != 1:
        raise ValueError("train_model drives one GPU; launch one process per GPU and pass a process group to FusedTrainer for data parallelism")
    return model_type, model_type in _COM_FORMATS


def train_model(train_dataset: WindowSubset, val_dataset: WindowSubset, test_dataset: Optional[WindowSubset], normalize: bool,
                testing_mode: bool = False, disable_logger: bool = False, logger_project_name: str = None, batch_size: int = 100,
                num_layers: int = 8, optimizer: str = "adam", lr: float = 0.003, epochs: int = 30, hidden_size: int = 10,
                regression: bool = True, seed: int = 0, devices: int = 1, early_stopping: bool = False, disable_test: bool = False,
                train_percentage_to_log=None, symmetry_mode: str = None, group_operator_path: str = None,
                subfoler_name: str = "default", data_path: Path = None, wandb_api_key: str = None,
                grf_body_to_world_frame: bool = True, grf_dimension: int = 3, ckpt_path: str = None, mode: str = "fp32") -> str:
    """Train with the reference's ``train_model`` contract (gnnLightning.py:L1099-1421).  Returns the checkpoint folder.
    ``mode``: arithmetic mode of the native kernels ('fp32', 'tc' or 'tc1x', ``NativeHGNN.set_mode``).

    COM formats build ``COM_HGNN_SYM_Lightning`` (a regression model whatever ``regression`` says) and monitor ``val_MSE_loss``;
    ``data_path`` is where its standardiser statistics are looked up (module docstring: what is not checked against the
    reference)."""
    model_type, com = _check_run_args(train_dataset, val_dataset, test_dataset, disable_test, hidden_size, devices)
    data_metadata = train_dataset.dataset.get_data_metadata()
    lim_train, lim_val, lim_test = (10, 5, 5) if testing_mode else (None, None, None)
    run = _Run(train_dataset, model_type, com, data_metadata, seed, batch_size, normalize, hidden_size, num_layers, optimizer, lr,
               regression, symmetry_mode, group_operator_path, grf_body_to_world_frame, grf_dimension, data_path,
               disable_logger, logger_project_name, subfoler_name, train_percentage_to_log)
    module, ds = run.module, run.ds
    module.model.set_mode(mode)

    trainer = FusedTrainer(module)
    start_epoch, global_step = 0, 0
    if ckpt_path is not None and os.path.exists(ckpt_path):
        from ..checkpoint import load_checkpoint
        ck = load_checkpoint(ckpt_path, "cpu")
        module.load_state_dict(ck["state_dict"], strict=False)
        module.to(ds.device)
        if ck.get("optimizer_states"):
            _load_adam_state(trainer, module, ck["optimizer_states"][0], ds.device)
        start_epoch, global_step = int(ck.get("epoch", -1)) + 1, int(ck.get("global_step", 0))
        resumed = ck.get("loop_state")
    else:
        resumed = None

    run.start()
    if resumed:
        run.resume(resumed)
    loss = torch.zeros(())
    for epoch in range(start_epoch, epochs):
        module.train()
        for idx in _loader(train_dataset, batch_size, True, run.gen, lim_train):
            loss = trainer.train_step(ds.batch(idx))
            global_step += 1
        run.end_epoch(trainer, val_dataset, batch_size, lim_val, epoch, global_step, loss, early_stopping)
        if run.stopped:
            break
    return run.finish(test_dataset, batch_size, lim_test, disable_test)


class _SeedOptimizerView:
    """Model ``i`` of a ModelBatchTrainer seen as a FusedTrainer by the checkpoint writer (its moments, step count, settings)."""

    def __init__(self, tr, i):
        self.exp_avg, self.exp_avg_sq = tr.exp_avg[i], tr.exp_avg_sq[i]
        self.step_count = tr.step_count[i]
        self.lr, self.betas, self.eps, self.weight_decay = tr.lr[i], tr.betas, tr.eps, tr.weight_decay


def _per_run(value, name: str, n: int) -> list:
    """A scalar for every run, or a sequence of one value per run."""
    if isinstance(value, (str, bytes)) or not hasattr(value, "__len__"):
        return [value] * n
    values = list(value)
    if len(values) != n:
        raise ValueError(f"{name} has {len(values)} entries for {n} runs (one per seed expected)")
    return values


def train_models(train_dataset: WindowSubset, val_dataset: WindowSubset, test_dataset: Optional[WindowSubset], normalize: bool,
                 testing_mode: bool = False, disable_logger: bool = False, logger_project_name: str = None, batch_size: int = 100,
                 num_layers: int = 8, optimizer: str = "adam", lr=0.003, epochs: int = 30, hidden_size=10,
                 regression: bool = True, seeds=(0,), devices: int = 1, early_stopping: bool = False, disable_test: bool = False,
                 train_percentage_to_log=None, symmetry_mode: str = None, group_operator_path: str = None,
                 subfoler_name: str = "default", data_path: Path = None, wandb_api_key: str = None,
                 grf_body_to_world_frame: bool = True, grf_dimension: int = 3, mode: str = "tc") -> List[str]:
    """``train_model`` for several runs at once: returns one checkpoint folder per run, each with what
    ``train_model(seed=s, hidden_size=h, lr=l)`` writes for that run - bit for bit the same checkpoints (parameters and
    optimizer state) and metrics.

    Run i is ``(seeds[i], hidden_size[i], lr[i])``: ``hidden_size`` and ``lr`` are a value for every run or a sequence as long
    as ``seeds`` (a seed may repeat), so one call trains a sweep over widths and learning rates.  Every run is built exactly as
    ``train_model`` builds it (global seed, its own shuffle generator, dummy batch, module); the training steps of all runs run
    as one model batch (``ModelBatchTrainer``, arithmetic ``mode`` 'tc' or 'tc1x', which every run's module uses for
    validation and test too); validation, test, checkpoints, top-k and early stopping stay per run.  A run that has stopped
    early still rides along in the batched step but gets no optimizer update and writes nothing more.  Resuming
    (``ckpt_path`` of ``train_model``) is not offered."""
    from ..model_batch import ModelBatch, ModelBatchTrainer
    seeds = list(seeds)
    if not seeds:
        raise ValueError("train_models needs at least one seed")
    hidden_sizes = _per_run(hidden_size, "hidden_size", len(seeds))
    lrs = _per_run(lr, "lr", len(seeds))
    for h in hidden_sizes:
        model_type, com = _check_run_args(train_dataset, val_dataset, test_dataset, disable_test, h, devices)
    data_metadata = train_dataset.dataset.get_data_metadata()
    lim_train, lim_val, lim_test = (10, 5, 5) if testing_mode else (None, None, None)
    runs = [_Run(train_dataset, model_type, com, data_metadata, seed, batch_size, normalize, h, num_layers, optimizer, l,
                 regression, symmetry_mode, group_operator_path, grf_body_to_world_frame, grf_dimension, data_path,
                 disable_logger, logger_project_name, subfoler_name, train_percentage_to_log) for seed, h, l in zip(seeds, hidden_sizes, lrs)]
    for r in runs:
        r.module.model.set_mode(mode)
        r.start()
    m0 = runs[0].module
    # the settings FusedTrainer(module) takes from each module
    tr = ModelBatchTrainer(ModelBatch([r.module.model for r in runs], mixed_hidden=True), optimizer=getattr(m0, "optimizer", "adam"),
                           lr=[float(getattr(r.module, "lr", 1e-3)) for r in runs],
                           regression=getattr(m0, "regression", getattr(m0.model, "regression", True)))
    ds = runs[0].ds
    global_step = 0
    losses = [torch.zeros(())] * len(runs)
    for epoch in range(epochs):
        live = [not r.stopped for r in runs]
        if not any(live):
            break
        for r in runs:
            r.module.train()
        loaders = [_loader(train_dataset, batch_size, True, r.gen, lim_train) for r in runs]
        for step in range(len(loaders[0])):
            loss = tr.train_step([ds.batch(ld[step]) for ld in loaders], active=live)
            losses = [loss[i] if live[i] else losses[i] for i in range(len(runs))]
            global_step += 1
        for i, r in enumerate(runs):
            if live[i]:
                r.end_epoch(_SeedOptimizerView(tr, i), val_dataset, batch_size, lim_val, epoch, global_step, losses[i], early_stopping)
    return [r.finish(test_dataset, batch_size, lim_test, disable_test) for r in runs]


def evaluate_model(path_to_checkpoint: Path, predict_dataset: WindowSubset, enable_testing_mode: bool = False,
                   symmetry_mode: str = None, group_operator_path: str = None, data_path: Path = None,
                   grf_body_to_world_frame: bool = False, grf_dimension: int = 1, test_only_on_z: bool = False,
                   batch_size: int = 100, task_type: str = "regression"):
    """Run a checkpoint over ``predict_dataset`` (gnnLightning.py:L913-1095): returns ``(pred, labels, *metrics)`` -
    classification: 16-class predictions / labels, accuracy, F1 of the four legs and their average; regression: predictions,
    labels, MSE, RMSE, L1; COM: predictions, labels, MSE, RMSE, lin MSE, ang MSE, lin and ang cosine similarity.  Works on
    reference checkpoints (``epoch=..ckpt`` from Lightning) and on ``train_model``'s.  For COM, ``data_path`` (when given)
    replaces the one stored in the checkpoint as the place of ``processed/rss_stats.npz``."""
    from . import gnnLightning as G
    ds = predict_dataset.dataset
    model_type = ds.get_data_format()
    if model_type == "heterogeneous_gnn":
        model = G.Heterogeneous_GNN_Lightning.load_from_checkpoint(str(path_to_checkpoint))
    elif model_type == "heterogeneous_gnn_k4":
        model = G.HGNN_K4_Lightning.load_from_checkpoint(str(path_to_checkpoint), symmetry_mode=symmetry_mode,
                                                         group_operator_path=group_operator_path, strict=False)
    elif model_type in _COM_FORMATS:
        from .gnnLightning_com import COM_HGNN_SYM_Lightning
        kw = {"data_path": data_path} if data_path is not None else {}
        model = COM_HGNN_SYM_Lightning.load_from_checkpoint(str(path_to_checkpoint), symmetry_mode=symmetry_mode,
                                                            group_operator_path=group_operator_path, model_type=model_type,
                                                            strict=False, **kw)
    elif model_type == "heterogeneous_gnn_c2":
        cls = G.HGNN_C2_Lightning_Reg if task_type == "regression" else G.HGNN_C2_Lightning_Cls
        kw = dict(grf_body_to_world_frame=grf_body_to_world_frame, grf_dimension=grf_dimension) if task_type == "regression" else {}
        model = cls.load_from_checkpoint(str(path_to_checkpoint), symmetry_mode=symmetry_mode, group_operator_path=group_operator_path,
                                         strict=False, **kw)
    else:
        raise ValueError("model_type must be mlp, heterogeneous_gnn, heterogeneous_gnn_k4, heterogeneous_gnn_c2, "
                         "heterogeneous_gnn_k4_com, heterogeneous_gnn_s4_com, or dynamics.")
    model.eval()
    model.freeze()
    model.to(ds.device)
    model.model.validate_edges = "cached"
    world = bool(getattr(model, "body_to_world_frame", False))
    if world:
        model.reset_all_metrics_worldframe()
    else:
        model.reset_all_metrics()
    preds, labels = [], []
    with torch.no_grad():
        for idx in _loader(predict_dataset, batch_size, False, None, None):
            batch = ds.batch(idx)
            labels_batch, y_pred = model.step_helper_function(batch)
            if world:
                # reference L1043-1045: world-frame metrics are what a body_to_world_frame model reports
                if not hasattr(batch, "r_o") or batch.r_o is None:
                    raise ValueError("grf_body_to_world_frame=True needs the body orientation r_o in every batch of predict_dataset")
                model.calculate_losses_step_worldframe(labels_batch, y_pred, batch.r_o.view(batch.batch_size, 4), test_only_on_z)
            elif hasattr(model, "calculate_losses_step_original"):
                model.calculate_losses_step_original(labels_batch, y_pred)
            else:
                model.calculate_losses_step(labels_batch, y_pred)
            if not model.regression:
                # 16-class prediction = the four per-foot argmaxes read as a binary number (the joint probability of
                # classification_conversion_16_class factorises over the feet)
                p = (y_pred.reshape(-1, 4, 2)[:, :, 1] > y_pred.reshape(-1, 4, 2)[:, :, 0]).long()
                w = torch.tensor([8, 4, 2, 1], device=p.device)
                preds.append((p * w).sum(1)); labels.append((labels_batch.long() * w).sum(1))
            else:
                preds.append(y_pred); labels.append(labels_batch)
        if world:
            model.calculate_losses_epoch_worldframe()
        elif hasattr(model, "calculate_losses_epoch_original"):
            model.calculate_losses_epoch_original()
        else:
            model.calculate_losses_epoch()
    pred, lab = torch.cat(preds), torch.cat(labels)
    if not model.regression:
        avg = (model.f1_leg0 + model.f1_leg1 + model.f1_leg2 + model.f1_leg3) / 4.0
        return pred, lab, model.acc, model.f1_leg0, model.f1_leg1, model.f1_leg2, model.f1_leg3, avg
    if world:
        return pred, lab, model.mse_loss_worldframe, model.rmse_loss_worldframe, model.l1_loss_worldframe
    if model_type in _COM_FORMATS:
        return pred, lab, model.mse_loss, model.rmse_loss, model.mse_loss_lin, model.mse_loss_ang, model.cos_sim_lin, model.cos_sim_ang
    return pred, lab, model.mse_loss, model.rmse_loss, model.l1_loss
