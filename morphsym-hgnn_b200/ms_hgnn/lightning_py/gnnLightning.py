"""Lightning-shaped training / evaluation modules on the B200-native engine.

Drop-in for the hot-path part of the reference's ``gnnLightning.py``: ``Base_Lightning`` (L28-348),
``Heterogeneous_GNN_Lightning`` (L415-462), ``HGNN_K4_Lightning`` (L464-513),
``HGNN_C2_Lightning_Cls`` (L515-562), ``HGNN_C2_Lightning_Reg`` (L564-778).  Same constructor
kwargs (incl. ``dummy_batch``), same method names.  Differences, all deliberate:

* the loss heads run in the native fused kernel (value + gradient in one pass) and connect to
  autograd, so ``training_step(...).backward()`` drives the native backward pass;
* accuracy / F1 are device-side reductions - no host sync, no python loop over the batch, no
  sklearn (the reference's per-step ``for i in range(B)`` loop, L326-327, made its step host-bound);
* the lazily-sized encoder is materialised from ``dummy_batch`` shapes without a dummy forward, so the
  module can be built on a machine without a GPU.
"""
import numpy as np
import torch
from torch import nn, optim

from .. import _native as N
from ..modules import native_loss
from ._lightning_shim import LightningModule
from .customMetrics import (BinaryF1Score, CrossEntropyLossMetric, FusedStepMetrics, MeanAbsoluteError, MeanSquaredError,
                            MulticlassAccuracy)
from .hgnn import GRF_HGNN
from .hgnn_c2 import GRF_HGNN_C2
from .hgnn_k4 import GRF_HGNN_K4


def _dims_of(dummy_batch):
    return {t: int(v.shape[1]) for t, v in dummy_batch.x_dict.items()} if dummy_batch is not None else None


class Base_Lightning(LightningModule):
    def __init__(self, optimizer: str, lr: float, regression: bool):
        super().__init__()
        self.optimizer = optimizer
        self.lr = lr
        self.regression = regression
        self.metric_mse = MeanSquaredError(squared=True)
        self.metric_rmse = MeanSquaredError(squared=False)
        self.metric_l1 = MeanAbsoluteError()
        self.metric_ce = CrossEntropyLossMetric()
        self.metric_acc = MulticlassAccuracy()
        self.metric_f1_leg0 = BinaryF1Score()
        self.metric_f1_leg1 = BinaryF1Score()
        self.metric_f1_leg2 = BinaryF1Score()
        self.metric_f1_leg3 = BinaryF1Score()
        self.mse_loss = self.rmse_loss = self.l1_loss = self.ce_loss = self.acc = None
        self.f1_leg0 = self.f1_leg1 = self.f1_leg2 = self.f1_leg3 = None
        # CUDA batches: one fused native call per step feeds every metric (mshgnn_step_metrics, SURVEY 8f-2)
        self._fused = FusedStepMetrics()
        f1 = BinaryF1Score._f1
        if regression:
            self.metric_mse.bind(self._fused, lambda e: e[0] / e[2])
            self.metric_rmse.bind(self._fused, lambda e: torch.sqrt(e[0] / e[2]))
            self.metric_l1.bind(self._fused, lambda e: e[1] / e[2])
        else:
            self.metric_ce.bind(self._fused, lambda e: e[0].float() / e[1])
            self.metric_acc.bind(self._fused, lambda e: e[2] / e[3])
            for leg, m in enumerate((self.metric_f1_leg0, self.metric_f1_leg1, self.metric_f1_leg2, self.metric_f1_leg3)):
                m.bind(self._fused, lambda e, k=leg: f1(e[4 + 4 * k], e[5 + 4 * k], e[6 + 4 * k]))

    # ---- logging ----
    def log_losses(self, step_name: str, on_step: bool):
        on_epoch = not on_step
        if self.regression:
            for k, v in (("_MSE_loss", self.mse_loss), ("_RMSE_loss", self.rmse_loss), ("_L1_loss", self.l1_loss)):
                self.log(step_name + k, v, on_step=on_step, on_epoch=on_epoch)
        else:
            self.log(step_name + "_CE_loss", self.ce_loss, on_step=on_step, on_epoch=on_epoch)
            self.log(step_name + "_Accuracy", self.acc, on_step=on_step, on_epoch=on_epoch)
            self.log(step_name + "_F1_Score_Leg_Avg", (self.f1_leg0 + self.f1_leg1 + self.f1_leg2 + self.f1_leg3) / 4.0,
                     on_step=on_step, on_epoch=on_epoch)
            for i, v in enumerate((self.f1_leg0, self.f1_leg1, self.f1_leg2, self.f1_leg3)):
                self.log(step_name + f"_F1_Score_Leg_{i}", v, on_step=on_step, on_epoch=on_epoch)

    # ---- loss heads ----
    def calculate_losses_step(self, y: torch.Tensor, y_pred: torch.Tensor):
        if self.regression and y_pred.is_cuda:
            self.mse_loss = native_loss(self.model, y_pred, y, N.LOSS_MSE)
            with torch.no_grad():
                b = self._fused.update(N.LOSS_MSE, y_pred.detach().reshape(-1), y, y_pred.numel(), 1)
                b = b[21:23].clone()             # the fused buffer is overwritten by the next step: logged values must not alias it
                self.rmse_loss, self.l1_loss = b[0], b[1]
        elif not self.regression and y_pred.is_cuda and y_pred.shape[1] == 8:
            # gradient-carrying CE from the fused loss head; accuracy / F1 / epoch states from ONE fused metrics call
            self.ce_loss = native_loss(self.model, y_pred, y, N.LOSS_CE2)
            with torch.no_grad():
                b = self._fused.update(N.LOSS_CE2, y_pred.detach().reshape(-1, 2), y, y_pred.shape[0], 4)
                b = b[21:26].clone()             # see above
                self.acc = b[0]
                self.f1_leg0, self.f1_leg1, self.f1_leg2, self.f1_leg3 = b[1], b[2], b[3], b[4]
        elif self.regression:
            # native fused MSE (gradient-carrying) + metric accumulation
            self.mse_loss = native_loss(self.model, y_pred, y, N.LOSS_MSE)
            with torch.no_grad():
                yf, pf = y.flatten(), y_pred.detach().flatten()
                self.metric_mse(pf, yf)
                self.rmse_loss = self.metric_rmse(pf, yf)
                self.l1_loss = self.metric_l1(pf, yf)
        else:
            batch_size = y_pred.shape[0]
            # CE: four 2-way cross-entropies per graph averaged over 4B rows (customMetrics.py:L6-25)
            self.ce_loss = native_loss(self.model, y_pred, y, N.LOSS_CE2)
            with torch.no_grad():
                self.metric_ce.accumulate_value(self.ce_loss, batch_size * 4)
                y_pred_per_foot, y_pred_per_foot_prob, p1 = self.classification_calculate_useful_values(y_pred.detach(), batch_size)
                y_pred_16, y_16 = self.classification_conversion_16_class(p1, y)
                self.acc = self.metric_acc(torch.argmax(y_pred_16, dim=1), y_16.squeeze(dim=1))
                y_pred_2 = torch.reshape(torch.argmax(y_pred_per_foot_prob, dim=1), (batch_size, 4))
                self.f1_leg0 = self.metric_f1_leg0(y_pred_2[:, 0], y[:, 0])
                self.f1_leg1 = self.metric_f1_leg1(y_pred_2[:, 1], y[:, 1])
                self.f1_leg2 = self.metric_f1_leg2(y_pred_2[:, 2], y[:, 2])
                self.f1_leg3 = self.metric_f1_leg3(y_pred_2[:, 3], y[:, 3])

    def calculate_losses_epoch(self) -> None:
        if self.regression:
            self.mse_loss = self.metric_mse.compute()
            self.rmse_loss = self.metric_rmse.compute()
            self.l1_loss = self.metric_l1.compute()
        else:
            self.ce_loss = self.metric_ce.compute()
            self.acc = self.metric_acc.compute()
            self.f1_leg0 = self.metric_f1_leg0.compute()
            self.f1_leg1 = self.metric_f1_leg1.compute()
            self.f1_leg2 = self.metric_f1_leg2.compute()
            self.f1_leg3 = self.metric_f1_leg3.compute()

    def reset_all_metrics(self) -> None:
        for m in (self.metric_mse, self.metric_rmse, self.metric_l1, self.metric_ce, self.metric_acc,
                  self.metric_f1_leg0, self.metric_f1_leg1, self.metric_f1_leg2, self.metric_f1_leg3):
            m.reset()

    # ---- steps ----
    def _loss(self):
        return self.mse_loss if self.regression else self.ce_loss

    def training_step(self, batch, batch_idx):
        y, y_pred = self.step_helper_function(batch)
        self.calculate_losses_step(y, y_pred)
        self.log_losses("train", on_step=True)
        return self._loss()

    def on_validation_epoch_start(self):
        self.reset_all_metrics()

    def validation_step(self, batch, batch_idx):
        y, y_pred = self.step_helper_function(batch)
        self.calculate_losses_step(y, y_pred)
        return self._loss()

    def on_validation_epoch_end(self):
        self.calculate_losses_epoch()
        self.log_losses("val", on_step=False)

    def on_test_epoch_start(self):
        self.reset_all_metrics()

    def test_step(self, batch, batch_idx):
        y, y_pred = self.step_helper_function(batch)
        self.calculate_losses_step(y, y_pred)
        return self._loss()

    def on_test_epoch_end(self):
        self.calculate_losses_epoch()
        self.log_losses("test", on_step=False)

    def on_predict_start(self):
        self.reset_all_metrics()

    def predict_step(self, batch, batch_idx):
        y, y_pred = self.step_helper_function(batch)
        self.calculate_losses_step(y, y_pred)
        if self.regression:
            return y, y_pred
        raise NotImplementedError("This prediction method is not fully tested for classification.")

    def on_predict_end(self):
        self.calculate_losses_epoch()

    def configure_optimizers(self):
        if self.optimizer == "adam":
            return optim.Adam(self.parameters(), lr=self.lr)
        if self.optimizer == "sgd":
            return optim.SGD(self.parameters(), lr=self.lr)
        raise ValueError("Invalid optimizer setting")

    def step_helper_function(self, batch):
        raise NotImplementedError

    # ---- classification helpers (L285-348), vectorised and device-resident ----
    def classification_calculate_useful_values(self, y_pred, batch_size):
        y_pred_per_foot = torch.reshape(y_pred, (batch_size * 4, 2))
        y_pred_per_foot_prob = torch.nn.functional.softmax(y_pred_per_foot, dim=1)
        y_pred_per_foot_prob_only_1 = torch.reshape(y_pred_per_foot_prob[:, 1], (batch_size, 4))
        return y_pred_per_foot, y_pred_per_foot_prob, y_pred_per_foot_prob_only_1

    def classification_conversion_16_class(self, y_pred_per_foot_prob_only_1: torch.Tensor, y: torch.Tensor):
        yl = y.long()
        y_new = (yl[:, 0] * 8 + yl[:, 1] * 4 + yl[:, 2] * 2 + yl[:, 3]).reshape(-1, 1)
        p = y_pred_per_foot_prob_only_1
        cols = []
        for j in range(16):
            f = [(p[:, k] if (j >> (3 - k)) & 1 else 1 - p[:, k]) for k in range(4)]
            cols.append(torch.mul(torch.mul(f[0], f[1]), torch.mul(f[2], f[3])))
        return torch.stack(cols, dim=1), y_new

    # ---- shared by the subclasses ----
    def _foot_step(self, batch, y_width):
        out_raw = self.model(x_dict=batch.x_dict, edge_index_dict=batch.edge_index_dict)
        batch_size = batch.batch_size if hasattr(batch, "batch_size") else 1
        y_pred = torch.reshape(out_raw.squeeze(), (batch_size, self.model.out_channels_per_foot * 4))
        y = torch.reshape(batch.y, (batch_size, y_width))
        return y, y_pred


class Heterogeneous_GNN_Lightning(Base_Lightning):
    def __init__(self, hidden_channels: int, num_layers: int, data_metadata, dummy_batch, optimizer: str = "adam",
                 lr: float = 0.003, regression: bool = True, activation_fn=nn.ReLU(), grf_dimension: int = 1):
        super().__init__(optimizer, lr, regression)
        self.model = GRF_HGNN(hidden_channels=hidden_channels, num_layers=num_layers, data_metadata=data_metadata,
                              regression=regression, activation_fn=activation_fn, grf_dimension=grf_dimension,
                              in_dims=_dims_of(dummy_batch))
        self.regression = regression
        self.save_hyperparameters()

    def step_helper_function(self, batch):
        return self._foot_step(batch, self.model.out_channels_per_foot * 4)


class HGNN_K4_Lightning(Base_Lightning):
    def __init__(self, hidden_channels: int, num_layers: int, data_metadata, dummy_batch, optimizer: str = "adam",
                 lr: float = 0.003, regression: bool = True, activation_fn=nn.ReLU(), symmetry_mode: str = None,
                 group_operator_path: str = None):
        super().__init__(optimizer, lr, regression)
        self.model = GRF_HGNN_K4(hidden_channels=hidden_channels, num_layers=num_layers, data_metadata=data_metadata,
                                 regression=regression, activation_fn=activation_fn, symmetry_mode=symmetry_mode,
                                 group_operator_path=group_operator_path, in_dims=_dims_of(dummy_batch))
        self.regression = regression
        self.save_hyperparameters()

    def step_helper_function(self, batch):
        return self._foot_step(batch, 4)


class HGNN_C2_Lightning_Cls(Base_Lightning):
    def __init__(self, hidden_channels: int, num_layers: int, data_metadata, dummy_batch, optimizer: str = "adam",
                 lr: float = 0.003, regression: bool = True, activation_fn=nn.ReLU(), symmetry_mode: str = None,
                 group_operator_path: str = None):
        super().__init__(optimizer, lr, regression)
        self.model = GRF_HGNN_C2(hidden_channels=hidden_channels, num_layers=num_layers, data_metadata=data_metadata,
                                 regression=regression, activation_fn=activation_fn, symmetry_mode=symmetry_mode,
                                 group_operator_path=group_operator_path, in_dims=_dims_of(dummy_batch))
        self.regression = regression
        self.save_hyperparameters()

    def step_helper_function(self, batch):
        return self._foot_step(batch, 4)


class HGNN_C2_Lightning_Reg(Base_Lightning):
    def __init__(self, hidden_channels: int, num_layers: int, data_metadata, dummy_batch, optimizer: str = "adam",
                 lr: float = 0.003, regression: bool = True, activation_fn=nn.ReLU(), symmetry_mode: str = None,
                 group_operator_path: str = None, grf_body_to_world_frame: bool = None, grf_dimension: int = 3):
        super().__init__(optimizer, lr, regression)
        self.model = GRF_HGNN_C2(hidden_channels=hidden_channels, num_layers=num_layers, data_metadata=data_metadata,
                                 regression=regression, activation_fn=activation_fn, symmetry_mode=symmetry_mode,
                                 group_operator_path=group_operator_path, grf_dimension=grf_dimension,
                                 in_dims=_dims_of(dummy_batch))
        self.regression = regression
        self.save_hyperparameters()
        self.body_to_world_frame = grf_body_to_world_frame if self.regression else False
        if self.body_to_world_frame:
            self.metric_mse_worldframe = MeanSquaredError(squared=True)
            self.metric_rmse_worldframe = MeanSquaredError(squared=False)
            self.metric_l1_worldframe = MeanAbsoluteError()
            self.mse_loss_worldframe = self.rmse_loss_worldframe = self.l1_loss_worldframe = None
            # the world-frame call (METRIC_GRF_WORLD) fills the body-frame states 0..2 too: the bindings above still hold
            self.metric_mse_worldframe.bind(self._fused, lambda e: e[N.GRF_SSE_WORLD] / e[N.GRF_N_WORLD])
            self.metric_rmse_worldframe.bind(self._fused, lambda e: torch.sqrt(e[N.GRF_SSE_WORLD] / e[N.GRF_N_WORLD]))
            self.metric_l1_worldframe.bind(self._fused, lambda e: e[N.GRF_SAE_WORLD] / e[N.GRF_N_WORLD])

    def calculate_losses_step_original(self, y, y_pred):
        Base_Lightning.calculate_losses_step(self, y, y_pred)

    def calculate_losses_step(self, y, y_pred, batch_r_quat=None, test_only_on_z: bool = False):
        if self.body_to_world_frame and batch_r_quat is not None:
            return self.calculate_losses_step_worldframe(y, y_pred, batch_r_quat, test_only_on_z)
        return self.calculate_losses_step_original(y, y_pred)

    def calculate_losses_step_worldframe(self, y, y_pred, batch_r_quat, test_only_on_z: bool = False):
        if y_pred.is_cuda and y_pred.shape[1] == 12:
            self.mse_loss = native_loss(self.model, y_pred, y, N.LOSS_MSE)
            with torch.no_grad():
                self._worldframe_metrics_fused(y, y_pred.detach(), batch_r_quat, test_only_on_z)
            return
        self.calculate_losses_step_original(y, y_pred)
        with torch.no_grad():
            self._worldframe_metrics_op_by_op(y, y_pred.detach(), batch_r_quat, test_only_on_z)

    def _worldframe_metrics_fused(self, y, y_pred, batch_r_quat, test_only_on_z):
        """Body- and world-frame metrics from ONE mshgnn_step_metrics_ex call (METRIC_GRF_WORLD, fp64)."""
        b = self._fused.update_grf_world(y_pred, y, batch_r_quat, test_only_on_z)
        b = b[N.GRF_RMSE:N.GRF_L1_WORLD + 1].clone()           # the fused buffer is overwritten by the next step
        self.rmse_loss, self.l1_loss, self.mse_loss_worldframe, self.rmse_loss_worldframe, self.l1_loss_worldframe = b.unbind()

    def _worldframe_metrics_op_by_op(self, y, y_pred, batch_r_quat, test_only_on_z):
        y_world = self.body_frame_to_world_frame(batch_r_quat, y)
        y_pred_world = self.body_frame_to_world_frame(batch_r_quat, y_pred)
        if test_only_on_z:
            z_index = [2, 5, 8, 11]
            y_world, y_pred_world = y_world[:, z_index], y_pred_world[:, z_index]
        self.mse_loss_worldframe = self.metric_mse_worldframe(y_pred_world, y_world)
        self.rmse_loss_worldframe = self.metric_rmse_worldframe(y_pred_world, y_world)
        self.l1_loss_worldframe = self.metric_l1_worldframe(y_pred_world, y_world)

    def body_frame_to_world_frame(self, batch_r_quat, grf_bodyFrame):
        """Rotate per-foot forces by the inverse of the (x, y, z, w) body quaternion, on the device
        (the reference goes through scipy on the host, L662-676)."""
        q = batch_r_quat.to(grf_bodyFrame.dtype)
        q = q / q.norm(dim=1, keepdim=True)
        x, y, z, w = q[:, 0], q[:, 1], q[:, 2], q[:, 3]
        R = torch.stack((1 - 2 * (y * y + z * z), 2 * (x * y - z * w), 2 * (x * z + y * w),
                         2 * (x * y + z * w), 1 - 2 * (x * x + z * z), 2 * (y * z - x * w),
                         2 * (x * z - y * w), 2 * (y * z + x * w), 1 - 2 * (x * x + y * y)), dim=1).view(-1, 3, 3)
        Rinv = R.transpose(1, 2)
        B = q.shape[0]
        f = grf_bodyFrame.view(B, 4, -1).permute(0, 2, 1)
        return (Rinv @ f).permute(0, 2, 1).flatten(start_dim=1)

    def step_helper_function(self, batch):
        return self._foot_step(batch, self.model.out_channels_per_foot * 4)

    # ---- world-frame epoch side (reference gnnLightning.py:L615-619, L701-711) ----
    def log_losses_worldframe(self, step_name: str, on_step: bool):
        self.log_losses(step_name, on_step)
        for k, v in (("_MSE_loss_WorldFrame", self.mse_loss_worldframe), ("_RMSE_loss_WorldFrame", self.rmse_loss_worldframe),
                     ("_L1_loss_WorldFrame", self.l1_loss_worldframe)):
            self.log(step_name + k, v, on_step=on_step, on_epoch=not on_step)

    def calculate_losses_epoch_worldframe(self) -> None:
        self.calculate_losses_epoch()
        self.mse_loss_worldframe = self.metric_mse_worldframe.compute()
        self.rmse_loss_worldframe = self.metric_rmse_worldframe.compute()
        self.l1_loss_worldframe = self.metric_l1_worldframe.compute()

    def reset_all_metrics_worldframe(self) -> None:
        self.reset_all_metrics()
        for m in (self.metric_mse_worldframe, self.metric_rmse_worldframe, self.metric_l1_worldframe):
            m.reset()

    def _quat_of(self, batch):
        if not hasattr(batch, "r_o") or batch.r_o is None:
            raise ValueError("grf_body_to_world_frame=True needs the body orientation batch.r_o (x, y, z, w per graph)")
        return batch.r_o.view(batch.batch_size, 4)

    def _step(self, batch):
        y, y_pred = self.step_helper_function(batch)
        if self.body_to_world_frame:
            self.calculate_losses_step_worldframe(y, y_pred, self._quat_of(batch))
        else:
            self.calculate_losses_step_original(y, y_pred)
        return self._loss()

    def training_step(self, batch, batch_idx):
        loss = self._step(batch)
        if self.body_to_world_frame:
            self.log_losses_worldframe("train", on_step=True)
        else:
            self.log_losses("train", on_step=True)
        return loss

    def _epoch_start(self):
        if self.body_to_world_frame:
            self.reset_all_metrics_worldframe()
        else:
            self.reset_all_metrics()

    def _epoch_end(self, name):
        if self.body_to_world_frame:
            self.calculate_losses_epoch_worldframe()
            self.log_losses_worldframe(name, on_step=False)
        else:
            self.calculate_losses_epoch()
            self.log_losses(name, on_step=False)

    def on_validation_epoch_start(self):
        self._epoch_start()

    def validation_step(self, batch, batch_idx):
        return self._step(batch)

    def on_validation_epoch_end(self):
        self._epoch_end("val")

    def on_test_epoch_start(self):
        self._epoch_start()

    def test_step(self, batch, batch_idx):
        return self._step(batch)

    def on_test_epoch_end(self):
        self._epoch_end("test")


# train_model / evaluate_model live next to the modules in the reference (gnnLightning.py:L913-1421)
from .trainer import WindowSubset, evaluate_model, train_model  # noqa: E402,F401
