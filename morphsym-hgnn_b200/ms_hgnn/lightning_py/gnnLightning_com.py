"""COM (centre-of-mass momentum) Lightning-shaped modules on the B200-native engine.

Drop-in for the hot-path part of the reference's ``gnnLightning_com.py``: ``COM_Base_Lightning``
(L28-231), ``COM_HGNN_Lightning`` (L290-341), ``COM_HGNN_SYM_Lightning`` (L343-410).  The loss is the
native fused MSE over ``[B, n_base*6]``; lin/ang MSE and cosine similarity are metrics only.  On CUDA
batches every metric of a step comes from one ``mshgnn_step_metrics_ex`` call (``METRIC_COM``, fp64);
other inputs take the op-by-op metric classes of ``customMetrics.py``.
``rss_stats.npz`` is optional here (identity standardiser when absent); the reference hard-codes
``device='cuda:0'`` for it (L52-57), we follow the tensors' device.
"""
import os

import numpy as np
import torch
from torch import nn, optim

from .. import _native as N
from ..modules import native_loss
from ._lightning_shim import LightningModule
from .customMetrics import CosineSimilarityMetric, FusedStepMetrics, MeanSquaredError
from .gnnLightning import _dims_of
from .hgnn import COM_HGNN
from .hgnn_c2_com import COM_HGNN_C2
from .hgnn_k4_com import COM_HGNN_K4
from .hgnn_s4_com import COM_HGNN_S4


class Standarizer:
    """y = yn * std + mean per output channel (soloDataset.py Standarizer)."""

    def __init__(self, x_mean, x_std, y_mean, y_std, device="cpu"):
        self.y_mean = torch.as_tensor(np.asarray(y_mean), dtype=torch.float64)
        self.y_std = torch.as_tensor(np.asarray(y_std), dtype=torch.float64)

    def to(self, device):
        self.y_mean = self.y_mean.to(device); self.y_std = self.y_std.to(device)
        return self

    def unstandarize(self, yn):
        return yn * self.y_std.to(yn.dtype) + self.y_mean.to(yn.dtype)


class COM_Base_Lightning(LightningModule):
    def __init__(self, optimizer: str, lr: float, data_path: str):
        super().__init__()
        self.optimizer = optimizer
        self.lr = lr
        self.data_path = data_path
        self.regression = True
        stats_file = os.path.join(str(data_path), "processed", "rss_stats.npz") if data_path is not None else None
        if stats_file is not None and os.path.exists(stats_file):
            st = np.load(stats_file)
            self.standarizer = Standarizer(st["x_mean"], st["x_std"], st["y_mean"], st["y_std"])
        else:
            self.standarizer = Standarizer(np.zeros(24), np.ones(24), np.zeros(6), np.ones(6))
        self.metric_mse = MeanSquaredError(squared=True)
        self.metric_rmse = MeanSquaredError(squared=False)
        self.metric_mse_lin = MeanSquaredError(squared=True)
        self.metric_mse_ang = MeanSquaredError(squared=True)
        self.metric_cos_sim_lin = CosineSimilarityMetric()
        self.metric_cos_sim_ang = CosineSimilarityMetric()
        # CUDA batches: one fused native call per step feeds every metric (mshgnn_step_metrics_ex, METRIC_COM)
        self._fused = FusedStepMetrics()
        self.metric_mse.bind(self._fused, lambda e: e[N.COM_SSE] / e[N.COM_N])
        self.metric_rmse.bind(self._fused, lambda e: torch.sqrt(e[N.COM_SSE] / e[N.COM_N]))
        self.metric_mse_lin.bind(self._fused, lambda e: e[N.COM_SSE_LIN] / e[N.COM_N_HALF])
        self.metric_mse_ang.bind(self._fused, lambda e: e[N.COM_SSE_ANG] / e[N.COM_N_HALF])
        self.metric_cos_sim_lin.bind(self._fused, lambda e: e[N.COM_COS_LIN] / e[N.COM_ROWS])
        self.metric_cos_sim_ang.bind(self._fused, lambda e: e[N.COM_COS_ANG] / e[N.COM_ROWS])
        self.mse_loss = self.rmse_loss = self.mse_loss_lin = self.mse_loss_ang = None
        self.cos_sim_lin = self.cos_sim_ang = self.avg_cos_sim = self.loss = None

    def log_losses(self, step_name: str, on_step: bool):
        on_epoch = not on_step
        for k, v in (("_MSE_loss", self.mse_loss), ("_RMSE_loss", self.rmse_loss), ("_MSE_loss_lin", self.mse_loss_lin),
                     ("_MSE_loss_ang", self.mse_loss_ang), ("_cos_sim_lin", self.cos_sim_lin), ("_cos_sim_ang", self.cos_sim_ang),
                     ("_avg_cos_sim", self.avg_cos_sim), ("_loss", self.loss)):
            self.log(step_name + k, v, on_step=on_step, on_epoch=on_epoch)

    def calculate_losses_step(self, y: torch.Tensor, y_pred: torch.Tensor):
        self.mse_loss = native_loss(self.model, y_pred, y, N.LOSS_MSE)
        with torch.no_grad():
            if y_pred.is_cuda and self.model.num_dimensions_per_base == 6:
                self._metrics_step_fused(y, y_pred.detach())
            else:
                self._metrics_step_op_by_op(y, y_pred.detach())
        self.loss = self.mse_loss

    def _metrics_step_fused(self, y, y_pred):
        """Every metric of the step from one mshgnn_step_metrics_ex call (METRIC_COM, fp64)."""
        st = self.standarizer
        if st.y_mean.device != y_pred.device:           # the stats move to the device once
            st.to(y_pred.device)
        b = self._fused.update_com(y_pred, y, self.model.num_bases, st.y_mean, st.y_std)
        b = b[N.COM_RMSE:N.COM_AVG_COS_SIM + 1].clone()         # the fused buffer is overwritten by the next step
        self.rmse_loss, self.mse_loss_lin, self.mse_loss_ang, self.cos_sim_lin, self.cos_sim_ang, self.avg_cos_sim = b.unbind()

    def _metrics_step_op_by_op(self, yd, pd):
        """gnnLightning_com.py:L70-95 with the metric classes of customMetrics.py (CPU inputs and other widths)."""
        nb, nd = self.model.num_bases, self.model.num_dimensions_per_base
        self.metric_mse(pd.flatten(), yd.flatten())
        self.rmse_loss = self.metric_rmse(pd.flatten(), yd.flatten())
        yv = yd.view(yd.shape[0], nb, nd); pv = pd.view(pd.shape[0], nb, nd)
        self.mse_loss_lin = self.metric_mse_lin(pv[:, :, :3].flatten(), yv[:, :, :3].flatten())
        self.mse_loss_ang = self.metric_mse_ang(pv[:, :, 3:].flatten(), yv[:, :, 3:].flatten())
        self.standarizer.to(yd.device)
        yu = self.standarizer.unstandarize(yv); pu = self.standarizer.unstandarize(pv)
        self.cos_sim_lin = self.metric_cos_sim_lin(pu[:, 0, :3], yu[:, 0, :3])
        self.cos_sim_ang = self.metric_cos_sim_ang(pu[:, 0, 3:], yu[:, 0, 3:])
        self.avg_cos_sim = (self.cos_sim_lin + self.cos_sim_ang) / 2

    def calculate_losses_epoch(self) -> None:
        self.mse_loss = self.metric_mse.compute()
        self.rmse_loss = self.metric_rmse.compute()
        self.mse_loss_lin = self.metric_mse_lin.compute()
        self.mse_loss_ang = self.metric_mse_ang.compute()
        self.cos_sim_lin = self.metric_cos_sim_lin.compute()
        self.cos_sim_ang = self.metric_cos_sim_ang.compute()
        self.avg_cos_sim = (self.cos_sim_lin + self.cos_sim_ang) / 2
        self.loss = self.metric_mse.compute()

    def reset_all_metrics(self) -> None:
        for m in (self.metric_mse, self.metric_rmse, self.metric_mse_lin, self.metric_mse_ang,
                  self.metric_cos_sim_lin, self.metric_cos_sim_ang):
            m.reset()

    def training_step(self, batch, batch_idx):
        y, y_pred = self.step_helper_function(batch)
        self.calculate_losses_step(y, y_pred)
        self.log_losses("train", on_step=True)
        return self.loss

    def on_validation_epoch_start(self):
        self.reset_all_metrics()

    def validation_step(self, batch, batch_idx):
        y, y_pred = self.step_helper_function(batch)
        self.calculate_losses_step(y, y_pred)
        return self.mse_loss

    def on_validation_epoch_end(self):
        self.calculate_losses_epoch()
        self.log_losses("val", on_step=False)

    on_test_epoch_start = on_validation_epoch_start
    test_step = validation_step

    def on_test_epoch_end(self):
        self.calculate_losses_epoch()
        self.log_losses("test", on_step=False)

    def on_predict_start(self):
        self.reset_all_metrics()

    def predict_step(self, batch, batch_idx):
        y, y_pred = self.step_helper_function(batch)
        self.calculate_losses_step(y, y_pred)
        return y, y_pred

    def on_predict_end(self):
        self.calculate_losses_epoch()

    def configure_optimizers(self):
        if self.optimizer == "adam":
            return optim.Adam(self.parameters(), lr=self.lr)
        if self.optimizer == "sgd":
            return optim.SGD(self.parameters(), lr=self.lr)
        raise ValueError("Invalid optimizer setting")

    def step_helper_function(self, batch):
        out_raw = self.model(x_dict=batch.x_dict, edge_index_dict=batch.edge_index_dict)
        batch_size = batch.batch_size if hasattr(batch, "batch_size") else 1
        w = self.model.num_bases * self.model.num_dimensions_per_base
        y_pred = torch.reshape(out_raw.squeeze(), (batch_size, w))
        y = torch.reshape(batch.y, (batch_size, w))
        return y, y_pred


class COM_HGNN_Lightning(COM_Base_Lightning):
    def __init__(self, hidden_channels: int, num_layers: int, data_metadata, dummy_batch, optimizer: str = "adam",
                 lr: float = 0.003, regression: bool = True, activation_fn=nn.ReLU(), com_dimension: int = 6,
                 data_path=None):
        super().__init__(optimizer, lr, data_path)
        self.model = COM_HGNN(hidden_channels=hidden_channels, num_layers=num_layers, data_metadata=data_metadata,
                              regression=regression, activation_fn=activation_fn, com_dimension=com_dimension,
                              in_dims=_dims_of(dummy_batch))
        self.regression = regression
        self.save_hyperparameters()


class COM_HGNN_SYM_Lightning(COM_Base_Lightning):
    def __init__(self, hidden_channels: int, num_layers: int, data_metadata, dummy_batch, optimizer: str = "adam",
                 lr: float = 0.003, regression: bool = True, activation_fn=nn.ReLU(), symmetry_mode: str = None,
                 group_operator_path: str = None, model_type: str = "heterogeneous_gnn_k4_com", data_path=None):
        super().__init__(optimizer, lr, data_path)
        kw = dict(hidden_channels=hidden_channels, num_layers=num_layers, data_metadata=data_metadata,
                  regression=regression, activation_fn=activation_fn, in_dims=_dims_of(dummy_batch))
        if model_type == "heterogeneous_gnn_k4_com":
            self.model = COM_HGNN_K4(symmetry_mode=symmetry_mode, group_operator_path=group_operator_path, **kw)
        elif model_type == "heterogeneous_gnn_c2_com":
            self.model = COM_HGNN_C2(symmetry_mode=symmetry_mode, group_operator_path=group_operator_path, **kw)
        elif model_type == "heterogeneous_gnn_s4_com":
            self.model = COM_HGNN_S4(**kw)
        else:
            raise ValueError(f"unknown model_type {model_type}")
        self.regression = regression
        self.save_hyperparameters()
