"""Epoch-accumulated metrics with torchmetrics-style semantics, device-resident (no host sync).

Mirrors the reference's ``customMetrics.py`` (``CrossEntropyLossMetric`` L6-25, ``BinaryF1Score``
L27-54, ``CosineSimilarityMetric`` L56-91) and the three torchmetrics regressions it uses.  Calling a
metric (``metric(preds, target)``) returns the value of THIS batch and accumulates the epoch state;
``compute()`` returns the epoch value; ``reset()`` clears it.  torchmetrics / sklearn are not
needed: the confusion counts are four device-side sums.
"""
import torch
from torch import nn


class FusedStepMetrics:
    """Device-side accumulators of ``mshgnn_step_metrics`` / ``mshgnn_step_metrics_ex`` (include/mshgnn_b200.h): one native call per step produces this
    batch's values (``batch``) and adds the counts to the epoch states (``epoch``), replacing ~80 small torch launches of
    the op-by-op path below (and the reference's host-side sklearn / python loop, gnnLightning.py:L285-348)."""

    def __init__(self):
        self.batch = self.epoch = self.scratch = None
        self.dirty = False

    def _operands(self, out2d: torch.Tensor, labels: torch.Tensor):
        from .. import _native as N
        dev = out2d.device
        if self.batch is None or self.batch.device != dev:
            self.batch = torch.zeros(N.METRIC_SLOTS, dtype=torch.float64, device=dev)
            self.epoch = torch.zeros(N.METRIC_SLOTS, dtype=torch.float64, device=dev)
            self.scratch = torch.empty(N.METRIC_SCRATCH, dtype=torch.float64, device=dev)
        if out2d.dtype != torch.float32 or not out2d.is_contiguous():
            out2d = out2d.float().contiguous()
        labels = labels.reshape(-1).contiguous()
        code = {torch.float32: N.F32, torch.float64: N.F64, torch.int64: N.I64}.get(labels.dtype)
        if code is None:
            labels, code = labels.double(), N.F64
        return out2d, labels, code

    def update(self, kind: int, out2d: torch.Tensor, labels: torch.Tensor, n: int, feet: int) -> torch.Tensor:
        from .. import _native as N
        out2d, labels, code = self._operands(out2d, labels)
        dev = out2d.device
        with torch.cuda.device(dev):
            N.step_metrics(kind, n, feet, out2d.data_ptr(), labels.data_ptr(), code, self.batch.data_ptr(), self.epoch.data_ptr(),
                           self.scratch.data_ptr(), torch.cuda.current_stream(dev).cuda_stream)
        self.dirty = True
        return self.batch

    def _update_ex(self, kind: int, out2d: torch.Tensor, labels: torch.Tensor, n: int, args) -> torch.Tensor:
        from .. import _native as N
        out2d, labels, code = self._operands(out2d, labels)
        dev = out2d.device
        with torch.cuda.device(dev):
            N.step_metrics_ex(kind, args, n, out2d.data_ptr(), labels.data_ptr(), code, self.batch.data_ptr(),
                              self.epoch.data_ptr(), self.scratch.data_ptr(), torch.cuda.current_stream(dev).cuda_stream)
        self.dirty = True
        return self.batch

    def update_com(self, pred: torch.Tensor, labels: torch.Tensor, n_base: int, y_mean: torch.Tensor, y_std: torch.Tensor) -> torch.Tensor:
        """COM momentum metrics (``METRIC_COM``): ``pred`` / ``labels`` [B, n_base*6] standardised, ``y_mean`` / ``y_std`` contiguous
        fp64 [6] tensors on the same device (the standardiser's stats).  Returns the slot buffer (batch values at 20..26)."""
        from .. import _native as N
        B = pred.shape[0]
        if pred.numel() != B * n_base * 6 or labels.numel() != pred.numel():
            raise ValueError(f"COM metrics need predictions and labels of [B, {n_base * 6}]")
        for t in (y_mean, y_std):
            if t.dtype != torch.float64 or t.numel() != 6 or not t.is_contiguous() or t.device != pred.device:
                raise ValueError("COM metrics need y_mean / y_std as contiguous float64 [6] tensors on the predictions' device")
        args = N.MetricArgs(n_base=n_base, y_mean=y_mean.data_ptr(), y_std=y_std.data_ptr())
        return self._update_ex(N.METRIC_COM, pred, labels, B, args)

    def update_grf_world(self, pred: torch.Tensor, labels: torch.Tensor, quat: torch.Tensor, z_only: bool = False) -> torch.Tensor:
        """Body- and world-frame GRF metrics (``METRIC_GRF_WORLD``): ``pred`` / ``labels`` [B, 12] body frame, ``quat`` [B, 4]
        (x, y, z, w).  Slots 0..2 are those of the MSE kind, so this call also feeds metrics bound to the body-frame states."""
        from .. import _native as N
        B = pred.shape[0]
        if pred.numel() != B * 12 or labels.numel() != B * 12 or quat.numel() != B * 4:
            raise ValueError("world-frame GRF metrics need predictions and labels of [B, 12] and quaternions of [B, 4]")
        if quat.device != pred.device:
            raise ValueError("the quaternions must be on the predictions' device")
        quat = quat.reshape(-1).contiguous()
        if quat.dtype not in (torch.float32, torch.float64):
            quat = quat.double()
        args = N.MetricArgs(quat=quat.data_ptr(), quat_dtype=N.F64 if quat.dtype == torch.float64 else N.F32, z_only=int(bool(z_only)))
        return self._update_ex(N.METRIC_GRF_WORLD, pred, labels, B, args)

    def reset(self):
        if self.epoch is not None:
            self.epoch.zero_()
        self.dirty = False


class _Metric(nn.Module):
    def __init__(self):
        super().__init__()
        self._state = {}
        self._fused = None
        self._fused_fn = None

    def bind(self, fused: FusedStepMetrics, fn):
        """Epoch value comes from the fused accumulators (``fn(epoch) -> tensor``) whenever the fused kernel fed this epoch."""
        self._fused, self._fused_fn = fused, fn
        return self

    def _from_fused(self):
        return self._fused is not None and self._fused.dirty and not self._state

    def _acc(self, name, value):
        v = value.detach().double()
        self._state[name] = v if name not in self._state else self._state[name] + v

    def reset(self):
        self._state = {}
        if self._fused is not None:
            self._fused.reset()

    def forward(self, preds, target):
        batch = self.update(preds, target)
        return batch


class MeanSquaredError(_Metric):
    def __init__(self, squared: bool = True):
        super().__init__()
        self.squared = squared

    def update(self, preds, target):
        d = preds.reshape(-1) - target.reshape(-1)
        sse = (d * d).sum()
        self._acc("sse", sse); self._acc("n", torch.tensor(float(d.numel()), device=d.device))
        mse = sse / d.numel()
        return mse if self.squared else torch.sqrt(mse)

    def compute(self):
        if self._from_fused():
            return self._fused_fn(self._fused.epoch)
        mse = self._state["sse"] / self._state["n"]
        return mse if self.squared else torch.sqrt(mse)


class MeanAbsoluteError(_Metric):
    def update(self, preds, target):
        d = (preds.reshape(-1) - target.reshape(-1)).abs()
        self._acc("sae", d.sum()); self._acc("n", torch.tensor(float(d.numel()), device=d.device))
        return d.mean()

    def compute(self):
        if self._from_fused():
            return self._fused_fn(self._fused.epoch)
        return self._state["sae"] / self._state["n"]


class CrossEntropyLossMetric(_Metric):
    """sum-reduced CE over the rows, epoch value = summed_loss.float() / total_num (customMetrics.py:L25)."""

    def update(self, preds, target):
        if preds.size(0) != target.size(0):
            raise ValueError("Both tensors must have the same number of batches.")
        s = torch.nn.functional.cross_entropy(preds, target, reduction="sum")
        self._acc("sum", s); self._acc("n", torch.tensor(float(preds.shape[0]), device=preds.device))
        return s.float() / preds.shape[0]

    def accumulate_value(self, batch_mean: torch.Tensor, n_rows: int):
        """Accumulate a batch mean computed elsewhere (the native fused CE kernel)."""
        self._acc("sum", batch_mean.detach().double() * n_rows)
        self._acc("n", torch.tensor(float(n_rows), device=batch_mean.device))

    def compute(self):
        if self._from_fused():
            return self._fused_fn(self._fused.epoch)
        return self._state["sum"].float() / self._state["n"]


class MulticlassAccuracy(_Metric):
    def update(self, preds, target):
        ok = (preds == target).sum()
        self._acc("ok", ok); self._acc("n", torch.tensor(float(preds.numel()), device=preds.device))
        return ok.double() / preds.numel()

    def compute(self):
        if self._from_fused():
            return self._fused_fn(self._fused.epoch)
        return self._state["ok"] / self._state["n"]


class BinaryF1Score(_Metric):
    def update(self, preds, target):
        if preds.size(0) != target.size(0):
            raise ValueError("Both tensors must have the same number of batches.")
        p = preds.reshape(-1) != 0
        t = target.reshape(-1) != 0
        tp = (p & t).sum(); fp = (p & ~t).sum(); fn = (~p & t).sum()
        self._acc("tp", tp); self._acc("fp", fp); self._acc("fn", fn)
        return self._f1(tp.double(), fp.double(), fn.double())

    @staticmethod
    def _f1(tp, fp, fn):
        precision = tp / (tp + fp)
        recall = tp / (tp + fn)
        return torch.nan_to_num(2 * (precision * recall) / (precision + recall))

    def compute(self):
        if self._from_fused():
            return self._fused_fn(self._fused.epoch)
        return self._f1(self._state["tp"], self._state["fp"], self._state["fn"])


class CosineSimilarityMetric(_Metric):
    def update(self, preds, target):
        if preds.size() != target.size():
            raise ValueError("Prediction and target tensors must have the same shape")
        sim = torch.nn.functional.cosine_similarity(preds, target, dim=1)
        self._acc("sum", sim.sum()); self._acc("n", torch.tensor(float(preds.shape[0]), device=preds.device))
        return sim.mean()

    def compute(self):
        if self._from_fused():
            return self._fused_fn(self._fused.epoch)
        return self._state["sum"] / self._state["n"]
