"""Model batches: M independent models of one architecture trained and run in one native step.

Every launch of a step serves all M models: model m's graphs are row block m of every activation slab, and each kernel
reads the weights of the model its row tile belongs to.  Model m gets bit for bit what the single-model calls give for
its parameters and graphs (include/mshgnn_b200.h, DESIGN.md).  The models may differ in hidden width (``mixed_hidden``):
each runs zero-padded on the 128-wide kernels, and the parameter buffer holds their own layouts end to end.  The parameters
of model m stay ordinary ``nn.Parameter`` views - of ``flat[m]``, its range of one contiguous buffer - so
``models[m].state_dict()``, checkpoints and a single-model ``models[m](x_dict, edge_index_dict)`` keep working.
"""
from __future__ import annotations

import numbers
from typing import List, Optional, Sequence, Union

import torch

from . import _native as N
from .engine import Engine


class ModelBatch:
    """M native models of one configuration (same class, layer count, node / edge types, feature widths and mode, and the
    same hidden width unless ``mixed_hidden``) whose parameters live in one contiguous fp32 buffer (``buffer``, built on the
    first step; ``flat[m]`` is model m's range of it)."""

    def __init__(self, models: Sequence[torch.nn.Module], mixed_hidden: bool = False):
        models = list(models)
        if not models:
            raise ValueError("a model batch needs at least one model")
        if len(models) > N.MAX_MODELS:
            raise ValueError(f"a model batch holds at most {N.MAX_MODELS} models, got {len(models)}")
        m0 = models[0]
        self.mixed_hidden = bool(mixed_hidden)
        for i, m in enumerate(models[1:], 1):
            if type(m) is not type(m0):
                raise ValueError(f"model {i} is a {type(m).__name__}, model 0 a {type(m0).__name__}: a model batch has one class")
            if self._config(m) != self._config(m0):
                raise ValueError(f"model {i} differs from model 0 in its configuration {self._config(m)} != {self._config(m0)}")
        self.models = models
        self.buffer: Optional[torch.Tensor] = None
        self.flat: Optional[List[torch.Tensor]] = None
        self.offsets: Optional[List[int]] = None
        self._engine: Optional[Engine] = None       # the batch's own plan (mshgnn_plan_create_models)
        self._eng0 = None                           # model 0's engine the batch plan was built from
        self._specs = {}

    def _config(self, m) -> tuple:
        enc = m.encoder
        in_dims = tuple((t, enc.lins[t].in_features) for t in m.node_types) if enc.materialized else None
        hidden = () if self.mixed_hidden else (m.hidden_channels,)
        return hidden + (m.num_layers, tuple(m.node_types), tuple(m.edge_types), m._out_channels, m.morph_sym,
                         getattr(m, "mode", None), in_dims, tuple(sorted((m._user_nodes_per_graph or {}).items())))

    def __len__(self) -> int:
        return len(self.models)

    def _engines(self, batches):
        """Validates every batch through its model's own edge check; returns (the batch's engine, graphs per model)."""
        if len(batches) != len(self.models):
            raise ValueError(f"{len(self.models)} batches expected (one per model), got {len(batches)}")
        eng0, B = None, None
        for i, (m, b) in enumerate(zip(self.models, batches)):
            eng, Bm = m._engine_for(b.x_dict, b.edge_index_dict)
            m._last_engine = eng
            if eng0 is None:
                eng0, B = eng, Bm
                continue
            if Bm != B:
                raise ValueError(f"batch {i} has {Bm} graphs, batch 0 {B}: a model batch runs the same graph count per model")
            key = (id(eng0), id(eng))
            if key not in self._specs:
                if dict(eng.spec, hidden=None) != dict(eng0.spec, hidden=None):
                    raise ValueError(f"batch {i} is a different morphology template than batch 0")
                self._specs[key] = True
        if self._eng0 is not eng0:
            self._engine = Engine(dict(eng0.spec, widths=[m.hidden_channels for m in self.models]), eng0.mode)
            self._eng0 = eng0
            self.buffer = self.flat = None
        self._engine.mode = eng0.mode
        return self._engine, B

    def _bind(self, device) -> torch.Tensor:
        """Make every model's parameters views of its range ``flat[m]`` of ``buffer`` (copying their current values in once)."""
        for m in self.models:
            m._ensure_flat(device)
        flat = self.flat
        if flat is not None and self.buffer.device == device and all(m._flat.data_ptr() == flat[i].data_ptr() for i, m in enumerate(self.models)):
            return self.buffer
        eng = self._engine
        offs = eng.model_offsets()
        buf = torch.empty(eng.n_params, dtype=torch.float32, device=device)
        flat = [buf[offs[i]:offs[i + 1]] for i in range(len(self.models))]
        with torch.no_grad():
            for i, m in enumerate(self.models):
                flat[i].copy_(m._flat)
                named = dict(m.named_parameters())
                for (name, off, shape) in eng.param_layout(i):
                    n = int(torch.Size(shape).numel())
                    named[name].data = buf[off:off + n].view(shape)
                m._flat = flat[i]
        self.buffer, self.flat, self.offsets = buf, flat, offs
        return buf


class ModelBatchTrainer:
    """Fused Adam / SGD training of a ModelBatch: one native forward + loss + backward for all M models per step, then one
    optimizer launch for all of them.  Model m's parameters, Adam moments and step count evolve exactly as a FusedTrainer's
    with learning rate ``lr[m]`` on model m alone."""

    def __init__(self, model_batch: ModelBatch, optimizer: str = "adam", lr: Union[float, Sequence[float]] = 1e-3, process_group=None,
                 betas=(0.9, 0.999), eps: float = 1e-8, weight_decay: float = 0.0, regression: Optional[bool] = None):
        """``lr``: one learning rate for every model or one per model.  ``regression``: MSE loss (True) or per-foot
        cross-entropy (False); None takes the models' ``regression``."""
        if process_group is not None:
            raise ValueError("model batches do not combine with data parallelism: pass no process group")
        if optimizer not in ("adam", "sgd"):
            raise ValueError("Invalid optimizer setting")
        M = len(model_batch)
        lrs = [float(lr)] * M if isinstance(lr, numbers.Real) else [float(v) for v in lr]
        if len(lrs) != M:
            raise ValueError(f"{len(lrs)} learning rates for a model batch of {M} models")
        self.mb = model_batch
        self.optimizer = optimizer
        self.lr = lrs
        self.regression = regression
        self.betas, self.eps, self.weight_decay = betas, eps, weight_decay
        self.step_count = [0] * M
        self.grads = None                           # contiguous, the layout of the batch's parameter buffer
        self.exp_avg = self.exp_avg_sq = None       # [m]: model m's moments, views of the two contiguous moment buffers
        self._moments = None

    def _loss_kind(self) -> int:
        reg = self.regression if self.regression is not None else getattr(self.mb.models[0], "regression", True)
        return N.LOSS_MSE if reg else N.LOSS_CE2

    def _prepare(self, batches):
        eng, B = self.mb._engines(batches)
        nt = self.mb.models[0].node_types
        dev = batches[0].x_dict[nt[0]].device
        flat = self.mb._bind(dev)
        M = len(self.mb)
        xs = [torch.cat([b.x_dict[t] for b in batches]) if M > 1 else batches[0].x_dict[t] for t in nt]
        return eng, B, xs, flat, dev

    def train_step(self, batches, active: Optional[Sequence[bool]] = None) -> torch.Tensor:
        """One optimisation step of every model on its batch (same graph count per batch); returns the losses [M] (device).
        ``active[m]`` false: model m's step is computed but its parameters, moments and step count are left as they are."""
        eng, B, xs, flat, dev = self._prepare(batches)
        M = len(self.mb)
        n = eng.n_params
        if self.grads is None or self.grads.device != dev or self.grads.numel() != n:
            self.grads = torch.empty(n, dtype=torch.float32, device=dev)
            self._moments = torch.zeros(2, n, dtype=torch.float32, device=dev)
            offs = self.mb.offsets
            self.exp_avg = [self._moments[0, offs[m]:offs[m + 1]] for m in range(M)]
            self.exp_avg_sq = [self._moments[1, offs[m]:offs[m + 1]] for m in range(M)]
        y = torch.cat([b.y.reshape(-1) for b in batches]) if M > 1 else batches[0].y
        out = eng.forward(xs, flat, train=True, n_models=M)
        for m in self.mb.models:
            m._fwd_token = object()
        loss, dout = eng.loss(out, y, self._loss_kind(), want_grad=True, n_models=M)
        eng.backward(dout, flat, grads=self.grads)
        self._optimizer_step(active, dev)
        return loss

    def _optimizer_step(self, active, dev) -> None:
        """One launch for every model: each with its own step count and learning rate, inactive ones untouched."""
        M = len(self.mb)
        act = [True] * M if active is None else [bool(a) for a in active]
        if len(act) != M:
            raise ValueError("one active flag per model expected")
        for m in range(M):
            if act[m]:
                self.step_count[m] += 1
        stream = torch.cuda.current_stream(dev).cuda_stream
        buf, offs = self.mb.buffer, self.mb.offsets
        with torch.cuda.device(dev):
            if self.optimizer == "adam":
                N.adam_step_models(buf.data_ptr(), self.grads.data_ptr(), self._moments[0].data_ptr(), self._moments[1].data_ptr(), offs,
                                   [self.step_count[m] if act[m] else 0 for m in range(M)], self.lr, self.betas[0], self.betas[1],
                                   self.eps, self.weight_decay, stream)
            else:
                N.sgd_step_models(buf.data_ptr(), self.grads.data_ptr(), offs, self.lr, act, stream)

    @torch.no_grad()
    def infer(self, batches) -> List[torch.Tensor]:
        """Inference of every model on its batch in one native forward; returns the M prediction tensors."""
        eng, B, xs, flat, dev = self._prepare(batches)
        M = len(self.mb)
        out = eng.forward(xs, flat, train=False, n_models=M)
        rows = out.shape[0] // M
        return [m._finish(out[i * rows:(i + 1) * rows], B) for i, m in enumerate(self.mb.models)]
