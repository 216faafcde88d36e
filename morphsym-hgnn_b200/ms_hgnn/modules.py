"""Drop-in ``nn.Module`` shell around the native engine.

Keeps the reference's module tree (so ``state_dict()`` / ``load_state_dict()`` use the
reference's key names, SURVEY 3.3) while the arithmetic runs in libmshgnn_b200.so:

    encoder.lins.<type>.{weight,bias}
    convs.<l>.convs.<src___rel___dst>.lin_rel.{weight,bias}, ...lin_root.weight
    base_transform.{0,2}.{weight,bias}
    decoder.{weight,bias}

All parameters are fp32 views into ONE flat buffer (the layout the kernels, the fused optimizer
and the data-parallel all-reduce work on).
"""
from __future__ import annotations

import math
from typing import Dict, List, Optional, Sequence, Tuple

import torch
from torch import nn

from . import _native as N
from .engine import Engine, build_spec

EdgeType = Tuple[str, str, str]


def edge_key(et: EdgeType) -> str:
    return "<" + "___".join(et) + ">"


class ParamLinear(nn.Module):
    """Parameter holder with torch_geometric.nn.Linear's shapes and initialisation."""

    def __init__(self, in_features: int, out_features: int, bias: bool = True):
        super().__init__()
        self.in_features, self.out_features = in_features, out_features
        self.weight = nn.Parameter(torch.empty(out_features, in_features, dtype=torch.float32))
        self.bias = nn.Parameter(torch.empty(out_features, dtype=torch.float32)) if bias else None
        self.reset_parameters()

    def reset_parameters(self):
        bound = 1.0 / math.sqrt(self.in_features) if self.in_features > 0 else 0.0
        with torch.no_grad():
            self.weight.uniform_(-bound, bound)
            if self.bias is not None:
                self.bias.uniform_(-bound, bound)

    def forward(self, *a, **k):  # pragma: no cover
        raise RuntimeError("ParamLinear only holds parameters; the arithmetic runs in the native engine")


class GraphConvParams(nn.Module):
    def __init__(self, hidden: int, aggr: str):
        super().__init__()
        self.aggr = aggr
        self.lin_rel = ParamLinear(hidden, hidden, bias=True)
        self.lin_root = ParamLinear(hidden, hidden, bias=False)

    def reset_parameters(self):
        self.lin_rel.reset_parameters()
        self.lin_root.reset_parameters()


class HeteroConvParams(nn.Module):
    def __init__(self, hidden: int, edge_types: Sequence[EdgeType], mean_relations: Sequence[str]):
        super().__init__()
        self.convs = nn.ModuleDict(
            {edge_key(e): GraphConvParams(hidden, "mean" if e[1] in mean_relations else "add") for e in edge_types})

    def reset_parameters(self):
        for c in self.convs.values():
            c.reset_parameters()


class LazyEncoder(nn.Module):
    """HeteroDictLinear(-1, H, node_types): per-type Linear sized on first use."""

    def __init__(self, hidden: int, node_types: Sequence[str]):
        super().__init__()
        self.hidden = hidden
        self.node_types = list(node_types)
        self.lins = nn.ModuleDict()

    @property
    def materialized(self) -> bool:
        return len(self.lins) == len(self.node_types)

    def materialize(self, in_dims: Dict[str, int], device=None):
        for t in self.node_types:
            if t not in self.lins:
                lin = ParamLinear(int(in_dims[t]), self.hidden, bias=True)
                self.lins[t] = lin.to(device) if device is not None else lin

    def reset_parameters(self):
        for l in self.lins.values():
            l.reset_parameters()


class _HGNNFn(torch.autograd.Function):
    """forward/backward through the native engine; gradients come back as views of one flat buffer."""

    @staticmethod
    def forward(ctx, model, engine, n_x, *tensors):
        x = tensors[:n_x]
        out = engine.forward(x, model._flat, train=True)
        ctx.model, ctx.engine = model, engine
        ctx.n_x = n_x
        ctx.x_dtype = x[0].dtype
        ctx.token = model._fwd_token = object()
        return out

    @staticmethod
    def backward(ctx, dout):
        model, engine = ctx.model, ctx.engine
        if model._fwd_token is not ctx.token:
            raise RuntimeError("the native workspace was overwritten by a later forward(); "
                               "call backward() before the next training forward of this model")
        n_x = ctx.n_x
        want_x = list(ctx.needs_input_grad[3:3 + n_x])
        # a frozen model runs the input-only backward; without input gradients the launches are those of a plain training step
        want_p = any(ctx.needs_input_grad[3 + n_x:]) or not any(want_x)
        g = engine.backward(dout, model._flat, param_grads=want_p)
        grads = [g[o:o + n].view(s) for (o, n, s) in model._views] if want_p else [None] * len(model._views)
        dx = [None] * n_x
        if any(want_x):
            dx = engine.input_grad(want_x, model._flat)
            dx = [d if (d is None or d.dtype == ctx.x_dtype) else d.to(ctx.x_dtype) for d in dx]
        return (None, None, None) + tuple(dx) + tuple(grads)


class NativeHGNN(nn.Module):
    """Shared implementation of the seven reference model classes."""

    morph_sym = False            # base_transform + residual (MS-HGNN) or plain ReLU (MI-HGNN)
    decode_node = "foot"
    mean_relations: Tuple[str, ...] = ()
    fixed_nodes_per_graph: Optional[Dict[str, int]] = None
    mode = N.MODE_FP32
    # edge_index validation (one native launch, mshgnn_check_edges): "always" = every call, mismatch reported without a host
    # sync (raises at the latest at the next forward / assert_edges_valid()); "sync" = every call, raises immediately (one
    # stream synchronisation per forward); "cached" = only tensor objects not seen before; "never"
    validate_edges = "always"

    def __init__(self, hidden_channels: int, num_layers: int, data_metadata, out_channels: int,
                 activation_fn=None, in_dims: Optional[Dict[str, int]] = None,
                 nodes_per_graph: Optional[Dict[str, int]] = None):
        super().__init__()
        if activation_fn is not None and not isinstance(activation_fn, nn.ReLU):
            raise NotImplementedError("the B200-native kernels fuse ReLU; other activation functions are not available")
        self.activation = activation_fn if activation_fn is not None else nn.ReLU()
        node_types, edge_types = data_metadata
        self.hidden_channels = int(hidden_channels)
        self.num_layers = int(num_layers)
        self.node_types = list(node_types)
        self.edge_types = [tuple(e) for e in edge_types]
        self._out_channels = int(out_channels)
        self._user_nodes_per_graph = dict(nodes_per_graph) if nodes_per_graph else None

        self.encoder = LazyEncoder(self.hidden_channels, self.node_types)
        self.convs = nn.ModuleList(
            [HeteroConvParams(self.hidden_channels, self.edge_types, self.mean_relations) for _ in range(self.num_layers)])
        if self.morph_sym:
            self.base_transform = nn.Sequential(nn.Linear(self.hidden_channels, self.hidden_channels), nn.ReLU(),
                                                nn.Linear(self.hidden_channels, self.hidden_channels))
        self.decoder = ParamLinear(self.hidden_channels, self._out_channels, bias=True)
        if in_dims is not None:
            self.encoder.materialize(in_dims)

        self._engines: Dict[tuple, Engine] = {}
        self._flat: Optional[torch.Tensor] = None
        self._views: List[Tuple[int, int, Tuple[int, ...]]] = []
        self._flat_params: List[nn.Parameter] = []
        self._edge_ok: Dict[tuple, tuple] = {}
        self._edge_first: set = set()
        self._edge_flag: Optional[torch.Tensor] = None
        self._fwd_token = None

    _MODES = {"fp32": N.MODE_FP32, "tc": N.MODE_TC, "tc1x": N.MODE_TC_1X}

    def set_mode(self, mode) -> "NativeHGNN":
        """Arithmetic mode of the native kernels: 'fp32' (SIMT fp32 FMA, the 1e-4 parity mode), 'tc' (tcgen05, split-fp16
        operands = 3 MMAs per product, fp32 accumulate: fp32-class accuracy) or 'tc1x' (tcgen05, one fp16 MMA per
        product: 1e-3 on predictions only, for inference)."""
        code = self._MODES[mode] if isinstance(mode, str) else int(mode)
        self.mode = code
        for e in self._engines.values():
            e.mode = code
        return self

    def __getstate__(self):
        # native handles / device buffers are rebuilt lazily after copy or unpickle
        d = self.__dict__.copy()
        d["_engines"] = {}
        d["_flat"] = None
        d["_views"] = []
        d["_flat_params"] = []
        d["_edge_ok"] = {}
        d["_edge_first"] = set()
        d["_edge_flag"] = None
        d["_fwd_token"] = None
        d.pop("_last_engine", None)
        return d

    # ---- reference API ----------------------------------------------------------------
    def reset_parameters(self):
        self.encoder.reset_parameters()
        for c in self.convs:
            c.reset_parameters()
        if self.morph_sym:
            self.base_transform[0].reset_parameters()
            self.base_transform[2].reset_parameters()
        self.decoder.reset_parameters()

    def load_state_dict(self, state_dict, strict: bool = True, assign: bool = False):
        if not self.encoder.materialized:
            dims = {}
            for t in self.node_types:
                k = f"encoder.lins.{t}.weight"
                if k in state_dict:
                    dims[t] = state_dict[k].shape[1]
            if len(dims) == len(self.node_types):
                dev = self.decoder.weight.device
                self.encoder.materialize(dims, dev)
        return super().load_state_dict(state_dict, strict=strict, assign=assign)

    # ---- hooks for subclasses -----------------------------------------------------------
    def _in_sign(self, in_dims: Dict[str, int]) -> Dict[str, Optional[List[float]]]:
        return {}

    def _out_sign(self) -> Optional[List[float]]:
        return None

    def _finish(self, out: torch.Tensor, B: int) -> torch.Tensor:
        return out

    # ---- flat parameter buffer ----------------------------------------------------------
    def _ordered_params(self) -> List[Tuple[str, nn.Parameter]]:
        named = dict(self.named_parameters())
        eng = next(iter(self._engines.values()))
        return [(name, named[name]) for (name, _, _) in eng.param_layout()]

    def _ensure_flat(self, device) -> None:
        eng = next(iter(self._engines.values()))
        layout = eng.param_layout()
        named = dict(self.named_parameters())
        ok = (self._flat is not None and self._flat.device == device)
        if ok:
            base = self._flat.data_ptr()
            for (name, off, shape) in layout:
                p = named[name]
                if p.data_ptr() != base + off * 4 or p.dtype != torch.float32 or tuple(p.shape) != tuple(shape):
                    ok = False
                    break
        if ok:
            return
        for (name, off, shape) in layout:
            p = named[name]
            if tuple(p.shape) != tuple(shape):
                raise RuntimeError(f"parameter {name} has shape {tuple(p.shape)}, expected {tuple(shape)}")
            if p.device != device:
                raise RuntimeError(f"parameter {name} is on {p.device} but the inputs are on {device}; "
                                   "move the model with .to(device) first")
        flat = torch.empty(eng.n_params, dtype=torch.float32, device=device)
        with torch.no_grad():
            for (name, off, shape) in layout:
                p = named[name]
                n = p.numel()
                flat[off:off + n].copy_(p.detach().reshape(-1))
                p.data = flat[off:off + n].view(shape)
        self._flat = flat
        self._views = [(off, int(torch.Size(shape).numel()), tuple(shape)) for (_, off, shape) in layout]
        self._flat_params = [named[name] for (name, _, _) in layout]

    @property
    def flat_parameters(self) -> torch.Tensor:
        """The flat fp32 buffer all parameters are views of (available after the first forward)."""
        if self._flat is None:
            raise RuntimeError("the flat parameter buffer exists after the first forward pass")
        return self._flat

    # ---- template handling --------------------------------------------------------------
    def _nodes_per_graph(self, x_dict) -> Tuple[int, Dict[str, int]]:
        fixed = self._user_nodes_per_graph or self.fixed_nodes_per_graph
        rows = {t: x_dict[t].shape[0] for t in self.node_types}
        if fixed:
            t0 = self.node_types[0]
            if rows[t0] % fixed[t0]:
                raise ValueError(f"x_dict['{t0}'] has {rows[t0]} rows, not a multiple of {fixed[t0]}")
            B = rows[t0] // fixed[t0]
            return B, {t: fixed[t] for t in self.node_types}
        # MI-HGNN datasets have exactly one base node per graph (flexibleDataset.py:L317-323)
        if "base" not in rows:
            raise ValueError("cannot infer the batch size: pass nodes_per_graph=... to the constructor")
        B = rows["base"]
        if B < 1:
            raise ValueError("empty batch")
        out = {}
        for t in self.node_types:
            if rows[t] % B:
                raise ValueError(f"x_dict['{t}'] has {rows[t]} rows for {B} graphs")
            out[t] = rows[t] // B
        return B, out

    def _template_from_batch(self, edge_index_dict, B: int, npg: Dict[str, int]):
        edges = {}
        for et in self.edge_types:
            if et not in edge_index_dict:
                raise KeyError(f"edge_index_dict is missing edge type {et}")
            ei = edge_index_dict[et]
            if ei.dim() != 2 or ei.shape[0] != 2 or ei.shape[1] % B:
                raise ValueError(f"edge_index of {et} must be [2, E*{B}], got {tuple(ei.shape)}")
            E = ei.shape[1] // B
            first = ei[:, :E].detach().to("cpu", torch.long)
            src, dst = first[0].tolist(), first[1].tolist()
            if any(s < 0 or s >= npg[et[0]] for s in src) or any(d < 0 or d >= npg[et[2]] for d in dst):
                raise ValueError(f"edge_index of {et} is not a graph-major batch of one morphology template")
            edges[et] = (src, dst)
        return edges

    def _raise_deferred_edge_error(self) -> None:
        """The native edge check raises a flag in pinned host memory; it is read here without synchronising, so a
        mismatch in step n is reported at the latest by the forward call of step n + 1 (or by assert_edges_valid())."""
        flag = self._edge_flag
        if flag is not None and int(flag[0]) != 0:
            code = int(flag[0])
            flag.zero_()
            raise ValueError(f"edge_index of edge type #{code - 1} in an EARLIER batch was not the morphology template tiled over "
                             "the batch (graph-major PyG batch layout); the results of that step are invalid.  The B200-native "
                             "path only runs fixed-template batches and has no fallback")

    def assert_edges_valid(self) -> None:
        """Synchronises and raises if any batch validated so far failed the native edge_index check."""
        if self._edge_flag is not None:
            torch.cuda.synchronize()
            self._raise_deferred_edge_error()

    def _edges_match(self, edge_index_dict, B: int, eng: Engine, device) -> bool:
        """True iff every edge_index equals the engine's template tiled B times (bit-exact, SURVEY 3.4).

        Shapes / dtypes are checked on the host; the values by ONE native kernel launch (mshgnn_check_edges) that raises a
        flag in pinned host memory.  The first batch of every (template, B, device) is checked synchronously - a wrong
        template fails right here - later batches without a host sync ('always': every call; 'cached': only tensor objects
        not seen before); a late mismatch raises at the next forward."""
        if self.validate_edges == "never":
            return True
        eis = []
        for et in self.edge_types:
            if et not in edge_index_dict:
                raise KeyError(f"edge_index_dict is missing edge type {et}")
            ei = edge_index_dict[et]
            if ei.device != device:
                raise ValueError("edge_index tensors must live on the same device as the node features")
            E = len(eng._edges[et][0])
            if ei.dim() != 2 or tuple(ei.shape) != (2, E * B):
                return False
            eis.append(ei)
        if self.validate_edges == "cached":
            key = (id(eng), B, tuple((id(e), e._version) for e in eis))
            hit = self._edge_ok.get(key)
            if hit is not None and all(a is b for a, b in zip(hit, eis)):      # the cache holds the tensors: ids cannot be reused
                return True
        if self._edge_flag is None:
            self._edge_flag = torch.zeros(1, dtype=torch.int32).pin_memory()
        eis_c = [e if (e.dtype == torch.long and e.is_contiguous()) else e.to(torch.long).contiguous() for e in eis]
        stream = torch.cuda.current_stream(device).cuda_stream
        with torch.cuda.device(device):
            eng.plan.check_edges(B, [e.data_ptr() for e in eis_c], self._edge_flag.data_ptr(), stream)
        first = (id(eng), B, str(device))
        if first not in self._edge_first or self.validate_edges == "sync":
            torch.cuda.current_stream(device).synchronize()
            if int(self._edge_flag[0]) != 0:
                self._edge_flag.zero_()
                return False
            if len(self._edge_first) > 256:
                self._edge_first.clear()
            self._edge_first.add(first)
        if self.validate_edges == "cached":
            if len(self._edge_ok) > 64:
                self._edge_ok.clear()
            self._edge_ok[key] = tuple(eis)
        return True

    def _engine_for(self, x_dict, edge_index_dict) -> Tuple[Engine, int]:
        self._raise_deferred_edge_error()
        B, npg = self._nodes_per_graph(x_dict)
        in_dims = {t: int(x_dict[t].shape[1]) for t in self.node_types}
        device = x_dict[self.node_types[0]].device
        if not self.encoder.materialized:
            self.encoder.materialize(in_dims, self.decoder.weight.device)
        for t in self.node_types:
            if self.encoder.lins[t].in_features != in_dims[t]:
                raise ValueError(f"x_dict['{t}'] has width {in_dims[t]}, the encoder expects {self.encoder.lins[t].in_features}")
        for eng in self._engines.values():
            if eng._npg == npg and self._edges_match(edge_index_dict, B, eng, device):
                return eng, B
        # unseen template: read the first graph's edges once (host copy), compile, then verify the whole batch
        edges = self._template_from_batch(edge_index_dict, B, npg)
        key = (tuple(sorted(npg.items())), tuple((et, tuple(edges[et][0]), tuple(edges[et][1])) for et in self.edge_types))
        eng = self._engines.get(key)
        if eng is None:
            spec = build_spec(self.node_types, npg, in_dims, self.edge_types, edges, self.mean_relations,
                              self.hidden_channels, self.num_layers, self.morph_sym, "base" if self.morph_sym else None,
                              self.decode_node, self._out_channels, self._in_sign(in_dims), self._out_sign(), pad_hidden=True)
            eng = Engine(spec, self.mode)
            eng._edges = edges
            eng._npg = npg
        if not self._edges_match(edge_index_dict, B, eng, device):
            raise ValueError("edge_index_dict is not one morphology template tiled over the batch (graph-major PyG "
                             "batch layout); the B200-native path only runs fixed-template batches and has no fallback")
        self._engines[key] = eng
        return eng, B

    # ---- forward ------------------------------------------------------------------------
    def forward(self, x_dict, edge_index_dict):
        x0 = x_dict[self.node_types[0]]
        if x0.device.type != "cuda":
            raise RuntimeError("ms_hgnn (B200-native) has no CPU path: move the batch and the model to a CUDA device")
        eng, B = self._engine_for(x_dict, edge_index_dict)
        self._last_engine = eng
        self._ensure_flat(x0.device)
        xs = [x_dict[t] for t in self.node_types]          # never mutated (the reference mutates its input dict)
        need_grad = torch.is_grad_enabled() and (any(p.requires_grad for p in self._flat_params) or any(t.requires_grad for t in xs))
        if need_grad:
            out = _HGNNFn.apply(self, eng, len(xs), *xs, *self._flat_params)
        else:
            out = eng.forward(xs, self._flat, train=False)
        out = self._finish(out, B)
        # fp16 node features (MSHGNN_F16: half the host -> device bytes of a batch) are an INPUT format: results stay fp32
        return out if (out.dtype == x0.dtype or x0.dtype == torch.float16) else out.to(x0.dtype)


class _NativeLossFn(torch.autograd.Function):
    """Fused loss head (value + d loss / d out in one native pass)."""

    @staticmethod
    def forward(ctx, out2d, labels, kind, engine):
        loss, dout = engine.loss(out2d, labels, kind, want_grad=True)
        ctx.save_for_backward(dout)
        return loss[0]

    @staticmethod
    def backward(ctx, g):
        (dout,) = ctx.saved_tensors
        return dout * g, None, None, None


def native_loss(model: "NativeHGNN", y_pred: torch.Tensor, y: torch.Tensor, kind: int) -> torch.Tensor:
    """MSE (kind=LOSS_MSE) or per-foot 2-way CE (LOSS_CE2) through the native fused loss kernel.

    ``y_pred`` is the (reshaped) model output; gradients flow back into the native backward pass."""
    eng = getattr(model, "_last_engine", None)
    if eng is None:
        raise RuntimeError("native_loss() needs a preceding forward pass of the model")
    C = eng.spec["out_channels"]
    out2d = y_pred.reshape(-1, C)
    if out2d.dtype != torch.float32:
        out2d = out2d.float()
    out2d = out2d.contiguous()
    labels = y.reshape(-1)
    if torch.is_grad_enabled() and out2d.requires_grad:
        return _NativeLossFn.apply(out2d, labels, kind, eng)
    loss, _ = eng.loss(out2d, labels, kind, want_grad=False)
    return loss[0]
