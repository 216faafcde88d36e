"""Host-side engine: owns the native plan, the flat parameter buffer and the device workspace.

PyTorch is used for device memory, streams and autograd plumbing only; all arithmetic of the
hot path runs in libmshgnn_b200.so.  There is no fallback: on a machine without CUDA (or with
inputs on the CPU) every compute entry point raises.
"""
from __future__ import annotations

from typing import Dict, List, Optional, Sequence, Tuple

import torch

from . import _native as N

EdgeType = Tuple[str, str, str]


def build_spec(node_types: Sequence[str], nodes_per_graph: Dict[str, int], in_width: Dict[str, int],
               edge_types: Sequence[EdgeType], edges: Dict[EdgeType, Tuple[List[int], List[int]]],
               mean_relations: Sequence[str], hidden: int, num_layers: int, morph_sym: bool, mlp_type: Optional[str],
               decode_type: str, out_channels: int, in_sign: Dict[str, Optional[List[float]]],
               out_sign: Optional[List[float]], pad_hidden: bool = False) -> dict:
    """Plain-dict model description for NativePlan.  ``pad_hidden``: accept hidden widths 1..128 (the model runs zero-padded
    on the 128-wide kernels; parameters and gradients stay in its own layout)."""
    ti = {t: i for i, t in enumerate(node_types)}
    spec = {
        "node_types": list(node_types),
        "edge_types": [tuple(e) for e in edge_types],
        "nodes_per_graph": [int(nodes_per_graph[t]) for t in node_types],
        "in_width": [int(in_width[t]) for t in node_types],
        "edges": [(ti[e[0]], ti[e[2]], e[1] in mean_relations, list(edges[tuple(e)][0]), list(edges[tuple(e)][1]))
                  for e in edge_types],
        "hidden": hidden, "num_layers": num_layers, "morph_sym": morph_sym,
        "mlp_type": ti[mlp_type] if (morph_sym and mlp_type is not None) else -1,
        "decode_type": ti[decode_type], "out_channels": out_channels,
        "in_sign": [in_sign.get(t) for t in node_types], "out_sign": out_sign,
    }
    if pad_hidden:
        spec["pad_hidden"] = True
    return spec


def _dtype_code(t: torch.Tensor) -> int:
    if t.dtype == torch.float32:
        return N.F32
    if t.dtype == torch.float64:
        return N.F64
    if t.dtype == torch.float16:
        return N.F16
    if t.dtype == torch.int64:
        return N.I64
    raise TypeError(f"unsupported dtype {t.dtype} (float32, float64, float16 features or int64 labels expected)")


class Engine:
    """One compiled (model, morphology template).  Not thread-safe (single workspace)."""

    def __init__(self, spec: dict, mode: int = N.MODE_FP32):
        self.spec = spec
        self.plan = N.NativePlan(spec)
        self.mode = mode
        self.n_params = self.plan.n_params
        self._ws: Optional[torch.Tensor] = None
        self._ws_key = None
        self._train_ctx = None        # (B, x tensors) of the last train-mode forward

    # ---- parameter layout ------------------------------------------------------------
    def param_layout(self) -> List[Tuple[str, int, Tuple[int, ...]]]:
        """[(reference state-dict name, flat offset, shape)] in named_parameters() order."""
        s = self.spec
        H = s["hidden"]
        out = []
        for i, t in enumerate(s["node_types"]):
            o, _ = self.plan.param_offset(N.P_ENC_W, 0, i); out.append((f"encoder.lins.{t}.weight", o, (H, s["in_width"][i])))
            o, _ = self.plan.param_offset(N.P_ENC_B, 0, i); out.append((f"encoder.lins.{t}.bias", o, (H,)))
        for l in range(s["num_layers"]):
            for e, et in enumerate(s["edge_types"]):
                key = "<" + "___".join(et) + ">"
                o, _ = self.plan.param_offset(N.P_REL_W, l, e); out.append((f"convs.{l}.convs.{key}.lin_rel.weight", o, (H, H)))
                o, _ = self.plan.param_offset(N.P_REL_B, l, e); out.append((f"convs.{l}.convs.{key}.lin_rel.bias", o, (H,)))
                o, _ = self.plan.param_offset(N.P_ROOT_W, l, e); out.append((f"convs.{l}.convs.{key}.lin_root.weight", o, (H, H)))
        if s["morph_sym"]:
            for i, j in ((0, 0), (1, 2)):
                o, _ = self.plan.param_offset(N.P_MLP_W, 0, i); out.append((f"base_transform.{j}.weight", o, (H, H)))
                o, _ = self.plan.param_offset(N.P_MLP_B, 0, i); out.append((f"base_transform.{j}.bias", o, (H,)))
        o, _ = self.plan.param_offset(N.P_DEC_W); out.append(("decoder.weight", o, (s["out_channels"], H)))
        o, _ = self.plan.param_offset(N.P_DEC_B); out.append(("decoder.bias", o, (s["out_channels"],)))
        return out

    # ---- workspace --------------------------------------------------------------------
    def workspace(self, B: int, train: bool, device) -> torch.Tensor:
        need = self.plan.workspace_bytes(B, train, self.mode)
        if self._ws is None or self._ws.numel() < need or self._ws.device != device:
            self._ws = None
            self._ws = torch.empty(need, dtype=torch.uint8, device=device)
        return self._ws

    # ---- compute ----------------------------------------------------------------------
    def _check_inputs(self, x: Sequence[torch.Tensor]) -> Tuple[int, int]:
        s = self.spec
        if len(x) != len(s["node_types"]):
            raise ValueError("one feature tensor per node type expected")
        dev = x[0].device
        if dev.type != "cuda":
            raise RuntimeError("ms_hgnn (B200-native) has no CPU path: node features must be CUDA tensors")
        B = None
        for i, t in enumerate(x):
            if t.device != dev:
                raise ValueError("all node feature tensors must live on the same device")
            if t.dim() != 2 or t.shape[1] != s["in_width"][i]:
                raise ValueError(f"x[{s['node_types'][i]}] must be [B*{s['nodes_per_graph'][i]}, {s['in_width'][i]}], got {tuple(t.shape)}")
            if t.shape[0] % s["nodes_per_graph"][i]:
                raise ValueError(f"x[{s['node_types'][i]}] has {t.shape[0]} rows, not a multiple of {s['nodes_per_graph'][i]}")
            b = t.shape[0] // s["nodes_per_graph"][i]
            if B is None:
                B = b
            elif b != B:
                raise ValueError("node feature tensors disagree on the number of graphs")
            if t.dtype != x[0].dtype:
                raise TypeError("all node feature tensors must share one dtype")
        if B is None or B < 1:
            raise ValueError("empty batch")
        return B, _dtype_code(x[0])

    def forward(self, x: Sequence[torch.Tensor], flat_params: torch.Tensor, train: bool) -> torch.Tensor:
        B, xd = self._check_inputs(x)
        x = [t.contiguous() for t in x]
        dev = x[0].device
        if flat_params.device != dev or flat_params.dtype != torch.float32 or flat_params.numel() != self.n_params:
            raise RuntimeError("flat parameter buffer mismatch")
        ws = self.workspace(B, train, dev)
        out = torch.empty(self.plan.out_rows(B), self.spec["out_channels"], dtype=torch.float32, device=dev)
        stream = torch.cuda.current_stream(dev).cuda_stream
        with torch.cuda.device(dev):
            self.plan.forward(B, [t.data_ptr() for t in x], xd, flat_params.data_ptr(), out.data_ptr(), ws.data_ptr(),
                              ws.numel(), train, self.mode, stream)
        self._train_ctx = (B, x, xd) if train else None
        return out

    def loss(self, out: torch.Tensor, labels: torch.Tensor, kind: int, want_grad: bool = True, loss_scale: float = 1.0):
        """Returns (loss [1] fp32 device tensor, dout or None)."""
        dev = out.device
        B = out.shape[0] // self.spec["nodes_per_graph"][self.spec["decode_type"]]
        labels = labels.contiguous()
        n_expected = out.numel() if kind == N.LOSS_MSE else out.shape[0]
        if labels.numel() != n_expected:
            raise ValueError(f"labels have {labels.numel()} elements, expected {n_expected}")
        if labels.device != dev:
            raise ValueError("labels must live on the same device as the predictions")
        ws = self.workspace(B, self._train_ctx is not None, dev)
        loss = torch.empty(1, dtype=torch.float32, device=dev)
        dout = torch.empty_like(out) if want_grad else None
        stream = torch.cuda.current_stream(dev).cuda_stream
        with torch.cuda.device(dev):
            self.plan.loss(B, kind, out.data_ptr(), labels.data_ptr(), _dtype_code(labels), float(loss_scale), loss.data_ptr(),
                           dout.data_ptr() if want_grad else None, ws.data_ptr(), ws.numel(), stream)
        return loss, dout

    def encoder_param_end(self) -> int:
        """Flat offset of the first non-encoder parameter (the encoder block comes first, reference named_parameters() order)."""
        return min(o for (name, o, _) in self.param_layout() if not name.startswith("encoder."))

    def backward(self, dout: torch.Tensor, flat_params: torch.Tensor, grads: Optional[torch.Tensor] = None,
                 layers_ready: Optional[torch.cuda.Event] = None, param_grads: bool = True) -> Optional[torch.Tensor]:
        """d loss / d params into ``grads`` (allocated when None) and returned.  ``param_grads=False`` runs the input-only
        backward of a frozen model: no weight gradient is computed and None is returned; input_grad() may follow."""
        if self._train_ctx is None:
            raise RuntimeError("backward() needs a preceding forward(train=True) on the same engine")
        B, x, xd = self._train_ctx
        dev = x[0].device
        dout = dout.contiguous()
        if dout.dtype != torch.float32:
            dout = dout.float()
        if dout.numel() != self.plan.out_rows(B) * self.spec["out_channels"]:
            raise ValueError("dout has the wrong number of elements")
        if not param_grads:
            grads = None
        elif grads is None:
            grads = torch.empty(self.n_params, dtype=torch.float32, device=dev)
        ws = self.workspace(B, True, dev)
        stream = torch.cuda.current_stream(dev).cuda_stream
        with torch.cuda.device(dev):
            if layers_ready is not None:
                # torch creates the CUDA event lazily at its first record(): make sure the handle exists
                if layers_ready.cuda_event == 0:
                    layers_ready.record(torch.cuda.current_stream(dev))
            self.plan.backward(B, [t.data_ptr() for t in x], xd, flat_params.data_ptr(), dout.data_ptr(),
                               grads.data_ptr() if grads is not None else None,
                               ws.data_ptr(), ws.numel(), self.mode, stream,
                               layers_ready.cuda_event if layers_ready is not None else None)
        return grads

    def input_grad(self, which: Sequence[bool], flat_params: torch.Tensor) -> List[Optional[torch.Tensor]]:
        """d loss / d x[t] (fp32, the shape of x[t]) for every node type t with which[t] true, None for the others.  Runs after
        backward() of the last train-mode forward, on the same workspace."""
        if self._train_ctx is None:
            raise RuntimeError("input_grad() needs a preceding forward(train=True) and backward() on the same engine")
        B, x, _ = self._train_ctx
        dev = x[0].device
        out = [torch.empty(t.shape, dtype=torch.float32, device=dev) if w else None for t, w in zip(x, which)]
        ws = self.workspace(B, True, dev)
        stream = torch.cuda.current_stream(dev).cuda_stream
        with torch.cuda.device(dev):
            self.plan.input_grad(B, flat_params.data_ptr(), [t.data_ptr() if t is not None else None for t in out], ws.data_ptr(),
                                 ws.numel(), self.mode, stream)
        return out
