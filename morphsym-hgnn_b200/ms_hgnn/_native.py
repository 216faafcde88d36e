"""ctypes binding of libmshgnn_b200.so (include/mshgnn_b200.h).

There is no CPU fallback: if the library cannot be built/loaded this module raises, and every
compute call raises ``RuntimeError`` with the library's error text when it returns non-zero.
"""
from __future__ import annotations

import ctypes as C
import importlib.util
import os
from typing import Optional, Sequence

_PKG = os.path.dirname(os.path.abspath(__file__))
_ROOT = os.path.dirname(_PKG)                      # morphsym-hgnn_b200/
LIB_PATH = os.path.join(_ROOT, "lib", "libmshgnn_b200.so")

MAX_NODE_TYPES = 4
MAX_EDGE_TYPES = 16

F32, F64, I64, F16 = 0, 1, 2, 3
MODE_FP32, MODE_TC, MODE_TC_1X = 0, 1, 2
PLAN_PAD_HIDDEN = 1
LOSS_MSE, LOSS_CE2 = 0, 1
METRIC_COM, METRIC_GRF_WORLD = 2, 3
# slots of mshgnn_step_metrics_ex (include/mshgnn_b200.h): 0..19 additive states (also added into epoch), 20+ derived values
COM_SSE, COM_N, COM_SSE_LIN, COM_SSE_ANG, COM_N_HALF, COM_COS_LIN, COM_COS_ANG, COM_ROWS = range(8)
COM_MSE, COM_RMSE, COM_MSE_LIN, COM_MSE_ANG, COM_COS_SIM_LIN, COM_COS_SIM_ANG, COM_AVG_COS_SIM = range(20, 27)
GRF_SSE, GRF_SAE, GRF_N, GRF_SSE_WORLD, GRF_SAE_WORLD, GRF_N_WORLD = range(6)
GRF_MSE, GRF_RMSE, GRF_L1, GRF_MSE_WORLD, GRF_RMSE_WORLD, GRF_L1_WORLD = range(20, 26)
P_ENC_W, P_ENC_B, P_REL_W, P_REL_B, P_ROOT_W, P_MLP_W, P_MLP_B, P_DEC_W, P_DEC_B = range(9)

# every symbol include/mshgnn_b200.h declares
EXPORTS = (
    "mshgnn_plan_create", "mshgnn_plan_destroy", "mshgnn_param_count", "mshgnn_param_offset",
    "mshgnn_workspace_bytes", "mshgnn_out_rows", "mshgnn_forward", "mshgnn_loss", "mshgnn_backward",
    "mshgnn_adam_step", "mshgnn_sgd_step", "mshgnn_plan_describe", "mshgnn_launch_count",
    "mshgnn_last_error", "mshgnn_version", "mshgnn_profile_enable", "mshgnn_profile_read", "mshgnn_kernel_kind_name",
    "mshgnn_relu_mask_offset", "mshgnn_build_windows", "mshgnn_step_metrics", "mshgnn_dw_layout",
    "mshgnn_check_edges", "mshgnn_set_option", "mshgnn_get_option", "mshgnn_stack_status",
    "mshgnn_backward_staged", "mshgnn_input_grad", "mshgnn_plan_create_ex", "mshgnn_step_metrics_ex",
    "mshgnn_workspace_bytes_models", "mshgnn_forward_models", "mshgnn_loss_models", "mshgnn_backward_models",
    "mshgnn_plan_create_models", "mshgnn_param_offset_model", "mshgnn_adam_step_models", "mshgnn_sgd_step_models",
)
MAX_MODELS = 1023


class Desc(C.Structure):
    _fields_ = [
        ("n_node_types", C.c_int32),
        ("nodes_per_graph", C.c_int32 * MAX_NODE_TYPES),
        ("in_width", C.c_int32 * MAX_NODE_TYPES),
        ("n_edge_types", C.c_int32),
        ("edge_src_type", C.c_int32 * MAX_EDGE_TYPES),
        ("edge_dst_type", C.c_int32 * MAX_EDGE_TYPES),
        ("edge_mean", C.c_int32 * MAX_EDGE_TYPES),
        ("edge_count", C.c_int32 * MAX_EDGE_TYPES),
        ("edge_src", C.POINTER(C.c_int32) * MAX_EDGE_TYPES),
        ("edge_dst", C.POINTER(C.c_int32) * MAX_EDGE_TYPES),
        ("hidden", C.c_int32),
        ("num_layers", C.c_int32),
        ("morph_sym", C.c_int32),
        ("mlp_type", C.c_int32),
        ("decode_type", C.c_int32),
        ("out_channels", C.c_int32),
        ("in_sign", C.POINTER(C.c_float) * MAX_NODE_TYPES),
        ("out_sign", C.POINTER(C.c_float)),
    ]


class WindowDesc(C.Structure):
    """mshgnn_window_desc (include/mshgnn_b200.h)."""
    _fields_ = [
        ("history_length", C.c_int32), ("seq_cols", C.c_int32), ("label_cols", C.c_int32), ("n_node_types", C.c_int32),
        ("nodes_per_graph", C.c_int32 * MAX_NODE_TYPES), ("blocks_per_node", C.c_int32 * MAX_NODE_TYPES),
        ("block_len", C.c_int32 * MAX_NODE_TYPES),
        ("normalize", C.c_int32), ("n_labels", C.c_int32),
        ("block_col", C.POINTER(C.c_int32)), ("block_sign", C.POINTER(C.c_int32)),
        ("label_col", C.POINTER(C.c_int32)), ("label_sign", C.POINTER(C.c_int32)),
    ]


class MetricArgs(C.Structure):
    """mshgnn_metric_args (include/mshgnn_b200.h)."""
    _fields_ = [("n_base", C.c_int32), ("y_mean", C.c_void_p), ("y_std", C.c_void_p), ("quat", C.c_void_p),
                ("quat_dtype", C.c_int32), ("z_only", C.c_int32)]


_lib: Optional[C.CDLL] = None


def _build_if_needed() -> None:
    spec = importlib.util.spec_from_file_location("_mshgnn_build", os.path.join(_ROOT, "build.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    mod.build()


def lib() -> C.CDLL:
    """Load (building in-tree when the .so is absent or stale and nvcc exists) the native library."""
    global _lib
    if _lib is not None:
        return _lib
    override = os.environ.get("MSHGNN_LIB")      # measurement hook: load another build of the same ABI (same-box A/B of two commits)
    if override:
        if not os.path.exists(override):
            raise RuntimeError(f"MSHGNN_LIB={override} does not exist")
        path = override
    else:
        path = LIB_PATH
        try:
            _build_if_needed()
        except Exception as e:  # no nvcc on the box: a prebuilt .so must be there
            if not os.path.exists(LIB_PATH):
                raise RuntimeError(f"libmshgnn_b200.so is missing and could not be built: {e}") from e
    L = C.CDLL(path)
    vp, i32, i64, f32 = C.c_void_p, C.c_int32, C.c_int64, C.c_float
    L.mshgnn_plan_create.argtypes = [C.POINTER(Desc), C.POINTER(vp)]; L.mshgnn_plan_create.restype = C.c_int
    if hasattr(L, "mshgnn_plan_create_ex"):      # absent from builds before it (MSHGNN_LIB A/B runs against an older commit)
        L.mshgnn_plan_create_ex.argtypes = [C.POINTER(Desc), i32, C.POINTER(vp)]; L.mshgnn_plan_create_ex.restype = C.c_int
    L.mshgnn_plan_destroy.argtypes = [vp]; L.mshgnn_plan_destroy.restype = None
    L.mshgnn_param_count.argtypes = [vp]; L.mshgnn_param_count.restype = i64
    L.mshgnn_param_offset.argtypes = [vp, i32, i32, i32, C.POINTER(i64), C.POINTER(i64)]; L.mshgnn_param_offset.restype = C.c_int
    L.mshgnn_workspace_bytes.argtypes = [vp, i64, i32, i32]; L.mshgnn_workspace_bytes.restype = i64
    L.mshgnn_dw_layout.argtypes = [vp, i64, i32, C.POINTER(C.c_int32), i64]; L.mshgnn_dw_layout.restype = i64
    L.mshgnn_out_rows.argtypes = [vp, i64]; L.mshgnn_out_rows.restype = i64
    L.mshgnn_forward.argtypes = [vp, i64, C.POINTER(vp), i32, vp, vp, vp, i64, i32, i32, vp]; L.mshgnn_forward.restype = C.c_int
    L.mshgnn_loss.argtypes = [vp, i64, i32, vp, vp, i32, f32, vp, vp, vp, i64, vp]; L.mshgnn_loss.restype = C.c_int
    L.mshgnn_backward.argtypes = [vp, i64, C.POINTER(vp), i32, vp, vp, vp, vp, i64, i32, vp]; L.mshgnn_backward.restype = C.c_int
    L.mshgnn_backward_staged.argtypes = [vp, i64, C.POINTER(vp), i32, vp, vp, vp, vp, i64, i32, vp, vp]; L.mshgnn_backward_staged.restype = C.c_int
    if hasattr(L, "mshgnn_input_grad"):          # absent from builds before it (MSHGNN_LIB A/B runs against an older commit)
        L.mshgnn_input_grad.argtypes = [vp, i64, vp, C.POINTER(vp), vp, i64, i32, vp]; L.mshgnn_input_grad.restype = C.c_int
    if hasattr(L, "mshgnn_forward_models"):      # absent from builds before it (MSHGNN_LIB A/B runs against an older commit)
        L.mshgnn_workspace_bytes_models.argtypes = [vp, i64, i64, i32, i32]; L.mshgnn_workspace_bytes_models.restype = i64
        L.mshgnn_forward_models.argtypes = [vp, i64, i64, C.POINTER(vp), i32, vp, vp, vp, i64, i32, i32, vp]; L.mshgnn_forward_models.restype = C.c_int
        L.mshgnn_loss_models.argtypes = [vp, i64, i64, i32, vp, vp, i32, f32, vp, vp, vp, i64, vp]; L.mshgnn_loss_models.restype = C.c_int
        L.mshgnn_backward_models.argtypes = [vp, i64, i64, C.POINTER(vp), i32, vp, vp, vp, vp, i64, i32, vp, vp]
        L.mshgnn_backward_models.restype = C.c_int
    if hasattr(L, "mshgnn_plan_create_models"):  # absent from builds before it (MSHGNN_LIB A/B runs against an older commit)
        L.mshgnn_plan_create_models.argtypes = [C.POINTER(Desc), i32, C.POINTER(i32), C.POINTER(vp)]
        L.mshgnn_plan_create_models.restype = C.c_int
        L.mshgnn_param_offset_model.argtypes = [vp, i32, i32, i32, i32, C.POINTER(i64), C.POINTER(i64)]
        L.mshgnn_param_offset_model.restype = C.c_int
        L.mshgnn_adam_step_models.argtypes = [vp, vp, vp, vp, i32, C.POINTER(i64), C.POINTER(i64), C.POINTER(f32), f32, f32, f32, f32, vp]
        L.mshgnn_adam_step_models.restype = C.c_int
        L.mshgnn_sgd_step_models.argtypes = [vp, vp, i32, C.POINTER(i64), C.POINTER(f32), C.POINTER(i32), vp]
        L.mshgnn_sgd_step_models.restype = C.c_int
    L.mshgnn_adam_step.argtypes = [vp, vp, vp, vp, i64, i64, f32, f32, f32, f32, f32, vp]; L.mshgnn_adam_step.restype = C.c_int
    L.mshgnn_sgd_step.argtypes = [vp, vp, i64, f32, vp]; L.mshgnn_sgd_step.restype = C.c_int
    L.mshgnn_plan_describe.argtypes = [vp, C.c_char_p, i64]; L.mshgnn_plan_describe.restype = i64
    L.mshgnn_launch_count.argtypes = []; L.mshgnn_launch_count.restype = i64
    L.mshgnn_last_error.argtypes = []; L.mshgnn_last_error.restype = C.c_char_p
    L.mshgnn_version.argtypes = []; L.mshgnn_version.restype = C.c_char_p
    L.mshgnn_profile_enable.argtypes = [i32]; L.mshgnn_profile_enable.restype = C.c_int
    L.mshgnn_profile_read.argtypes = [C.POINTER(C.c_double), C.POINTER(i64), i32]; L.mshgnn_profile_read.restype = C.c_int
    L.mshgnn_kernel_kind_name.argtypes = [i32]; L.mshgnn_kernel_kind_name.restype = C.c_char_p
    L.mshgnn_relu_mask_offset.argtypes = [vp, i64, i32, i32, C.POINTER(i64), C.POINTER(i64), C.POINTER(i64)]
    L.mshgnn_relu_mask_offset.restype = C.c_int
    L.mshgnn_build_windows.argtypes = [C.POINTER(WindowDesc), vp, vp, i32, i64, vp, i64, C.POINTER(vp), vp, vp]
    L.mshgnn_build_windows.restype = C.c_int
    L.mshgnn_step_metrics.argtypes = [i32, i64, i32, vp, vp, i32, vp, vp, vp, vp]; L.mshgnn_step_metrics.restype = C.c_int
    if hasattr(L, "mshgnn_step_metrics_ex"):     # absent from builds before it (MSHGNN_LIB A/B runs against an older commit)
        L.mshgnn_step_metrics_ex.argtypes = [i32, C.POINTER(MetricArgs), i64, vp, vp, i32, vp, vp, vp, vp]
        L.mshgnn_step_metrics_ex.restype = C.c_int
    L.mshgnn_check_edges.argtypes = [vp, i64, C.POINTER(vp), vp, vp]; L.mshgnn_check_edges.restype = C.c_int
    L.mshgnn_set_option.argtypes = [C.c_char_p, i32]; L.mshgnn_set_option.restype = C.c_int
    L.mshgnn_get_option.argtypes = [C.c_char_p]; L.mshgnn_get_option.restype = i32
    L.mshgnn_stack_status.argtypes = [vp, i64, i32, i32, vp, C.POINTER(i32)]; L.mshgnn_stack_status.restype = C.c_int
    _lib = L
    return L


def check(rc: int, what: str) -> None:
    if rc != 0:
        raise RuntimeError(f"{what} failed (code {rc}): {lib().mshgnn_last_error().decode()}")


NUM_KERNEL_KINDS = 21


def profile_enable(on: bool) -> None:
    check(lib().mshgnn_profile_enable(int(on)), "mshgnn_profile_enable")


def profile_read() -> dict:
    """{kernel kind name: (total ms, launches)} since the last read (synchronises the recorded events)."""
    ms = (C.c_double * NUM_KERNEL_KINDS)()
    cnt = (C.c_int64 * NUM_KERNEL_KINDS)()
    check(lib().mshgnn_profile_read(ms, cnt, NUM_KERNEL_KINDS), "mshgnn_profile_read")
    out = {}
    for k in range(NUM_KERNEL_KINDS):
        name = lib().mshgnn_kernel_kind_name(k).decode()
        if name and cnt[k]:
            out[name] = (float(ms[k]), int(cnt[k]))
    return out


def launch_count() -> int:
    return int(lib().mshgnn_launch_count())


def set_option(name: str, value: int) -> None:
    """Library switches: 'stack' (1 = cross-layer persistent kernel for the layer loop, 0 = one launch per layer),
    'stack_pair' (0 = never, 1 = CTA-pair stack kernel for batches >= 6144 graphs, 2 = always)."""
    check(lib().mshgnn_set_option(name.encode(), int(value)), "mshgnn_set_option")


def get_option(name: str) -> int:
    return int(lib().mshgnn_get_option(name.encode()))


class NativePlan:
    """Owns a mshgnn_plan*.  ``spec`` is a plain dict (see engine.build_spec); ``spec["pad_hidden"]`` true creates the plan
    with MSHGNN_PLAN_PAD_HIDDEN (hidden 1..128, run zero-padded on the 128-wide kernels).  ``spec["widths"]`` (a list of M
    widths) creates the plan of a model batch of M models of those widths (mshgnn_plan_create_models); ``models`` is then M,
    and None for other plans."""

    def __init__(self, spec: dict):
        L = lib()
        d = Desc()
        nt = len(spec["nodes_per_graph"])
        d.n_node_types = nt
        self._keep = []
        for t in range(nt):
            d.nodes_per_graph[t] = int(spec["nodes_per_graph"][t])
            d.in_width[t] = int(spec["in_width"][t])
            s = spec["in_sign"][t]
            if s is not None:
                arr = (C.c_float * len(s))(*[float(v) for v in s])
                self._keep.append(arr)
                d.in_sign[t] = C.cast(arr, C.POINTER(C.c_float))
        edges = spec["edges"]
        d.n_edge_types = len(edges)
        for e, (st, dt, mean, src, dst) in enumerate(edges):
            d.edge_src_type[e] = st; d.edge_dst_type[e] = dt; d.edge_mean[e] = int(bool(mean)); d.edge_count[e] = len(src)
            a = (C.c_int32 * max(len(src), 1))(*[int(v) for v in src]); b = (C.c_int32 * max(len(dst), 1))(*[int(v) for v in dst])
            self._keep += [a, b]
            d.edge_src[e] = C.cast(a, C.POINTER(C.c_int32)); d.edge_dst[e] = C.cast(b, C.POINTER(C.c_int32))
        d.hidden = int(spec["hidden"]); d.num_layers = int(spec["num_layers"])
        d.morph_sym = int(bool(spec["morph_sym"])); d.mlp_type = int(spec["mlp_type"])
        d.decode_type = int(spec["decode_type"]); d.out_channels = int(spec["out_channels"])
        if spec.get("out_sign") is not None:
            arr = (C.c_float * len(spec["out_sign"]))(*[float(v) for v in spec["out_sign"]])
            self._keep.append(arr)
            d.out_sign = C.cast(arr, C.POINTER(C.c_float))
        h = C.c_void_p()
        self.models = None
        if spec.get("widths") is not None:
            w = [int(v) for v in spec["widths"]]
            arr = (C.c_int32 * max(len(w), 1))(*w)
            check(L.mshgnn_plan_create_models(C.byref(d), len(w), arr, C.byref(h)), "mshgnn_plan_create_models")
            self.models = len(w)
        elif spec.get("pad_hidden") and hasattr(L, "mshgnn_plan_create_ex"):     # older builds (MSHGNN_LIB): 128 wide only
            check(L.mshgnn_plan_create_ex(C.byref(d), PLAN_PAD_HIDDEN, C.byref(h)), "mshgnn_plan_create_ex")
        else:
            check(L.mshgnn_plan_create(C.byref(d), C.byref(h)), "mshgnn_plan_create")
        self.handle = h
        self.spec = spec
        self.n_params = int(L.mshgnn_param_count(h))

    def __del__(self):
        try:
            if getattr(self, "handle", None):
                lib().mshgnn_plan_destroy(self.handle)
                self.handle = None
        except Exception:
            pass

    def param_offset(self, kind: int, layer: int = 0, idx: int = 0, model: Optional[int] = None):
        """(offset, numel) of one parameter tensor; ``model``: of model m of a model-batch plan (absolute offset)."""
        off, n = C.c_int64(), C.c_int64()
        if model is None:
            check(lib().mshgnn_param_offset(self.handle, kind, layer, idx, C.byref(off), C.byref(n)), "mshgnn_param_offset")
        else:
            check(lib().mshgnn_param_offset_model(self.handle, model, kind, layer, idx, C.byref(off), C.byref(n)),
                  "mshgnn_param_offset_model")
        return off.value, n.value

    def workspace_bytes(self, B: int, train: bool, mode: int = MODE_FP32) -> int:
        n = int(lib().mshgnn_workspace_bytes(self.handle, B, int(train), mode))
        if n < 0:
            raise RuntimeError("mshgnn_workspace_bytes failed")
        return n

    def workspace_bytes_models(self, M: int, B: int, train: bool, mode: int) -> int:
        """Workspace of a model batch of M models with B graphs each (mshgnn_workspace_bytes_models)."""
        n = int(lib().mshgnn_workspace_bytes_models(self.handle, M, B, int(train), mode))
        if n < 0:
            raise RuntimeError(f"mshgnn_workspace_bytes_models failed: no model batch of {M} x {B} graphs in mode {mode} "
                               "(M > 1 needs a tensor-core mode and the stack kernel)")
        return n

    def dw_layout(self, B: int, mode: int = MODE_TC):
        """Per layer launch of the weight-gradient GEMM: (tasks, row splits, rows per split, first partial slot)."""
        buf = (C.c_int32 * 64)()
        n = int(lib().mshgnn_dw_layout(self.handle, B, mode, buf, 64))
        if n < 0:
            raise RuntimeError("mshgnn_dw_layout failed")
        return [tuple(buf[4 * l + k] for k in range(4)) for l in range(n)]

    def out_rows(self, B: int) -> int:
        return int(lib().mshgnn_out_rows(self.handle, B))

    def relu_mask_offset(self, B: int, mode: int, layer: int):
        """(byte offset in the training workspace, slots, padded rows) of the stored ReLU sign pattern (layer -1 = encoder)."""
        off, ns, bp = C.c_int64(), C.c_int64(), C.c_int64()
        check(lib().mshgnn_relu_mask_offset(self.handle, B, mode, layer, C.byref(off), C.byref(ns), C.byref(bp)), "mshgnn_relu_mask_offset")
        return off.value, ns.value, bp.value

    def describe(self) -> dict:
        import json
        n = int(lib().mshgnn_plan_describe(self.handle, None, 0))
        buf = C.create_string_buffer(n)
        lib().mshgnn_plan_describe(self.handle, buf, n)
        return json.loads(buf.value.decode())

    def check_edges(self, B, ei_ptrs: Sequence[int], flag_ptr, stream):
        """One launch: raises *flag when an edge_index is not the plan's template tiled over B graphs (no host sync)."""
        arr = (C.c_void_p * len(ei_ptrs))(*ei_ptrs)
        check(lib().mshgnn_check_edges(self.handle, B, arr, flag_ptr, stream), "mshgnn_check_edges")

    def stack_status(self, B, train, mode, ws_ptr) -> int:
        """1 when a dependency wait of the last cross-layer launch on this workspace timed out (synchronises)."""
        out = C.c_int32()
        check(lib().mshgnn_stack_status(self.handle, B, int(train), mode, ws_ptr, C.byref(out)), "mshgnn_stack_status")
        return out.value

    # ---- compute (raw device pointers) ----
    def forward(self, B, x_ptrs: Sequence[int], x_dtype, params_ptr, out_ptr, ws_ptr, ws_bytes, train, mode, stream):
        arr = (C.c_void_p * len(x_ptrs))(*x_ptrs)
        check(lib().mshgnn_forward(self.handle, B, arr, x_dtype, params_ptr, out_ptr, ws_ptr, ws_bytes, int(train), mode, stream),
              "mshgnn_forward")

    def loss(self, B, kind, out_ptr, labels_ptr, label_dtype, loss_scale, loss_ptr, dout_ptr, ws_ptr, ws_bytes, stream):
        check(lib().mshgnn_loss(self.handle, B, kind, out_ptr, labels_ptr, label_dtype, loss_scale, loss_ptr, dout_ptr,
                                ws_ptr, ws_bytes, stream), "mshgnn_loss")

    def backward(self, B, x_ptrs, x_dtype, params_ptr, dout_ptr, grads_ptr, ws_ptr, ws_bytes, mode, stream, layers_ready_event=None):
        """grads_ptr None: input-only backward (dX chain for input_grad, no weight gradient)."""
        arr = (C.c_void_p * len(x_ptrs))(*x_ptrs)
        check(lib().mshgnn_backward_staged(self.handle, B, arr, x_dtype, params_ptr, dout_ptr, grads_ptr, ws_ptr, ws_bytes, mode, stream,
                                           layers_ready_event), "mshgnn_backward")

    # ---- model batches: M models of this plan, B graphs each (include/mshgnn_b200.h) ----
    def forward_models(self, M, B, x_ptrs, x_dtype, params_ptr, out_ptr, ws_ptr, ws_bytes, train, mode, stream):
        arr = (C.c_void_p * len(x_ptrs))(*x_ptrs)
        check(lib().mshgnn_forward_models(self.handle, M, B, arr, x_dtype, params_ptr, out_ptr, ws_ptr, ws_bytes, int(train), mode, stream),
              "mshgnn_forward_models")

    def loss_models(self, M, B, kind, out_ptr, labels_ptr, label_dtype, loss_scale, loss_ptr, dout_ptr, ws_ptr, ws_bytes, stream):
        check(lib().mshgnn_loss_models(self.handle, M, B, kind, out_ptr, labels_ptr, label_dtype, loss_scale, loss_ptr, dout_ptr,
                                       ws_ptr, ws_bytes, stream), "mshgnn_loss_models")

    def backward_models(self, M, B, x_ptrs, x_dtype, params_ptr, dout_ptr, grads_ptr, ws_ptr, ws_bytes, mode, stream, layers_ready_event=None):
        arr = (C.c_void_p * len(x_ptrs))(*x_ptrs)
        check(lib().mshgnn_backward_models(self.handle, M, B, arr, x_dtype, params_ptr, dout_ptr, grads_ptr, ws_ptr, ws_bytes, mode, stream,
                                           layers_ready_event), "mshgnn_backward_models")

    def input_grad(self, B, params_ptr, dx_ptrs, ws_ptr, ws_bytes, mode, stream):
        """d loss / d x[t] into the fp32 buffers dx_ptrs[t] (None: skip type t), after backward on the same workspace."""
        arr = (C.c_void_p * len(dx_ptrs))(*dx_ptrs)
        check(lib().mshgnn_input_grad(self.handle, B, params_ptr, arr, ws_ptr, ws_bytes, mode, stream), "mshgnn_input_grad")


METRIC_SLOTS, METRIC_SCRATCH = 32, 296 * 32


def step_metrics(kind, n, feet, out_ptr, labels_ptr, label_dtype, batch_ptr, epoch_ptr, scratch_ptr, stream):
    check(lib().mshgnn_step_metrics(kind, n, feet, out_ptr, labels_ptr, label_dtype, batch_ptr, epoch_ptr, scratch_ptr, stream),
          "mshgnn_step_metrics")


def step_metrics_ex(kind, args: MetricArgs, n, out_ptr, labels_ptr, label_dtype, batch_ptr, epoch_ptr, scratch_ptr, stream):
    """METRIC_COM / METRIC_GRF_WORLD: ``n`` = graphs, ``args`` the kind's inputs (n_base and stats, or quaternions)."""
    check(lib().mshgnn_step_metrics_ex(kind, C.byref(args), n, out_ptr, labels_ptr, label_dtype, batch_ptr, epoch_ptr, scratch_ptr,
                                       stream), "mshgnn_step_metrics_ex")


def adam_step(params_ptr, grads_ptr, m_ptr, v_ptr, n, step, lr, b1, b2, eps, wd, stream):
    check(lib().mshgnn_adam_step(params_ptr, grads_ptr, m_ptr, v_ptr, n, step, lr, b1, b2, eps, wd, stream), "mshgnn_adam_step")


def sgd_step(params_ptr, grads_ptr, n, lr, stream):
    check(lib().mshgnn_sgd_step(params_ptr, grads_ptr, n, lr, stream), "mshgnn_sgd_step")


def adam_step_models(params_ptr, grads_ptr, m_ptr, v_ptr, offsets: Sequence[int], steps: Sequence[int], lrs: Sequence[float],
                     b1, b2, eps, wd, stream):
    """One Adam launch for M models: model m owns [offsets[m], offsets[m+1]), takes step steps[m] (0: untouched) at lr lrs[m]."""
    M = len(steps)
    if len(offsets) != M + 1 or len(lrs) != M:
        raise ValueError(f"{M} models need {M + 1} offsets and {M} learning rates")
    check(lib().mshgnn_adam_step_models(params_ptr, grads_ptr, m_ptr, v_ptr, M, (C.c_int64 * (M + 1))(*offsets), (C.c_int64 * M)(*steps),
                                        (C.c_float * M)(*lrs), b1, b2, eps, wd, stream), "mshgnn_adam_step_models")


def sgd_step_models(params_ptr, grads_ptr, offsets: Sequence[int], lrs: Sequence[float], active: Sequence[bool], stream):
    """One SGD launch for M models (model m: [offsets[m], offsets[m+1]) at lr lrs[m], untouched when not active[m])."""
    M = len(lrs)
    if len(offsets) != M + 1 or len(active) != M:
        raise ValueError(f"{M} models need {M + 1} offsets and {M} active flags")
    check(lib().mshgnn_sgd_step_models(params_ptr, grads_ptr, M, (C.c_int64 * (M + 1))(*offsets), (C.c_float * M)(*lrs),
                                       (C.c_int32 * M)(*[int(bool(a)) for a in active]), stream), "mshgnn_sgd_step_models")
