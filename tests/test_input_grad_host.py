"""CPU checks of mshgnn_input_grad: argument validation, and a compute call without a device fails loudly."""
import ctypes

import pytest

from ms_hgnn import _native as N
from ms_hgnn import morphology as M
from ms_hgnn.engine import build_spec

ERR_ARG, ERR_CUDA, ERR_WORKSPACE = -1, -2, -3


def _plan():
    tpl = M.K4_SOLO_COM
    spec = build_spec(tpl.node_types, tpl.nodes_per_graph, {"base": 6, "joint": 2}, tpl.edge_types, tpl.edges,
                      ("gt", "gs", "center_bb"), 128, 2, True, "base", "base", 6, {}, None)
    return N.NativePlan(spec)


def _call(plan, B, params, dx, ws, ws_bytes, mode):
    arr = (ctypes.c_void_p * len(dx))(*dx) if dx is not None else None
    return N.lib().mshgnn_input_grad(plan.handle if plan is not None else None, B, params, arr, ws, ws_bytes, mode, None)


@pytest.fixture(scope="module")
def setup():
    plan = _plan()
    need = plan.workspace_bytes(4, True, N.MODE_TC)
    buf = ctypes.create_string_buffer(need + 1024)
    ws = (ctypes.addressof(buf) + 255) & ~255
    return plan, buf, ws, need


def test_input_grad_rejects_bad_arguments(setup):
    plan, _, ws, need = setup
    dx = [ws, ws]
    for mode in (N.MODE_FP32, N.MODE_TC, N.MODE_TC_1X):
        n = plan.workspace_bytes(4, True, mode)
        assert _call(None, 4, ws, dx, ws, n, mode) == ERR_ARG
        assert _call(plan, 4, ws, dx, ws, n, 7) == ERR_ARG
        assert _call(plan, 4, None, dx, ws, n, mode) == ERR_ARG
        assert _call(plan, 4, ws, None, ws, n, mode) == ERR_ARG
        assert _call(plan, 0, ws, dx, ws, n, mode) == ERR_ARG
        assert _call(plan, 4, ws, dx, None, n, mode) == ERR_ARG
        assert _call(plan, 4, ws, dx, ws + 16, n, mode) == ERR_ARG                  # workspace not 256-byte aligned
        assert _call(plan, 4, ws, dx, ws, n - 1, mode) == ERR_WORKSPACE
        assert b"workspace too small" in N.lib().mshgnn_last_error()
        assert _call(plan, 4, ws, [ws + 2, None], ws, n, mode) == ERR_ARG          # dx rows must be 4-byte aligned
        assert _call(plan, 4, ws, [None, None], ws, n, mode) == 0                   # nothing requested: nothing to do


def test_input_grad_without_gpu_fails_with_cuda_error(setup):
    import torch
    if torch.cuda.is_available():
        pytest.skip("CUDA present")
    plan, _, ws, need = setup
    for mode in (N.MODE_FP32, N.MODE_TC):
        assert _call(plan, 4, ws, [ws, None], ws, plan.workspace_bytes(4, True, mode), mode) == ERR_CUDA
    with pytest.raises(RuntimeError, match="mshgnn_input_grad failed"):
        plan.input_grad(4, ws, [ws, ws], ws, need, N.MODE_TC, None)


def test_profile_read_accepts_the_old_kind_count():
    ms = (ctypes.c_double * N.NUM_KERNEL_KINDS)()
    cnt = (ctypes.c_int64 * N.NUM_KERNEL_KINDS)()
    assert N.lib().mshgnn_profile_read(ms, cnt, 19) == 0
    assert N.lib().mshgnn_profile_read(ms, cnt, 18) == ERR_ARG
    assert N.lib().mshgnn_kernel_kind_name(19) == b"dx_encoder"
