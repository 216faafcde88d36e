"""CPU checks of model batches of different hidden widths (mshgnn_plan_create_models): the ragged parameter layout, argument
checks of plan creation and of the entry points, and the Python front ends (no compute calls)."""
import ctypes

import pytest

from ms_hgnn import _native as N
from ms_hgnn.engine import Engine
from ms_hgnn.model_batch import ModelBatch, ModelBatchTrainer
from ms_hgnn.synthetic import CONFIGS, build_model
from test_hidden_width_host import _raw_desc, _spec_of

ERR_ARG = -1
WIDTHS = [128, 10, 64, 1, 37]
NAMES = ["mini_cheetah-k4-contact", "a1-c2-grf", "solo12-k4-com", "mi-com", "mi-grf"]


def _models_plan(spec, widths):
    d = _raw_desc(spec)
    h = ctypes.c_void_p()
    rc = N.lib().mshgnn_plan_create_models(ctypes.byref(d), len(widths), (ctypes.c_int32 * max(len(widths), 1))(*widths), ctypes.byref(h))
    return rc, h


def _single_offsets(plan, spec):
    """Every (kind, layer, idx) -> (offset, numel) of a single-model plan."""
    keys = [(N.P_ENC_W, 0, t) for t in range(len(spec["node_types"]))] + [(N.P_ENC_B, 0, t) for t in range(len(spec["node_types"]))]
    for l in range(spec["num_layers"]):
        for e in range(len(spec["edges"])):
            keys += [(N.P_REL_W, l, e), (N.P_REL_B, l, e), (N.P_ROOT_W, l, e)]
    if spec["morph_sym"]:
        keys += [(N.P_MLP_W, 0, 0), (N.P_MLP_W, 0, 1), (N.P_MLP_B, 0, 0), (N.P_MLP_B, 0, 1)]
    keys += [(N.P_DEC_W, 0, 0), (N.P_DEC_B, 0, 0)]
    return {k: plan.param_offset(*k) for k in keys}


@pytest.mark.parametrize("name", NAMES)
def test_ragged_layout_is_the_single_layouts_end_to_end(name):
    cfg = CONFIGS[name]
    spec = _spec_of(cfg, 128, 3)
    singles = [N.NativePlan(_spec_of(cfg, h, 3)) for h in WIDTHS]
    mixed = N.NativePlan(dict(spec, widths=WIDTHS))
    assert mixed.models == len(WIDTHS)
    assert mixed.n_params == sum(p.n_params for p in singles)
    base = 0
    for m, single in enumerate(singles):
        for key, (off, numel) in _single_offsets(single, spec).items():
            assert mixed.param_offset(*key, model=m) == (base + off, numel), (m, key)
        base += single.n_params
    assert mixed.describe()["hidden_models"] == WIDTHS
    # the Engine front end: model m's named tensors at the absolute offsets, model_offsets the model ranges
    eng = Engine(dict(spec, widths=WIDTHS))
    offs = eng.model_offsets()
    assert offs[0] == 0 and offs[-1] == eng.n_params
    for m, single in enumerate(singles):
        assert offs[m + 1] - offs[m] == single.n_params
        ref = Engine(_spec_of(cfg, WIDTHS[m], 3)).param_layout()
        assert eng.param_layout(m) == [(n, o + offs[m], s) for (n, o, s) in ref]


def test_equal_widths_are_the_uniform_layout():
    cfg = CONFIGS["mini_cheetah-k4-contact"]
    spec = _spec_of(cfg, 128, 3)
    plain = N.NativePlan(spec)
    mixed = N.NativePlan(dict(spec, widths=[128] * 4))
    assert mixed.n_params == 4 * plain.n_params
    for key, (off, numel) in _single_offsets(plain, spec).items():
        for m in range(4):
            assert mixed.param_offset(*key, model=m) == (m * plain.n_params + off, numel)
    for B in (1, 200, 6144):
        for train in (0, 1):
            assert mixed.workspace_bytes_models(4, B, train, N.MODE_TC) == plain.workspace_bytes_models(4, B, train, N.MODE_TC)


def test_one_model_is_the_single_plan():
    spec = _spec_of(CONFIGS["solo12-k4-com"], 37, 3)
    single = N.NativePlan(spec)
    one = N.NativePlan(dict(spec, widths=[37]))
    assert one.models == 1 and one.n_params == single.n_params
    assert one.param_offset(N.P_DEC_W) == single.param_offset(N.P_DEC_W)          # M = 1: mshgnn_param_offset works
    for mode in (N.MODE_FP32, N.MODE_TC):
        assert one.workspace_bytes(100, True, mode) == single.workspace_bytes(100, True, mode)


def test_plan_creation_validates_its_arguments():
    spec = _spec_of(CONFIGS["mini_cheetah-k4-contact"], 128, 2)
    L = N.lib()
    for widths, M, what in (([], 0, b"M must be"), ([16] * 1024, 1024, b"M must be"), ([16, 0], 2, b"hidden=0"), ([129], 1, b"hidden=129"),
                            ([64, 16, 129], 3, b"model 2")):
        d = _raw_desc(spec)
        h = ctypes.c_void_p()
        arr = (ctypes.c_int32 * max(len(widths), 1))(*widths)
        assert L.mshgnn_plan_create_models(ctypes.byref(d), M, arr, ctypes.byref(h)) == ERR_ARG, widths[:4]
        assert what in L.mshgnn_last_error()
        assert not h.value
    d = _raw_desc(spec)
    h = ctypes.c_void_p()
    assert L.mshgnn_plan_create_models(ctypes.byref(d), 2, None, ctypes.byref(h)) == ERR_ARG
    assert b"hidden" in L.mshgnn_last_error()
    rc, h = _models_plan(spec, [16] * 1023)
    assert rc == 0
    L.mshgnn_plan_destroy(h)


def test_entry_points_take_only_the_plan_model_count():
    spec = _spec_of(CONFIGS["mini_cheetah-k4-contact"], 128, 2)
    plan = N.NativePlan(dict(spec, widths=[16, 64, 128]))
    L, h = N.lib(), plan.handle
    off, n = ctypes.c_int64(), ctypes.c_int64()
    assert L.mshgnn_param_offset(h, N.P_DEC_W, 0, 0, ctypes.byref(off), ctypes.byref(n)) == ERR_ARG
    assert b"mshgnn_param_offset_model" in L.mshgnn_last_error()
    assert L.mshgnn_param_offset_model(h, 3, N.P_DEC_W, 0, 0, ctypes.byref(off), ctypes.byref(n)) == ERR_ARG
    assert L.mshgnn_param_offset_model(h, -1, N.P_DEC_W, 0, 0, ctypes.byref(off), ctypes.byref(n)) == ERR_ARG
    assert L.mshgnn_workspace_bytes_models(h, 3, 64, 1, N.MODE_TC) > 0
    for M in (1, 2, 4):
        assert L.mshgnn_workspace_bytes_models(h, M, 64, 1, N.MODE_TC) == -1
    assert L.mshgnn_workspace_bytes(h, 64, 1, N.MODE_TC) == -1
    x = (ctypes.c_void_p * 3)(1, 1, 1)        # never dereferenced: every call below fails its argument checks first
    dummy = ctypes.c_void_p(256)
    for M in (1, 2, 4):
        assert L.mshgnn_forward_models(h, M, 64, x, N.F32, dummy, dummy, dummy, 1 << 40, 1, N.MODE_TC, None) == ERR_ARG
        assert b"M must be 3" in L.mshgnn_last_error()
        assert L.mshgnn_backward_models(h, M, 64, x, N.F32, dummy, dummy, dummy, dummy, 1 << 40, N.MODE_TC, None, None) == ERR_ARG
        assert L.mshgnn_loss_models(h, M, 64, N.LOSS_CE2, dummy, dummy, 0, 1.0, dummy, dummy, dummy, 1 << 40, None) == ERR_ARG
    assert L.mshgnn_forward(h, 64, x, N.F32, dummy, dummy, dummy, 1 << 40, 1, N.MODE_TC, None) == ERR_ARG
    assert L.mshgnn_backward(h, 64, x, N.F32, dummy, dummy, dummy, dummy, 1 << 40, N.MODE_TC, None) == ERR_ARG
    assert L.mshgnn_loss(h, 64, N.LOSS_CE2, dummy, dummy, 0, 1.0, dummy, dummy, dummy, 1 << 40, None) == ERR_ARG
    assert L.mshgnn_input_grad(h, 64, dummy, x, dummy, 1 << 40, N.MODE_TC, None) == ERR_ARG
    # a mixed plan is a model batch: MODE_FP32 is refused as for any M > 1
    assert L.mshgnn_workspace_bytes_models(h, 3, 64, 1, N.MODE_FP32) == -1


def test_optimizer_entry_points_validate_their_arguments():
    L = N.lib()
    p = ctypes.c_void_p(256)
    offs = (ctypes.c_int64 * 3)(0, 10, 5)                # decreasing
    good = (ctypes.c_int64 * 3)(0, 10, 20)
    steps = (ctypes.c_int64 * 2)(1, 1)
    lrs = (ctypes.c_float * 2)(1e-3, 1e-4)
    assert L.mshgnn_adam_step_models(p, p, p, p, 2, offs, steps, lrs, 0.9, 0.999, 1e-8, 0.0, None) == ERR_ARG
    assert b"decrease" in L.mshgnn_last_error()
    assert L.mshgnn_adam_step_models(p, p, p, p, 0, good, steps, lrs, 0.9, 0.999, 1e-8, 0.0, None) == ERR_ARG
    assert L.mshgnn_adam_step_models(p, p, p, p, 1024, good, steps, lrs, 0.9, 0.999, 1e-8, 0.0, None) == ERR_ARG
    assert L.mshgnn_adam_step_models(p, p, p, p, 2, good, (ctypes.c_int64 * 2)(1, -1), lrs, 0.9, 0.999, 1e-8, 0.0, None) == ERR_ARG
    assert L.mshgnn_adam_step_models(p, p, p, p, 2, good, None, lrs, 0.9, 0.999, 1e-8, 0.0, None) == ERR_ARG
    assert L.mshgnn_adam_step_models(p, p, p, p, 2, good, steps, None, 0.9, 0.999, 1e-8, 0.0, None) == ERR_ARG
    assert L.mshgnn_sgd_step_models(p, p, 2, offs, lrs, None, None) == ERR_ARG
    assert L.mshgnn_sgd_step_models(p, p, 2, None, lrs, None, None) == ERR_ARG
    assert L.mshgnn_sgd_step_models(None, p, 2, good, lrs, None, None) == ERR_ARG
    with pytest.raises(ValueError):
        N.adam_step_models(256, 256, 256, 256, [0, 10], [1, 1], [1e-3, 1e-3], 0.9, 0.999, 1e-8, 0.0, None)


def test_model_batch_mixed_hidden_accepts_widths_only():
    cfg = CONFIGS["mini_cheetah-k4-contact"]
    a = build_model(cfg, hidden=16, layers=2, seed=0)
    mb = ModelBatch([a, build_model(cfg, hidden=32, layers=2), build_model(cfg, hidden=128, layers=2)], mixed_hidden=True)
    assert len(mb) == 3
    with pytest.raises(ValueError, match="configuration"):
        ModelBatch([a, build_model(cfg, hidden=32, layers=3)], mixed_hidden=True)
    with pytest.raises(ValueError, match="class"):
        ModelBatch([a, build_model(CONFIGS["mi-contact"], hidden=16, layers=2)], mixed_hidden=True)
    with pytest.raises(ValueError, match="configuration"):
        ModelBatch([a, build_model(cfg, hidden=32, layers=2).set_mode("tc1x")], mixed_hidden=True)
    with pytest.raises(ValueError, match="configuration"):
        ModelBatch([a, build_model(cfg, hidden=32, layers=2)])                 # the default still wants one width


def test_learning_rates_per_model():
    cfg = CONFIGS["mini_cheetah-k4-contact"]
    mb = ModelBatch([build_model(cfg, hidden=h, layers=2) for h in (8, 16, 32)], mixed_hidden=True)
    assert ModelBatchTrainer(mb, lr=1e-3).lr == [1e-3] * 3
    assert ModelBatchTrainer(mb, lr=(1e-4, 1e-3, 2e-3)).lr == [1e-4, 1e-3, 2e-3]
    for bad in ([1e-3, 1e-4], [1e-3] * 4, []):
        with pytest.raises(ValueError, match="learning rates"):
            ModelBatchTrainer(mb, lr=bad)


def test_train_models_checks_sequence_lengths():
    from ms_hgnn.lightning_py.trainer import _per_run, train_models
    assert _per_run(16, "hidden_size", 3) == [16, 16, 16]
    assert _per_run([8, 16, 32], "hidden_size", 3) == [8, 16, 32]
    # the lengths are checked before any dataset is touched
    with pytest.raises(ValueError, match="hidden_size"):
        train_models(None, None, None, True, seeds=[0, 5], hidden_size=[16, 8, 32])
    with pytest.raises(ValueError, match="lr"):
        train_models(None, None, None, True, seeds=[0, 0, 5], lr=[1e-3, 1e-4])
    with pytest.raises(ValueError, match="lr"):
        train_models(None, None, None, True, seeds=[0], hidden_size=16, lr=())
