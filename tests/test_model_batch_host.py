"""CPU checks of model batches (mshgnn_*_models): the M = 1 layout equals the single-model one, model row blocks are padded to
the stack kernel's row tiles with the single-model splits inside, and unsupported requests are refused before any device work."""
import ctypes

import pytest

from ms_hgnn import _native as N
from ms_hgnn.model_batch import ModelBatch, ModelBatchTrainer
from ms_hgnn.synthetic import CONFIGS, build_model
from test_hidden_width_host import _spec_of

ERR_ARG = -1
MODES = [N.MODE_FP32, N.MODE_TC, N.MODE_TC_1X]


@pytest.fixture
def restore_options():
    saved = {k: N.get_option(k) for k in ("stack", "stack_pair")}
    yield
    for k, v in saved.items():
        N.set_option(k, v)


@pytest.mark.parametrize("name", ["mini_cheetah-k4-contact", "solo12-k4-com", "mi-grf"])
@pytest.mark.parametrize("B", [1, 100, 2048, 6144, 16384])
@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("train", [0, 1])
def test_one_model_is_the_single_model_layout(name, B, mode, train):
    plan = N.NativePlan(_spec_of(CONFIGS[name], 128, 3))
    L = N.lib()
    assert L.mshgnn_workspace_bytes_models(plan.handle, 1, B, train, mode) == plan.workspace_bytes(B, train, mode)


def _layout_line(capfd, plan, M, B):
    """The MSHGNN_DEBUG_LAYOUT line of a tensor-core training layout: (M, B, Bm, per-model split and partial-slot text)."""
    capfd.readouterr()
    assert plan.workspace_bytes_models(M, B, True, N.MODE_TC) > 0
    line = [l for l in capfd.readouterr().err.splitlines() if l.startswith("mshgnn layout")][-1]
    head, rest = line.split(":", 1)
    kv = dict(t.split("=") for t in head.split()[2:])
    return int(kv["M"]), int(kv["B"]), int(kv["Bm"]), rest


@pytest.mark.parametrize("hidden", [10, 128])
@pytest.mark.parametrize("B,M,Bm", [(1, 2, 128), (64, 5, 128), (100, 2, 128), (129, 5, 256), (300, 2, 384), (300, 32, 512),
                                    (2048, 2, 2048), (2048, 4, 2048), (100, 64, 256)])
def test_per_model_blocks_and_splits(capfd, monkeypatch, restore_options, hidden, B, M, Bm):
    """Model m's rows are a block of Bm = B rounded up to 128 rows, or to 256 once M * B reaches the CTA-pair kernel's 6144
    graphs; its weight-gradient splits and partial slots are exactly those of a single-model call on B graphs."""
    monkeypatch.setenv("MSHGNN_DEBUG_LAYOUT", "1")
    N.set_option("stack", 1)
    N.set_option("stack_pair", 1)
    plan = N.NativePlan(_spec_of(CONFIGS["mini_cheetah-k4-contact"], hidden, 3))
    m1, b1, bm1, rest1 = _layout_line(capfd, plan, 1, B)
    m, b, bm, rest = _layout_line(capfd, plan, M, B)
    assert (m1, b1, m, b, bm) == (1, B, M, B, Bm)
    assert bm1 == -(-B // (256 if B >= 6144 else 128)) * (256 if B >= 6144 else 128)
    assert rest == rest1
    assert plan.workspace_bytes_models(M, B, True, N.MODE_TC) > plan.workspace_bytes(B, True, N.MODE_TC)


def test_entry_points_refuse_bad_model_counts_and_modes(restore_options):
    plan = N.NativePlan(_spec_of(CONFIGS["mini_cheetah-k4-contact"], 128, 2))
    L = N.lib()
    h = plan.handle
    assert L.mshgnn_workspace_bytes_models(h, 0, 64, 1, N.MODE_TC) == -1
    assert L.mshgnn_workspace_bytes_models(h, 2, 0, 1, N.MODE_TC) == -1
    assert L.mshgnn_workspace_bytes_models(h, 2, 64, 1, N.MODE_FP32) == -1
    assert L.mshgnn_workspace_bytes_models(h, 1024, 64, 1, N.MODE_TC) == -1          # grid limits: at most 1023 models
    assert L.mshgnn_workspace_bytes_models(h, 1023, 1, 1, N.MODE_TC) > 0
    x = (ctypes.c_void_p * 3)(1, 1, 1)        # never dereferenced: every call below fails its argument checks first
    dummy = ctypes.c_void_p(256)
    for M, mode in ((0, N.MODE_TC), (-1, N.MODE_TC), (2, N.MODE_FP32)):
        assert L.mshgnn_forward_models(h, M, 64, x, N.F32, dummy, dummy, dummy, 1 << 40, 1, mode, None) == ERR_ARG
        assert L.mshgnn_backward_models(h, M, 64, x, N.F32, dummy, dummy, dummy, dummy, 1 << 40, mode, None, None) == ERR_ARG
    assert L.mshgnn_loss_models(h, 0, 64, N.LOSS_CE2, dummy, dummy, 0, 1.0, dummy, dummy, dummy, 1 << 40, None) == ERR_ARG
    N.set_option("stack", 0)
    assert L.mshgnn_workspace_bytes_models(h, 2, 64, 1, N.MODE_TC) == -1
    assert L.mshgnn_forward_models(h, 2, 64, x, N.F32, dummy, dummy, dummy, 1 << 40, 1, N.MODE_TC, None) == ERR_ARG
    assert b"stack" in L.mshgnn_last_error()
    assert L.mshgnn_backward_models(h, 2, 64, x, N.F32, dummy, dummy, dummy, dummy, 1 << 40, N.MODE_TC, None, None) == ERR_ARG


def test_model_batch_rejects_mixed_configurations():
    cfg = CONFIGS["mini_cheetah-k4-contact"]
    a, b = build_model(cfg, hidden=16, layers=2, seed=0), build_model(cfg, hidden=16, layers=2, seed=1)
    assert len(ModelBatch([a, b])) == 2
    with pytest.raises(ValueError, match="configuration"):
        ModelBatch([a, build_model(cfg, hidden=32, layers=2)])
    with pytest.raises(ValueError, match="configuration"):
        ModelBatch([a, build_model(cfg, hidden=16, layers=3)])
    with pytest.raises(ValueError, match="class"):
        ModelBatch([a, build_model(CONFIGS["mi-contact"], hidden=16, layers=2)])
    with pytest.raises(ValueError, match="configuration"):
        ModelBatch([a, build_model(cfg, hidden=16, layers=2).set_mode("tc1x")])
    with pytest.raises(ValueError):
        ModelBatch([])
    with pytest.raises(ValueError, match="process group"):
        ModelBatchTrainer(ModelBatch([a, b]), process_group=object())
