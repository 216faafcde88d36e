"""CPU checks of hidden widths below 128 (MSHGNN_PLAN_PAD_HIDDEN): the caller's parameter layout, plan validation and the
unchanged H = 128 plan (no compute calls)."""
import ctypes

import pytest
import torch

from helpers import oracle_model
from ms_hgnn import _native as N
from ms_hgnn import morphology as M
from ms_hgnn.engine import Engine, build_spec
from ms_hgnn.synthetic import CONFIGS, build_model

ERR_ARG = -1
WIDTHS = [1, 10, 64, 100, 127, 128]


def _spec_of(cfg, hidden, layers, pad_hidden=True):
    """The spec NativeHGNN._engine_for builds for cfg's model class at this width."""
    nm = build_model(cfg, hidden=hidden, layers=layers)
    tpl = M.TEMPLATES[cfg.template]
    return build_spec(nm.node_types, tpl.nodes_per_graph, cfg.in_width, nm.edge_types, tpl.edges, nm.mean_relations, hidden, layers,
                      nm.morph_sym, "base" if nm.morph_sym else None, nm.decode_node, nm._out_channels, nm._in_sign(dict(cfg.in_width)),
                      nm._out_sign(), pad_hidden=pad_hidden)


@pytest.mark.parametrize("hidden", WIDTHS)
@pytest.mark.parametrize("name", sorted(CONFIGS))
def test_param_layout_matches_the_oracle_model(name, hidden):
    cfg = CONFIGS[name]
    layers = 3
    eng = Engine(_spec_of(cfg, hidden, layers))
    om = oracle_model(cfg, hidden=hidden, layers=layers)
    named = [(n, tuple(p.shape)) for n, p in om.named_parameters()]
    layout = eng.param_layout()
    assert [(n, s) for n, _, s in layout] == named
    off = 0
    for (n, o, s) in layout:
        assert o == off, n
        off += int(torch.Size(s).numel())
    assert eng.n_params == off == sum(p.numel() for p in om.parameters())
    assert eng.plan.describe()["hidden"] == hidden and eng.plan.describe()["kernel_hidden"] == 128


def test_plan_create_ex_validates_the_width():
    spec = _spec_of(CONFIGS["mini_cheetah-k4-contact"], 64, 2, pad_hidden=False)
    with pytest.raises(RuntimeError, match="H=128"):
        N.NativePlan(spec)                                                  # mshgnn_plan_create
    with pytest.raises(RuntimeError, match="H=128"):
        N.NativePlan(dict(spec, pad_hidden=False))
    N.NativePlan(dict(spec, pad_hidden=True))
    for bad in (0, 129, 256):
        with pytest.raises(RuntimeError, match="128") as e:
            N.NativePlan(dict(spec, hidden=bad, pad_hidden=True))
        assert "mshgnn_plan_create_ex" in str(e.value)


def test_unknown_plan_flags_are_rejected():
    spec = _spec_of(CONFIGS["solo-c2-com"], 128, 2, pad_hidden=False)
    plan = N.NativePlan(spec)
    h = ctypes.c_void_p()
    # rebuild the same Desc through the binding's own struct, then call the raw entry point with an unknown bit
    d = _raw_desc(spec)
    assert N.lib().mshgnn_plan_create_ex(ctypes.byref(d), 2, ctypes.byref(h)) == ERR_ARG
    assert b"flags" in N.lib().mshgnn_last_error()
    assert N.lib().mshgnn_plan_create_ex(ctypes.byref(d), 0, ctypes.byref(h)) == 0
    assert N.lib().mshgnn_param_count(h) == plan.n_params
    N.lib().mshgnn_plan_destroy(h)


def _raw_desc(spec):
    d = N.Desc()
    keep = []
    d.n_node_types = len(spec["nodes_per_graph"])
    for t in range(d.n_node_types):
        d.nodes_per_graph[t] = spec["nodes_per_graph"][t]
        d.in_width[t] = spec["in_width"][t]
    d.n_edge_types = len(spec["edges"])
    for e, (st, dt, mean, src, dst) in enumerate(spec["edges"]):
        d.edge_src_type[e] = st; d.edge_dst_type[e] = dt; d.edge_mean[e] = int(bool(mean)); d.edge_count[e] = len(src)
        a = (ctypes.c_int32 * max(len(src), 1))(*src); b = (ctypes.c_int32 * max(len(dst), 1))(*dst)
        keep += [a, b]
        d.edge_src[e] = ctypes.cast(a, ctypes.POINTER(ctypes.c_int32)); d.edge_dst[e] = ctypes.cast(b, ctypes.POINTER(ctypes.c_int32))
    d.hidden = spec["hidden"]; d.num_layers = spec["num_layers"]; d.morph_sym = int(bool(spec["morph_sym"]))
    d.mlp_type = spec["mlp_type"]; d.decode_type = spec["decode_type"]; d.out_channels = spec["out_channels"]
    d._keep = keep
    return d


@pytest.mark.parametrize("name", ["mini_cheetah-k4-contact", "a1-c2-grf", "solo12-k4-com", "mi-grf"])
def test_width_128_with_the_flag_is_the_plain_plan(name):
    cfg = CONFIGS[name]
    plain = Engine(_spec_of(cfg, 128, 8, pad_hidden=False))
    flagged = Engine(_spec_of(cfg, 128, 8, pad_hidden=True))
    assert "pad_hidden" not in plain.spec and flagged.spec["pad_hidden"]
    assert plain.n_params == flagged.n_params
    assert plain.param_layout() == flagged.param_layout()
    assert plain.plan.describe() == flagged.plan.describe()
    for B in (1, 200, 6144, 16384):
        for mode in (N.MODE_FP32, N.MODE_TC, N.MODE_TC_1X):
            assert plain.plan.dw_layout(B, mode) == flagged.plan.dw_layout(B, mode)
            for train in (False, True):
                assert plain.plan.workspace_bytes(B, train, mode) == flagged.plan.workspace_bytes(B, train, mode)


def test_padded_workspace_adds_the_internal_parameter_and_gradient_buffers():
    cfg = CONFIGS["mini_cheetah-k4-contact"]
    wide = Engine(_spec_of(cfg, 128, 8, pad_hidden=False))
    narrow = Engine(_spec_of(cfg, 10, 8))
    internal = -(-wide.n_params * 4 // 256) * 256
    for B in (1, 16384):
        for mode in (N.MODE_FP32, N.MODE_TC):
            assert narrow.plan.workspace_bytes(B, False, mode) == wide.plan.workspace_bytes(B, False, mode) + internal
            assert narrow.plan.workspace_bytes(B, True, mode) == wide.plan.workspace_bytes(B, True, mode) + 2 * internal
            for layer in range(-1, 8):                        # the ReLU masks keep their 128-bit rows
                assert narrow.plan.relu_mask_offset(B, mode, layer) == wide.plan.relu_mask_offset(B, mode, layer)


def test_profile_read_accepts_every_kind_count_since_19():
    ms = (ctypes.c_double * N.NUM_KERNEL_KINDS)()
    cnt = (ctypes.c_int64 * N.NUM_KERNEL_KINDS)()
    assert N.NUM_KERNEL_KINDS == 21
    for n in (19, 20, 21):
        assert N.lib().mshgnn_profile_read(ms, cnt, n) == 0
    assert N.lib().mshgnn_profile_read(ms, cnt, 18) == ERR_ARG
    assert N.lib().mshgnn_kernel_kind_name(19) == b"dx_encoder"
    assert N.lib().mshgnn_kernel_kind_name(20) == b"pad_params"
