"""GPU tests of the cross-layer stack kernel (csrc/kernels_stack.cuh) and the native edge_index check.

The stack kernel runs the same tiles as the per-layer launch sequence - same operands, same MMA order, same epilogue
arithmetic - so predictions and loss must be bit-identical between the two paths (and the gradients equal up to the
summation order of the weight-gradient row splits); the oracle parity of the stack path itself is what
tests/test_gpu_parity.py checks (the stack path is the default there).
"""
import pytest
import torch

from helpers import TOL_FP32, oracle_model, oracle_run, rel_err
from ms_hgnn import _native as N
from ms_hgnn.synthetic import CONFIGS, build_model, make_batch

pytestmark = pytest.mark.gpu


@pytest.fixture
def restore_stack_option():
    before, before_pair = N.get_option("stack"), N.get_option("stack_pair")
    yield
    N.set_option("stack", before)
    N.set_option("stack_pair", before_pair)


def _step(nm, cfg, b):
    nm.zero_grad()
    out = nm(b.x_dict, b.edge_index_dict)
    eng = nm._last_engine
    C = eng.spec["out_channels"]
    loss, dout = eng.loss(out.detach().reshape(-1, C).float().contiguous(), b.y, N.LOSS_CE2 if cfg.loss == "ce" else N.LOSS_MSE)
    out.backward(dout.view_as(out).to(out.dtype))
    torch.cuda.synchronize()
    ws = eng._ws
    assert eng.plan.stack_status(b.batch_size, True, eng.mode, ws.data_ptr()) == 0, "a dependency wait of the stack kernel timed out"
    grads = {n: (p.grad.clone() if p.grad is not None else torch.zeros_like(p)) for n, p in nm.named_parameters()}
    return out.detach().clone(), loss.item(), grads


# 5000 / 7000 graphs = 40 / 55 row tiles: two and three L2 chunks (24 row tiles each for the 20-slot templates), the last one short
STACK_CASES = [("mini_cheetah-k4-contact", 1, 3), ("mini_cheetah-k4-contact", 200, 8), ("mini_cheetah-k4-contact", 5000, 8),
               ("mini_cheetah-c2-contact", 1100, 8), ("a1-c2-grf", 300, 8), ("solo12-k4-com", 7000, 8), ("solo-c2-com", 33, 4),
               ("mi-contact", 400, 8), ("mi-com", 77, 2),
               ("mini_cheetah-k4-contact", 300, 15), ("solo12-k4-com", 257, 15)]           # MAX_LAYERS: the longest stack programs


@pytest.mark.parametrize("name,B,layers", STACK_CASES)
def test_stack_kernel_is_bit_identical_to_the_per_layer_launches(name, B, layers, restore_stack_option):
    cfg = CONFIGS[name]
    b = make_batch(cfg, B, seed=B + 1).to("cuda:0")
    nm = build_model(cfg, layers=layers, seed=3).set_mode("tc").to("cuda:0")
    N.set_option("stack", 1)
    n0 = N.launch_count()
    out_s, loss_s, g_s = _step(nm, cfg, b)
    launches_stack = N.launch_count() - n0
    with torch.no_grad():
        inf_s = nm(b.x_dict, b.edge_index_dict).clone()
    N.set_option("stack", 0)
    n0 = N.launch_count()
    out_l, loss_l, g_l = _step(nm, cfg, b)
    launches_layer = N.launch_count() - n0
    with torch.no_grad():
        inf_l = nm(b.x_dict, b.edge_index_dict).clone()
    assert torch.equal(out_s, out_l)
    assert torch.equal(inf_s, inf_l) and torch.equal(inf_s, out_s)
    assert loss_s == loss_l
    # gradients: the dX chain is bit-identical too, but the stack path sums the weight gradients of ALL layers in one launch
    # with its own row-split count (ws_layout), i.e. in a different fp32 summation order over the graphs
    worst = 0.0
    for k in g_l:
        if g_l[k].norm() == 0:
            assert g_s[k].abs().max().item() == 0.0, k
        else:
            worst = max(worst, rel_err(g_s[k], g_l[k]))
    assert worst <= TOL_FP32, worst      # sums over graphs split differently (measured <= 3e-5; both paths are checked against the oracle at 1e-4)
    print(f"stack[{name} B={B} L={layers}]: {launches_stack} launches per train step with the stack kernel, {launches_layer} per layer; "
          f"worst gradient difference between the two paths {worst:.1e}")
    assert launches_stack < launches_layer or layers < 2


# CTA-pair kernel (csrc/kernels_stack2.cuh, cta_group::2 MMAs on two row tiles at once) against the one-CTA stack kernel: the same
# products accumulate in the same order into the same kind of accumulator, so every bit must agree.  B = 129 / 385: the last
# row-tile pair is half padding; 5000 graphs: 20 pairs; 1 graph: a single pair
@pytest.mark.parametrize("name,B,layers,mode", [("mini_cheetah-k4-contact", 1, 3, "tc"), ("mini_cheetah-k4-contact", 129, 8, "tc"),
                                                ("mini_cheetah-k4-contact", 5000, 8, "tc"), ("mini_cheetah-c2-contact", 385, 8, "tc"),
                                                ("solo12-k4-com", 2100, 8, "tc"), ("mi-contact", 400, 8, "tc"),
                                                ("mini_cheetah-k4-contact", 3300, 8, "tc1x"), ("mini_cheetah-k4-contact", 385, 15, "tc"),
                                                ("mi-contact", 400, 15, "tc")])
def test_cta_pair_stack_kernel_is_bit_identical_to_the_one_cta_kernel(name, B, layers, mode, restore_stack_option):
    cfg = CONFIGS[name]
    b = make_batch(cfg, B, seed=B + 2).to("cuda:0")
    nm = build_model(cfg, layers=layers, seed=3).set_mode(mode).to("cuda:0")
    N.set_option("stack", 1)
    res = []
    for pair in (2, 0, 2):                   # 2 = the pair kernel whatever the batch size (1 = only for large batches)
        N.set_option("stack_pair", pair)
        if mode == "tc":
            out, loss, g = _step(nm, cfg, b)
        else:
            out, loss, g = None, 0.0, {}
        with torch.no_grad():
            inf = nm(b.x_dict, b.edge_index_dict).clone()
        torch.cuda.synchronize()
        res.append((out, loss, g, inf))
    for a, c in ((res[0], res[1]), (res[2], res[1])):
        assert torch.equal(a[3], c[3])
        if mode == "tc":
            assert torch.equal(a[0], c[0]) and a[1] == c[1]
            for k in a[2]:
                assert torch.equal(a[2][k], c[2][k]), k


def test_stack_kernel_single_pass_mode_is_bit_identical_too(restore_stack_option):
    cfg = CONFIGS["mini_cheetah-k4-contact"]
    b = make_batch(cfg, 3300, seed=4).to("cuda:0")
    nm = build_model(cfg, layers=8, seed=3).set_mode("tc1x").to("cuda:0")
    outs = []
    for on in (1, 0):
        N.set_option("stack", on)
        with torch.no_grad():
            outs.append(nm(b.x_dict, b.edge_index_dict).clone())
    assert torch.equal(outs[0], outs[1])


@pytest.mark.parametrize("name,B,layers", [("mini_cheetah-k4-contact", 200, 8), ("solo12-k4-com", 257, 8), ("mi-grf", 20, 8)])
def test_per_layer_launch_path_still_matches_the_oracle(name, B, layers, restore_stack_option):
    """Option "stack" = 0 keeps the round-1 launch sequence alive for A/B measurements: same 1e-4 bound."""
    from test_gpu_parity import check_gradients
    N.set_option("stack", 0)
    check_gradients(CONFIGS[name], B, layers, mode="tc")


def test_stack_kernel_repeated_steps_are_deterministic():
    """Dependency counters are reset per launch and nothing depends on CTA timing: ten steps, identical bits."""
    cfg = CONFIGS["mini_cheetah-k4-contact"]
    b = make_batch(cfg, 4000, seed=9).to("cuda:0")
    nm = build_model(cfg, layers=8, seed=3).set_mode("tc").to("cuda:0")
    ref = _step(nm, cfg, b)
    for _ in range(9):
        out, loss, g = _step(nm, cfg, b)
        assert torch.equal(out, ref[0]) and loss == ref[1]
        for k in g:
            assert torch.equal(g[k], ref[2][k]), k


# ---- native edge_index validation (mshgnn_check_edges) ------------------------------------------------------------
def test_wrong_template_is_rejected_immediately():
    cfg = CONFIGS["mini_cheetah-k4-contact"]
    b = make_batch(cfg, 64, seed=1).to("cuda:0")
    nm = build_model(cfg, layers=2, seed=3).to("cuda:0")
    ei = b.edge_index_dict
    et = nm.edge_types[2]
    bad = {k: v.clone() for k, v in ei.items()}
    bad[et][1, 70] += 1                                  # one destination of graph 4 points at the wrong node
    with pytest.raises(ValueError, match="morphology template"):
        nm(b.x_dict, bad)
    nm(b.x_dict, ei)                                     # the good batch still runs


def test_late_mismatch_is_reported_without_a_sync_in_the_forward():
    cfg = CONFIGS["mini_cheetah-k4-contact"]
    b = make_batch(cfg, 64, seed=1).to("cuda:0")
    nm = build_model(cfg, layers=2, seed=3).to("cuda:0")
    assert nm.validate_edges == "always"
    with torch.no_grad():
        nm(b.x_dict, b.edge_index_dict)                  # first batch of this (template, B): checked synchronously
        n0 = N.launch_count()
        nm(b.x_dict, b.edge_index_dict)
        per_forward = N.launch_count() - n0
        bad = {k: v.clone() for k, v in b.edge_index_dict.items()}
        bad[nm.edge_types[0]][0, 5] = 3
        nm(b.x_dict, bad)                                # deferred: this call itself does not synchronise
        with pytest.raises(ValueError, match="EARLIER batch"):
            nm.assert_edges_valid()
        nm.validate_edges = "never"
        n0 = N.launch_count()
        nm(b.x_dict, b.edge_index_dict)
        assert per_forward - (N.launch_count() - n0) == 1   # the check is exactly one native launch


def test_cached_validation_checks_a_tensor_once():
    cfg = CONFIGS["mini_cheetah-k4-contact"]
    b = make_batch(cfg, 64, seed=1).to("cuda:0")
    nm = build_model(cfg, layers=2, seed=3).to("cuda:0")
    nm.validate_edges = "cached"
    ei = b.edge_index_dict
    with torch.no_grad():
        nm(b.x_dict, ei)
        n0 = N.launch_count()
        nm(b.x_dict, ei)
        a = N.launch_count() - n0
        fresh = {k: v.clone() for k, v in ei.items()}    # new tensor objects: validated again
        n0 = N.launch_count()
        nm(b.x_dict, fresh)
        assert N.launch_count() - n0 == a + 1


@pytest.mark.parametrize("name,B", [("mini_cheetah-k4-contact", 2400), ("mini_cheetah-c2-contact", 1100), ("mini_cheetah-k4-contact", 96),
                                    ("mini_cheetah-k4-contact", 70001)])
def test_encoder_kernels_are_bit_identical(name, B):
    """Encoder forward: persistent TMA-fed kernel (one / two row tiles per item; 2400 and 1100 graphs end on a one-tile item and give
    some CTAs several items; 70001 graphs give every CTA many items and take the CTA-pair stack kernel) against the one-item-per-CTA
    kernels, and the encoder weight gradient with TMA-fed against register-staged feature rows: same bits in the predictions, the loss
    and EVERY gradient (all variants accumulate the same products in the same order; hgnn_k4.py:L159-160 and its autograd)."""
    from test_gpu_large_batch import device_batch
    cfg = CONFIGS[name]
    b = device_batch(cfg, B, seed=B + 7) if B > 16384 else make_batch(cfg, B, seed=B + 7).to("cuda:0")
    nm = build_model(cfg, layers=8, seed=5).set_mode("tc").to("cuda:0")
    ref = None
    try:
        for enc, tpi, dw in ((2, 0, 0), (1, 0, 0), (0, 1, 0), (0, 2, 0), (0, 0, 1)):
            N.set_option("encoder", enc); N.set_option("encoder_tpi", tpi); N.set_option("encoder_dw_tma", dw)
            out, loss, g = _step(nm, cfg, b)
            if ref is None:
                ref = (out.clone(), loss, {k: v.clone() for k, v in g.items()})
                continue
            assert torch.equal(out, ref[0]) and loss == ref[1], (enc, tpi, dw)
            for k in g:
                assert torch.equal(g[k], ref[2][k]), (k, enc, tpi, dw)
    finally:
        N.set_option("encoder", -1); N.set_option("encoder_tpi", 0); N.set_option("encoder_dw_tma", -1)
