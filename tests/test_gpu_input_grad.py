"""GPU checks of the input gradient d loss / d x_dict (mshgnn_input_grad and the input-only backward).

The oracle's x.grad (fp64 autograd through the reference ops) is the checker.  Like the parameter gradients, the input gradient
is discontinuous in the forward numerics (ReLU), so the strict bound (1e-4 norm-wise per node type) holds under the ReLU sign
pattern the native forward took; the plain (unforced) error is printed next to it.
"""
import pytest
import torch

from helpers import (TOL_FP32, forced_native_pattern, native_relu_pattern, oracle_grads_with_forced, oracle_model, oracle_run,
                     rel_err)
from ms_hgnn import _native as N
from ms_hgnn.synthetic import CONFIGS, build_model, make_batch

pytestmark = pytest.mark.gpu
PLAIN_BOUND = 1e-1

# the CASES sizes of test_gpu_parity.py (partial last row tiles), 2400 K4 graphs (19 row tiles) and the narrow widths
# (A1 joint 450 / foot 1, Solo 6 / 2, MI 3: rows that are not a multiple of 16 bytes take the plain-store path)
CASES = [
    ("mini_cheetah-k4-contact", 64, 8), ("mini_cheetah-k4-contact", 200, 8), ("mini_cheetah-k4-contact", 1, 3),
    ("mini_cheetah-k4-contact", 2400, 8), ("mini_cheetah-c2-contact", 96, 8), ("a1-c2-grf", 64, 8), ("k4-grf-regression", 130, 8),
    ("solo12-k4-com", 257, 8), ("solo-c2-com", 33, 4), ("mi-grf", 20, 8), ("mi-contact", 30, 8), ("mi-com", 77, 2),
]


def native_step(cfg, nm, batch, x_dtype=torch.float32, which=None, freeze=False):
    """forward + native loss + backward with x.requires_grad on the types in `which` (all by default); returns out, {type: x.grad}."""
    dev = torch.device("cuda:0")
    b = batch.to(dev)
    nm.requires_grad_(not freeze)
    x = {k: v.to(x_dtype).detach().requires_grad_(which is None or k in which) for k, v in b.x_dict.items()}
    nm.zero_grad(set_to_none=True)
    out = nm(x, b.edge_index_dict)
    eng = nm._last_engine
    C = eng.spec["out_channels"]
    _, dout = eng.loss(out.detach().float().reshape(-1, C).contiguous(), b.y.float() if x_dtype == torch.float16 else b.y.to(x_dtype),
                       N.LOSS_CE2 if cfg.loss == "ce" else N.LOSS_MSE)
    out.backward(dout.view_as(out).to(out.dtype))
    return out.detach(), {k: v.grad for k, v in x.items()}


def models(cfg, layers):
    om = oracle_model(cfg, layers=layers, seed=1)
    nm = build_model(cfg, layers=layers, seed=2)
    nm.load_state_dict({k: v.float() for k, v in om.state_dict().items()})
    return om, nm


def check_input_grads(cfg, B, layers, mode, x_dtype=torch.float32, freeze=False):
    batch = make_batch(cfg, B, seed=B + 11)
    om, nm = models(cfg, layers)
    nm = nm.set_mode(mode).to("cuda:0")
    out_n, dx_n = native_step(cfg, nm, batch, x_dtype, freeze=freeze)
    out_o, _, _, dx_plain = oracle_run(cfg, om, batch, x_grad=True)
    e_out = rel_err(out_n, out_o)
    assert e_out <= TOL_FP32
    forced, flips, ratio, error = forced_native_pattern(om, batch, native_relu_pattern(nm, B), e_out)
    assert error is None and ratio <= 1.0, (error, "native ReLU pattern differs from the oracle at a non-ambiguous pre-activation", ratio)
    _, dx_o = oracle_grads_with_forced(cfg, om, batch, forced, x_grad=True)
    worst, plain = 0.0, 0.0
    for k in dx_o:
        assert dx_n[k] is not None and dx_n[k].dtype == x_dtype and dx_n[k].shape == batch.x_dict[k].shape, k
        if dx_o[k].norm() == 0:
            assert dx_n[k].abs().max().item() == 0.0, k
            continue
        worst = max(worst, rel_err(dx_n[k], dx_o[k]))
        plain = max(plain, rel_err(dx_n[k], dx_plain[k]))
    print(f"input grad[{cfg.name} B={B} L={layers} {mode} {x_dtype}]: worst (native ReLU pattern) {worst:.2e}  plain {plain:.2e}  flips {flips}")
    assert worst <= TOL_FP32
    assert plain <= (PLAIN_BOUND if flips else TOL_FP32)
    return nm


@pytest.mark.parametrize("mode", ["fp32", "tc"])
@pytest.mark.parametrize("name,B,layers", CASES)
def test_input_grad_matches_oracle(name, B, layers, mode):
    check_input_grads(CONFIGS[name], B, layers, mode)


def test_dead_slots_are_exact_zeros_and_every_element_is_written():
    cfg = CONFIGS["mini_cheetah-k4-contact"]
    B = 300
    batch = make_batch(cfg, B, seed=5)
    nm = build_model(cfg, layers=1, seed=3).set_mode("tc").to("cuda:0")
    _, dx = native_step(cfg, nm, batch)
    eng = nm._last_engine
    need0 = eng.plan.describe()["need"][0]
    spec = eng.spec
    assert 0 in need0, "the L = 1 K4 model is expected to have dead encoder slots"
    first = 0
    for t, name in enumerate(spec["node_types"]):
        n = spec["nodes_per_graph"][t]
        rows = dx[name].view(B, n, -1)
        for j in range(n):
            if not need0[first + j]:
                assert torch.equal(rows[:, j], torch.zeros_like(rows[:, j])), (name, j)
            else:
                assert rows[:, j].abs().max().item() > 0, (name, j)
        first += n
    # raw binding on NaN-filled buffers, both modes: no element is left unwritten, and the result is the autograd one
    for mode in (N.MODE_TC, N.MODE_FP32):
        nm.set_mode("tc" if mode == N.MODE_TC else "fp32")
        _, dx = native_step(cfg, nm, batch)
        eng = nm._last_engine
        bufs = [torch.full_like(dx[k], float("nan")) for k in spec["node_types"]]
        ws = eng._ws
        eng.plan.input_grad(B, nm._flat.data_ptr(), [t.data_ptr() for t in bufs], ws.data_ptr(), ws.numel(), mode,
                            torch.cuda.current_stream().cuda_stream)
        for k, t in zip(spec["node_types"], bufs):
            assert not torch.isnan(t).any(), (mode, k)
            assert torch.equal(t, dx[k]), (mode, k)


def test_float64_and_float16_features():
    cfg = CONFIGS["mini_cheetah-k4-contact"]
    check_input_grads(cfg, 64, 8, "tc", x_dtype=torch.float64)
    check_input_grads(cfg, 64, 8, "fp32", x_dtype=torch.float64)
    batch = make_batch(cfg, 200, seed=9)
    rounded = type(batch)({k: v.half().float() for k, v in batch.x_dict.items()}, batch.edge_index_dict, batch.y, batch.batch_size)
    for mode in ("tc", "fp32"):
        nm = build_model(cfg, layers=8, seed=4).set_mode(mode).to("cuda:0")
        _, dx16 = native_step(cfg, nm, batch, torch.float16)
        _, dx32 = native_step(cfg, nm, rounded, torch.float32)
        for k in dx16:
            assert dx16[k].dtype == torch.float16
            assert torch.equal(dx16[k], dx32[k].half()), (mode, k)


@pytest.mark.parametrize("mode", ["fp32", "tc"])
def test_frozen_model_and_partial_requests(mode):
    cfg = CONFIGS["mini_cheetah-k4-contact"]
    B = 200
    batch = make_batch(cfg, B, seed=B + 11)
    nm = check_input_grads(cfg, B, 8, mode, freeze=True)          # all parameters frozen: still meets the oracle bound
    assert all(p.grad is None for p in nm.parameters())
    # the input-only backward issues no weight-gradient work
    N.profile_enable(True)
    try:
        N.profile_read()
        native_step(cfg, nm, batch, freeze=True)
        prof = N.profile_read()
    finally:
        N.profile_enable(False)
    assert "dx_encoder" in prof
    assert not {"dw_layers", "dw_encoder", "reduce_partials"} & set(prof), prof
    # trainable model: same x gradient, and it changes no parameter gradient bit
    _, dx_full = native_step(cfg, nm, batch)
    g_x = {n: p.grad.clone() for n, p in nm.named_parameters()}
    _, dx_frozen = native_step(cfg, nm, batch, freeze=True)
    for k in dx_full:
        assert torch.equal(dx_full[k], dx_frozen[k]), k
    _, none = native_step(cfg, nm, batch, which=())
    assert all(v is None for v in none.values())
    for n, p in nm.named_parameters():
        assert torch.equal(p.grad, g_x[n]), n
    # only one type requested
    _, part = native_step(cfg, nm, batch, which=("joint",))
    assert torch.equal(part["joint"], dx_full["joint"])
    assert part["base"] is None and part["foot"] is None
    # torch.autograd.grad
    b = batch.to("cuda:0")
    x = {k: v.detach().requires_grad_() for k, v in b.x_dict.items()}
    out = nm(x, b.edge_index_dict)
    _, dout = nm._last_engine.loss(out.detach().reshape(-1, 2).contiguous(), b.y, N.LOSS_CE2)
    gx = torch.autograd.grad(out, [x[k] for k in nm.node_types], grad_outputs=dout.view_as(out))
    for k, g in zip(nm.node_types, gx):
        assert torch.equal(g, dx_full[k]), k


@pytest.fixture
def restore_options():
    before = N.get_option("stack"), N.get_option("stack_pair")
    yield
    N.set_option("stack", before[0])
    N.set_option("stack_pair", before[1])


@pytest.mark.parametrize("name,B", [("mini_cheetah-k4-contact", 1000), ("a1-c2-grf", 300), ("solo-c2-com", 520)])
def test_input_grad_across_stack_kernels_and_steps(name, B, restore_options):
    """One-CTA and CTA-pair stack kernels and repeated steps: identical bits.  The per-layer launches (stack option 0) are held
    to the bound test_gpu_stack.py holds their parameter gradients to; whether they agree bit for bit is printed."""
    cfg = CONFIGS[name]
    batch = make_batch(cfg, B, seed=B + 3)
    nm = build_model(cfg, layers=8, seed=7).set_mode("tc").to("cuda:0")
    res = {}
    for tag, stack, pair in (("one-CTA", 1, 0), ("CTA-pair", 1, 2), ("per-layer", 0, 0), ("one-CTA again", 1, 0)):
        N.set_option("stack", stack)
        N.set_option("stack_pair", pair)
        res[tag] = native_step(cfg, nm, batch)[1]
    ref = res["one-CTA"]
    for tag in ("CTA-pair", "one-CTA again"):
        for k in ref:
            assert torch.equal(res[tag][k], ref[k]), (tag, k)
    worst = max(rel_err(res["per-layer"][k], ref[k]) for k in ref)
    same = all(torch.equal(res["per-layer"][k], ref[k]) for k in ref)
    print(f"input grad [{name} B={B}] per-layer launches against the stack kernel: {'bit for bit' if same else f'worst {worst:.1e}'}")
    assert worst <= TOL_FP32


@pytest.mark.parametrize("mode", ["tc", "fp32"])
def test_full_size_properties_16384_graphs(mode):
    """16384 K4 Mini Cheetah graphs: shard invariance (the full batch's dx x 2 against its two shards', mean loss), K4
    equivariance of dx, and every graph against the fp64 oracle (test_gpu_large_batch.check_training_batch: x.grad and every
    parameter gradient under the native ReLU pattern, and every row tile of 128 graphs on its own)."""
    from ms_hgnn import morphology as M
    from ms_hgnn.synthetic import HeteroBatch
    cfg = CONFIGS["mini_cheetah-k4-contact"]
    B = 16384
    batch = make_batch(cfg, B, seed=77)
    om, nm = models(cfg, 8)
    nm = nm.set_mode(mode).to("cuda:0")
    nm.validate_edges = "cached"
    _, dx = native_step(cfg, nm, batch)
    _, d0 = native_step(cfg, nm, batch.shard(0, 2))
    _, d1 = native_step(cfg, nm, batch.shard(1, 2))
    bit = True
    for k in dx:
        shards = torch.cat((d0[k], d1[k]))
        e = rel_err(2 * dx[k], shards)
        bit = bit and torch.equal(2 * dx[k], shards)
        assert e <= 1e-6, (k, e)
    print(f"input grad shard invariance [{mode}]: {'bit for bit' if bit else 'within 1e-6, not bit for bit'}")
    # equivariance: gs acts on the features as a node permutation + per-column sign, on the labels by perm_ls
    g = M.GROUPS["mini_cheetah-k4"]
    T = 150
    pj, rj = torch.tensor(g["permutation_Q_js"][0]), torch.tensor(g["reflection_Q_js"][0], dtype=torch.float32)
    pf, rf = torch.tensor(g["permutation_Q_fs"][0]), torch.tensor(g["reflection_Q_fs"][0], dtype=torch.float32)
    pb = torch.tensor(g["permutation_Q_bs"][0])
    rbl, rba = torch.tensor(g["reflection_Q_bs_lin"][0], dtype=torch.float32), torch.tensor(g["reflection_Q_bs_ang"][0], dtype=torch.float32)

    def act(x):
        x = {k: v.float().cpu() for k, v in x.items()}
        xj = x["joint"].view(B, 12, 2, T)[:, pj] * rj.view(1, 12, 1, 1)
        xf = x["foot"].view(B, 4, 2, 3, T).permute(0, 2, 4, 1, 3).reshape(B, 2, T, 12)[..., pf] * rf
        xf = xf.view(B, 2, T, 4, 3).permute(0, 3, 1, 4, 2).reshape(B * 4, 6 * T)
        xb = x["base"].view(B, 4, 2, 3, T).permute(0, 2, 4, 1, 3).reshape(B, 2, T, 12)[..., pb]
        xb = torch.stack((xb[:, 0] * rbl, xb[:, 1] * rba), dim=1).view(B, 2, T, 4, 3).permute(0, 3, 1, 4, 2).reshape(B * 4, 6 * T)
        return {"base": xb.contiguous(), "joint": xj.reshape(B * 12, 2 * T).contiguous(), "foot": xf.contiguous()}

    y_g = batch.y.view(B, 4)[:, g["permutation_Q_ls"][0]].reshape(batch.y.shape).contiguous()
    gb = HeteroBatch(act(batch.x_dict), batch.edge_index_dict, y_g, B)
    _, dx_g = native_step(cfg, nm, gb)
    want = act(dx)
    for k in dx_g:
        e = rel_err(dx_g[k], want[k])
        assert e <= TOL_FP32, (k, e)
    # every graph against the fp64 oracle
    from test_gpu_large_batch import check_training_batch
    check_training_batch(cfg, nm, om, batch.to("cuda:0"), mode, "input grad full-size properties")
