"""GPU checks of hidden widths below 128 (MSHGNN_PLAN_PAD_HIDDEN).

A width-H model runs on the 128-wide kernels as the 128-wide model whose weights are its zero-padded copy (its "twin").  That
gives two checkers: the twin, against which everything must agree bit for bit, and the fp64 oracle built at width H, against
which the usual 1e-4 bounds hold (gradients under the ReLU sign pattern the native forward took, as in test_gpu_input_grad.py).
"""
import contextlib
import json
import os
import socket
import subprocess
import sys

import pytest
import torch

import mshgnn_oracle as O
from helpers import TOL_FP32, native_relu_pattern, oracle_loss, oracle_model, rel_err
from ms_hgnn import _native as N
from ms_hgnn import morphology as M
from ms_hgnn.synthetic import CONFIGS, HeteroBatch, build_model, make_batch
from ms_hgnn.train import FusedTrainer
from test_gpu_input_grad import CASES

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture
def restore_options():
    before = N.get_option("stack"), N.get_option("stack_pair")
    yield
    N.set_option("stack", before[0])
    N.set_option("stack_pair", before[1])


def _kind(cfg):
    return N.LOSS_CE2 if cfg.loss == "ce" else N.LOSS_MSE


def padded_state(narrow, wide):
    """The wide model's state dict holding the narrow model's weights in the top-left corner of every tensor, zeros elsewhere."""
    out = {}
    for (name, p), (_, q) in zip(narrow.state_dict().items(), wide.state_dict().items()):
        z = torch.zeros_like(q)
        z[tuple(slice(0, s) for s in p.shape)] = p
        out[name] = z
    return out


def twins(cfg, hidden, layers, mode, seed=3):
    nm = build_model(cfg, hidden=hidden, layers=layers, seed=seed)
    tw = build_model(cfg, hidden=128, layers=layers, seed=seed)
    tw.load_state_dict(padded_state(nm, tw))
    return nm.set_mode(mode).to(DEV), tw.set_mode(mode).to(DEV)


def native_step(cfg, model, batch):
    """forward + native loss + backward with every feature tensor requiring grad: out, loss, {param: grad}, {type: x.grad}."""
    b = batch.to(DEV)
    x = {k: v.detach().requires_grad_() for k, v in b.x_dict.items()}
    model.zero_grad(set_to_none=True)
    out = model(x, b.edge_index_dict)
    eng = model._last_engine
    loss, dout = eng.loss(out.detach().reshape(-1, eng.spec["out_channels"]).contiguous(), b.y, _kind(cfg))
    out.backward(dout.view_as(out))
    return out.detach(), loss.clone(), {n: p.grad for n, p in model.named_parameters()}, {k: v.grad for k, v in x.items()}


def corner(t, shape):
    return t[tuple(slice(0, s) for s in shape)]


def check_twin_step(cfg, nm, tw, batch, tag):
    H = nm.hidden_channels
    out_n, loss_n, g_n, dx_n = native_step(cfg, nm, batch)
    out_t, loss_t, g_t, dx_t = native_step(cfg, tw, batch)
    assert torch.equal(out_n, out_t), tag
    assert torch.equal(loss_n, loss_t), tag
    for name, g in g_n.items():
        gt = g_t[name]
        assert torch.equal(g, corner(gt, g.shape)), (tag, name)
        rest = gt.clone()
        corner(rest, g.shape).zero_()
        assert rest.abs().max().item() == 0.0, (tag, name, "padded gradient entries must be exact zeros")
    for k in dx_n:
        assert torch.equal(dx_n[k], dx_t[k]), (tag, k)
    # the ReLU pattern the narrow model stored: channels >= H never fire
    for key, (bits, live) in native_relu_pattern(nm, batch.batch_size).items():
        assert not bits[live][:, H:].any(), (tag, key)


def check_params_equal(nm, tw, tag):
    wide = dict(tw.named_parameters())
    for name, p in nm.named_parameters():
        assert torch.equal(p.detach(), corner(wide[name].detach(), p.shape)), (tag, name)


TWIN_CASES = [("mini_cheetah-k4-contact", 200), ("mini_cheetah-k4-contact", 6144), ("a1-c2-grf", 96), ("solo12-k4-com", 130),
              ("mi-grf", 64)]


@pytest.mark.parametrize("mode", ["fp32", "tc"])
@pytest.mark.parametrize("hidden", [10, 64, 100])
@pytest.mark.parametrize("name,B", TWIN_CASES)
def test_padded_twin_is_bit_identical(name, B, hidden, mode):
    """Outputs, loss, gradients (against the twin's sub-blocks), x.grad and the ReLU masks; then 5 Adam steps eager and 5
    graphed leave both models with the same weights; tc1x inference agrees too."""
    cfg = CONFIGS[name]
    nm, tw = twins(cfg, hidden, 4, mode)
    batch = make_batch(cfg, B, seed=B + hidden)
    check_twin_step(cfg, nm, tw, batch, f"{name} B={B} H={hidden} {mode}")
    b = batch.to(DEV)
    trainers = [FusedTrainer(m, optimizer="adam", lr=1e-3) for m in (nm, tw)]
    for _ in range(5):
        for tr in trainers:
            tr.train_step(b)
    check_params_equal(nm, tw, "eager adam")
    for _ in range(5):
        for tr in trainers:
            tr.train_step_graphed(b)
    torch.cuda.synchronize()
    check_params_equal(nm, tw, "graphed adam")
    with torch.no_grad():
        outs = [m.set_mode("tc1x")(b.x_dict, b.edge_index_dict) for m in (nm, tw)]
    assert torch.equal(outs[0], outs[1])


def test_padded_twin_with_per_layer_launches(restore_options):
    N.set_option("stack", 0)
    cfg = CONFIGS["mini_cheetah-k4-contact"]
    nm, tw = twins(cfg, 10, 8, "tc")
    check_twin_step(cfg, nm, tw, make_batch(cfg, 200, seed=4), "stack 0")


# ---------------------------------------------------------------------------------------------------------------------------
# the fp64 oracle at the model's own width
# ---------------------------------------------------------------------------------------------------------------------------
def oracle_all(cfg, om, batch, forced=None):
    """fp64 forward / loss / backward, optionally under a forced ReLU pattern: out, loss, {param: grad}, {type: x.grad}."""
    leaves = {k: v.double().clone().requires_grad_() for k, v in batch.x_dict.items()}
    om.zero_grad()
    with (O.ReluTap(forced=forced) if forced is not None else contextlib.nullcontext()):
        out = om(dict(leaves), batch.edge_index_dict)
        loss = oracle_loss(cfg, out, batch.y.double(), batch.batch_size)
        loss.backward()
    grads = {n: (p.grad.clone() if p.grad is not None else torch.zeros_like(p)) for n, p in om.named_parameters()}
    dx = {k: (v.grad if v.grad is not None else torch.zeros_like(v)) for k, v in leaves.items()}
    return out.detach(), loss.detach(), grads, dx


def native_pattern_for_oracle(om, batch, nm, fwd_err):
    """The first H bits of the native ReLU masks where they differ from the oracle's own signs (only at numerically ambiguous
    pre-activations), in the form O.ReluTap(forced=...) takes."""
    H = nm.hidden_channels
    pattern = native_relu_pattern(nm, batch.batch_size)
    with torch.no_grad(), O.ReluTap(record=True) as tap:
        om({k: v.double() for k, v in batch.x_dict.items()}, batch.edge_index_dict)
    forced, flips = {}, 0
    for i, (pre, tag) in enumerate(zip(tap.pre, tap.tags)):
        bits, live = pattern[tag]
        bits = bits[:, :H]
        v = pre.detach()
        assert tuple(v.shape) == tuple(bits.shape), tag
        diff = ((v > 0) != bits) & live[:, None]
        if diff.any():
            thr = 16.0 * max(fwd_err, 1e-7) * v.pow(2).mean().sqrt().item()
            assert v.abs()[diff].max().item() <= thr, f"native ReLU pattern differs from the oracle at a non-ambiguous pre-activation ({tag})"
            idx = torch.nonzero(diff.reshape(-1)).reshape(-1)
            forced[i] = (idx, bits.reshape(-1)[idx])
            flips += int(idx.numel())
    return forced, flips


@pytest.mark.parametrize("mode", ["fp32", "tc"])
@pytest.mark.parametrize("hidden", [10, 64])
@pytest.mark.parametrize("name,B,layers", CASES)
def test_oracle_parity_at_the_model_width(name, B, layers, hidden, mode):
    cfg = CONFIGS[name]
    om = oracle_model(cfg, hidden=hidden, layers=layers, seed=1)
    nm = build_model(cfg, hidden=hidden, layers=layers, seed=2)
    nm.load_state_dict({k: v.float() for k, v in om.state_dict().items()}, strict=True)
    nm = nm.set_mode(mode).to(DEV)
    batch = make_batch(cfg, B, seed=B + 13)
    out_n, loss_n, g_n, dx_n = native_step(cfg, nm, batch)
    out_o, loss_o, _, _ = oracle_all(cfg, om, batch)
    e_out = rel_err(out_n, out_o)
    assert e_out <= TOL_FP32 and rel_err(loss_n, loss_o.reshape(1)) <= TOL_FP32
    forced, flips = native_pattern_for_oracle(om, batch, nm, e_out)
    _, _, g_o, dx_o = oracle_all(cfg, om, batch, forced)
    worst = 0.0
    for n, g in g_o.items():
        if g.norm() == 0:
            assert g_n[n].abs().max().item() == 0.0, n
            continue
        worst = max(worst, rel_err(g_n[n], g))
    for k, g in dx_o.items():
        if g.norm() == 0:
            assert dx_n[k].abs().max().item() == 0.0, k
            continue
        worst = max(worst, rel_err(dx_n[k], g))
    print(f"H={hidden} [{name} B={B} L={layers} {mode}]: out {e_out:.2e}, worst gradient (native ReLU pattern) {worst:.2e}, flips {flips}")
    assert worst <= TOL_FP32


def test_k4_equivariance_at_width_10():
    """gs acts on the K4 features as a node permutation + per-column sign and on the labels by perm_ls: the loss is invariant
    and d loss / d x transforms like x (the construction of test_gpu_input_grad.py at 16384 graphs)."""
    cfg = CONFIGS["mini_cheetah-k4-contact"]
    B, T = 512, 150
    batch = make_batch(cfg, B, seed=31)
    nm = build_model(cfg, hidden=10, layers=8, seed=5).set_mode("tc").to(DEV)
    g = M.GROUPS["mini_cheetah-k4"]
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

    _, loss, _, dx = native_step(cfg, nm, batch)
    y_g = batch.y.view(B, 4)[:, g["permutation_Q_ls"][0]].reshape(batch.y.shape).contiguous()
    _, loss_g, _, dx_g = native_step(cfg, nm, HeteroBatch(act(batch.x_dict), batch.edge_index_dict, y_g, B))
    assert rel_err(loss_g, loss) <= TOL_FP32
    want = act(dx)
    for k in dx_g:
        e = rel_err(dx_g[k], want[k])
        assert e <= TOL_FP32, (k, e)


@pytest.mark.parametrize("mode", ["tc", "fp32"])
def test_staged_backward_layers_are_final_at_the_event(mode):
    """Everything from encoder_param_end() on is final (compacted into the caller's layout) when layers_ready is recorded."""
    cfg = CONFIGS["mini_cheetah-k4-contact"]
    B = 2048
    nm = build_model(cfg, hidden=10, layers=8, seed=6).set_mode(mode).to(DEV)
    b = make_batch(cfg, B, seed=8).to(DEV)
    xs = [b.x_dict[t] for t in nm.node_types]
    nm(b.x_dict, b.edge_index_dict)                                   # builds the engine and the flat buffer
    eng = nm._last_engine
    end = eng.encoder_param_end()
    out = eng.forward(xs, nm._flat, train=True)
    _, dout = eng.loss(out, b.y, N.LOSS_CE2)
    grads = torch.full((eng.n_params,), float("nan"), device=DEV)
    ev, side = torch.cuda.Event(), torch.cuda.Stream()
    eng.backward(dout, nm._flat, grads, layers_ready=ev)
    with torch.cuda.stream(side):
        side.wait_event(ev)
        early = grads[end:].clone()
    torch.cuda.synchronize()
    assert not torch.isnan(grads).any()
    assert torch.equal(early, grads[end:])
    plain = eng.backward(dout, nm._flat)
    assert torch.equal(plain, grads)


def test_train_model_at_width_10_and_oracle_checkpoint(tmp_path, monkeypatch):
    import numpy as np
    import window_oracle as WO
    from ms_hgnn import GRF_HGNN_K4
    from ms_hgnn.lightning_py.gnnLightning import WindowSubset, evaluate_model, train_model
    from ms_hgnn.windows import DeviceSequence, WindowSpec
    monkeypatch.chdir(tmp_path)
    mat = WO.synthetic_mat(900, seed=23, dtype=np.float32)
    mat["contacts"] = (mat["qd"][:, [2, 5, 8, 11]] > 0).astype(np.float32)
    ds = DeviceSequence(mat, WindowSpec("heterogeneous_gnn_k4", 150, True), DEV, torch.float32)
    n = len(ds)
    tr, va, te = WindowSubset(ds, torch.arange(0, 500)), WindowSubset(ds, torch.arange(500, 650)), WindowSubset(ds, torch.arange(650, n))
    group = M.cfg_path("mini_cheetah-k4")
    path = train_model(tr, va, te, normalize=True, disable_logger=True, batch_size=100, num_layers=2, optimizer="adam", lr=1e-3,
                       epochs=3, hidden_size=10, regression=False, seed=3, symmetry_mode="MorphSym", group_operator_path=group)
    rows = [json.loads(l) for l in open(os.path.join(path, "metrics.jsonl"))]
    val = dict(enumerate(r for r in rows if "val_CE_loss" in r))          # one validation row per epoch, in order
    best = min(val, key=lambda e: val[e]["val_CE_loss"])
    ckpt = os.path.join(path, next(c for c in os.listdir(path) if c.startswith(f"epoch={best}-")))
    sd = torch.load(ckpt, weights_only=False)["state_dict"]
    assert tuple(sd["model.encoder.lins.base.weight"].shape) == (10, 900)
    assert tuple(sd["model.decoder.weight"].shape) == (2, 10)
    res = evaluate_model(ckpt, va, symmetry_mode="MorphSym", group_operator_path=group, batch_size=64, task_type="classification")
    acc, favg = res[2].item(), res[7].item()
    print(f"best epoch {best}: logged acc {val[best]['val_Accuracy']:.6f} F1 {val[best]['val_F1_Score_Leg_Avg']:.6f}, "
          f"evaluate_model acc {acc:.6f} F1 {favg:.6f}")
    assert abs(acc - val[best]["val_Accuracy"]) <= 1e-6
    assert abs(favg - val[best]["val_F1_Score_Leg_Avg"]) <= 1e-5
    # an oracle state_dict at width 10 loads strictly into the native model
    cfg = CONFIGS["mini_cheetah-k4-contact"]
    om = oracle_model(cfg, hidden=10, layers=2, seed=4)
    nm = GRF_HGNN_K4(hidden_channels=10, num_layers=2, data_metadata=M.TEMPLATES[cfg.template].metadata, regression=False,
                     symmetry_mode="MorphSym", group_operator_path=group)
    nm.load_state_dict({k: v.float() for k, v in om.state_dict().items()}, strict=True)
    assert tuple(nm.encoder.lins["joint"].weight.shape) == (10, 300)


@pytest.mark.skipif(not torch.cuda.is_available() or torch.cuda.device_count() < 2, reason="needs at least 2 GPUs")
def test_nccl_reduced_gradients_at_width_10():
    n = min(torch.cuda.device_count(), 4)
    s = socket.socket(); s.bind(("127.0.0.1", 0)); port = s.getsockname()[1]; s.close()
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={n}", "--master-addr", "127.0.0.1",
                        "--master-port", str(port), os.path.join(ROOT, "tests", "_dp_hidden_worker.py")],
                       capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert r.returncode == 0, (r.stdout[-3000:], r.stderr[-3000:])
    line = next(l for l in r.stdout.splitlines() if l.startswith("DPRESULT "))
    for out in json.loads(line[len("DPRESULT "):]):
        for mode in ("tc", "fp32"):
            assert out[f"{mode}_err"] <= 2e-5, out
            assert out[f"{mode}_overlap_equals_plain"], out
