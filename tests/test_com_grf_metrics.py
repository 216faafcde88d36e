"""Fused COM-momentum and world-frame GRF metrics (mshgnn_step_metrics_ex), the Lightning modules that use them, and the COM
formats of train_model / evaluate_model.

Host tests: the ABI constants and argument validation.  GPU tests: the fused values against the op-by-op metric classes of
customMetrics.py computed in fp64 on the same tensors (1e-10 relative), the modules' fused path against their CPU fallback,
and the train / evaluate loops on a synthetic Solo12 sequence.
"""
import ctypes
import json
import os
import re

import numpy as np
import pytest
import torch

from ms_hgnn import _native as N
from ms_hgnn import morphology as M

ERR_ARG, ERR_CUDA = -1, -2
REL = 1e-10
DEV = "cuda:0"
HEADER = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "include", "mshgnn_b200.h")
# dyadic standardiser stats: mean / std is exact in fp32, so a row of -mean / std un-standardises to exactly zero on both paths
Y_MEAN = [0.5, -1.25, 2.0, 0.75, -0.375, 1.5]
Y_STD = [0.5, 1.25, 0.25, 1.5, 0.75, 3.0]
COM_TYPES = [("heterogeneous_gnn_k4_com", "solo12-k4", 4), ("heterogeneous_gnn_c2_com", "solo-c2", 2), ("heterogeneous_gnn_s4_com", None, 1)]


def _close(a, b, rel=REL):
    a, b = float(a), float(b)
    return abs(a - b) <= rel * abs(b) or a == b


# ---------------------------------------------------------------- host ----------------------------------------------------------

def test_new_metric_kinds_and_slots_are_exported():
    header = open(HEADER).read()
    assert int(re.search(r"#define MSHGNN_METRIC_COM\s+(\d+)", header).group(1)) == N.METRIC_COM == 2
    assert int(re.search(r"#define MSHGNN_METRIC_GRF_WORLD\s+(\d+)", header).group(1)) == N.METRIC_GRF_WORLD == 3
    assert "mshgnn_step_metrics_ex" in N.EXPORTS and hasattr(N.lib(), "mshgnn_step_metrics_ex")
    assert (N.COM_SSE, N.COM_N, N.COM_SSE_LIN, N.COM_SSE_ANG, N.COM_N_HALF, N.COM_COS_LIN, N.COM_COS_ANG, N.COM_ROWS) == tuple(range(8))
    assert (N.COM_MSE, N.COM_RMSE, N.COM_MSE_LIN, N.COM_MSE_ANG, N.COM_COS_SIM_LIN, N.COM_COS_SIM_ANG, N.COM_AVG_COS_SIM) == tuple(range(20, 27))
    assert (N.GRF_SSE, N.GRF_SAE, N.GRF_N, N.GRF_SSE_WORLD, N.GRF_SAE_WORLD, N.GRF_N_WORLD) == tuple(range(6))
    assert (N.GRF_MSE, N.GRF_RMSE, N.GRF_L1, N.GRF_MSE_WORLD, N.GRF_RMSE_WORLD, N.GRF_L1_WORLD) == tuple(range(20, 26))
    # the body-frame states of the world-frame kind are those of the MSE kind (sse, sae, n): one call feeds both metric sets
    assert N.GRF_MSE == 20 and N.GRF_L1 == 22 and N.METRIC_SLOTS >= 27
    # the C struct and the ctypes mirror agree on the field order
    fields = re.search(r"typedef struct \{(.*?)\} mshgnn_metric_args;", header, re.S).group(1)
    assert re.findall(r"\*?\s*(\w+);", fields) == [f[0] for f in N.MetricArgs._fields_]


def _ex(kind, args, n=4, out=1, labels=1, label_dtype=N.F32, batch=1, scratch=1):
    buf = _ex.buf
    p = lambda v: ctypes.addressof(buf) if v else None
    a = ctypes.byref(args) if args is not None else None
    return N.lib().mshgnn_step_metrics_ex(kind, a, n, p(out), p(labels), label_dtype, p(batch), None, p(scratch), None)


_ex.buf = ctypes.create_string_buffer(4096)


def test_step_metrics_ex_rejects_bad_arguments():
    """Every rejected call returns before anything is launched (host pointers stand in for device buffers)."""
    mean = std = ctypes.addressof(_ex.buf)
    com = lambda nb=2, m=mean, s=std: N.MetricArgs(n_base=nb, y_mean=m, y_std=s)
    grf = lambda q=mean, qd=N.F32: N.MetricArgs(quat=q, quat_dtype=qd)
    for kind, args in ((N.METRIC_COM, com()), (N.METRIC_GRF_WORLD, grf())):
        assert _ex(kind, None) == ERR_ARG
        assert _ex(kind, args, n=0) == ERR_ARG
        assert _ex(kind, args, out=0) == ERR_ARG
        assert _ex(kind, args, labels=0) == ERR_ARG
        assert _ex(kind, args, batch=0) == ERR_ARG
        assert _ex(kind, args, scratch=0) == ERR_ARG
        assert _ex(kind, args, label_dtype=3) == ERR_ARG
    for kind in (N.LOSS_MSE, N.LOSS_CE2, 4, -1):
        assert _ex(kind, com()) == ERR_ARG
        assert b"bad metric kind" in N.lib().mshgnn_last_error()
    for nb in (0, 5, -1):
        assert _ex(N.METRIC_COM, com(nb=nb)) == ERR_ARG
        assert b"n_base" in N.lib().mshgnn_last_error()
    assert _ex(N.METRIC_COM, com(m=None)) == ERR_ARG
    assert _ex(N.METRIC_COM, com(s=None)) == ERR_ARG
    assert b"y_mean and y_std" in N.lib().mshgnn_last_error()
    assert _ex(N.METRIC_GRF_WORLD, grf(q=None)) == ERR_ARG
    assert b"quaternions" in N.lib().mshgnn_last_error()
    for qd in (N.I64, N.F16, 7):
        assert _ex(N.METRIC_GRF_WORLD, grf(qd=qd)) == ERR_ARG


def test_step_metrics_ex_without_gpu_fails_with_cuda_error():
    if torch.cuda.is_available():
        pytest.skip("CUDA present")
    args = N.MetricArgs(n_base=1, y_mean=ctypes.addressof(_ex.buf), y_std=ctypes.addressof(_ex.buf))
    assert _ex(N.METRIC_COM, args) == ERR_CUDA


# ---------------------------------------------------------------- fused vs op by op (GPU) ---------------------------------------

BATCHES = (1, 63, 129, 16384)


def _com_inputs(B, n_base, label_dtype, gen):
    w = n_base * 6
    pred = torch.randn(B, w, generator=gen)
    lab = (pred.double() + 0.6 * torch.randn(B, w, generator=gen, dtype=torch.float64)).to(label_dtype)
    mean, std = torch.tensor(Y_MEAN, dtype=torch.float64), torch.tensor(Y_STD, dtype=torch.float64)
    if B > 1:
        pred[1, :6] = (-mean / std).float()                   # un-standardised prediction of base 0 is the zero vector
        pred[2] = 0.0                                          # all-zero standardised prediction row
        lab[3, :6] = (-mean / std).to(label_dtype)             # zero label vector
        pred[3, :6] = (-mean / std).float()                    # ... and zero prediction in the same row
    return pred, lab


def _com_op_by_op(metrics, pred, lab, n_base):
    """COM_Base_Lightning.calculate_losses_step's metric side, op by op in fp64."""
    from ms_hgnn.lightning_py.gnnLightning_com import Standarizer
    st = Standarizer(np.zeros(24), np.ones(24), np.array(Y_MEAN), np.array(Y_STD))
    mse, rmse, lin, ang, cl, ca = metrics
    pd, yd = pred.double(), lab.double()
    mse(pd.flatten(), yd.flatten())
    r = rmse(pd.flatten(), yd.flatten())
    pv, yv = pd.view(-1, n_base, 6), yd.view(-1, n_base, 6)
    ml = lin(pv[:, :, :3].flatten(), yv[:, :, :3].flatten())
    ma = ang(pv[:, :, 3:].flatten(), yv[:, :, 3:].flatten())
    pu, yu = st.unstandarize(pv), st.unstandarize(yv)
    c1 = cl(pu[:, 0, :3], yu[:, 0, :3])
    c2 = ca(pu[:, 0, 3:], yu[:, 0, 3:])
    return [((pd - yd) ** 2).mean(), r, ml, ma, c1, c2, (c1 + c2) / 2]


@pytest.mark.gpu
@pytest.mark.parametrize("label_dtype", [torch.float32, torch.float64])
@pytest.mark.parametrize("n_base", [1, 2, 4])
def test_com_fused_equals_op_by_op(n_base, label_dtype):
    from ms_hgnn.lightning_py import customMetrics as CM
    gen = torch.Generator().manual_seed(10 + n_base)
    fused = CM.FusedStepMetrics()
    metrics = [CM.MeanSquaredError(), CM.MeanSquaredError(squared=False), CM.MeanSquaredError(), CM.MeanSquaredError(),
               CM.CosineSimilarityMetric(), CM.CosineSimilarityMetric()]
    mean, std = torch.tensor(Y_MEAN, dtype=torch.float64, device=DEV), torch.tensor(Y_STD, dtype=torch.float64, device=DEV)
    rows = 0
    for B in BATCHES:
        pred, lab = _com_inputs(B, n_base, label_dtype, gen)
        b = fused.update_com(pred.to(DEV), lab.to(DEV), n_base, mean, std).cpu()
        ref = _com_op_by_op(metrics, pred, lab, n_base)
        for slot, r in zip(range(N.COM_MSE, N.COM_AVG_COS_SIM + 1), ref):
            assert _close(b[slot], r), (B, slot, b[slot].item(), r.item())
        rows += B
        assert b[N.COM_ROWS].item() == B and b[N.COM_N].item() == B * n_base * 6 and b[N.COM_N_HALF].item() == B * n_base * 3
    e = fused.epoch.cpu()
    assert e[N.COM_ROWS].item() == rows
    derived = [e[N.COM_SSE] / e[N.COM_N], torch.sqrt(e[N.COM_SSE] / e[N.COM_N]), e[N.COM_SSE_LIN] / e[N.COM_N_HALF],
               e[N.COM_SSE_ANG] / e[N.COM_N_HALF], e[N.COM_COS_LIN] / e[N.COM_ROWS], e[N.COM_COS_ANG] / e[N.COM_ROWS]]
    for d, m in zip(derived, metrics):
        assert _close(d, m.compute()), (d.item(), m.compute().item())
    # rows whose un-standardised base-0 vectors are zero (cosine eps case) score exactly 0 on both paths
    pred, lab = _com_inputs(8, n_base, label_dtype, gen)
    z = CM.FusedStepMetrics().update_com(pred[[1, 3]].to(DEV), lab[[1, 3]].to(DEV), n_base, mean, std).cpu()
    ref = _com_op_by_op([CM.MeanSquaredError(), CM.MeanSquaredError(squared=False), CM.MeanSquaredError(), CM.MeanSquaredError(),
                         CM.CosineSimilarityMetric(), CM.CosineSimilarityMetric()], pred[[1, 3]], lab[[1, 3]], n_base)
    assert z[N.COM_COS_LIN].item() == z[N.COM_COS_ANG].item() == 0.0 and ref[4].item() == ref[5].item() == 0.0


@pytest.mark.gpu
@pytest.mark.parametrize("n_base", [1, 4])
def test_com_fused_is_deterministic_and_epoch_adds(n_base):
    from ms_hgnn.lightning_py import customMetrics as CM
    gen = torch.Generator().manual_seed(3)
    pred, lab = _com_inputs(16384, n_base, torch.float32, gen)
    pred, lab = pred.to(DEV), lab.to(DEV)
    mean, std = torch.tensor(Y_MEAN, dtype=torch.float64, device=DEV), torch.tensor(Y_STD, dtype=torch.float64, device=DEV)
    f1, f2 = CM.FusedStepMetrics(), CM.FusedStepMetrics()
    a = f1.update_com(pred, lab, n_base, mean, std).clone()
    b = f2.update_com(pred, lab, n_base, mean, std).clone()
    assert torch.equal(a, b)
    assert torch.equal(f1.epoch[:20], a[:20]) and f1.epoch[20:].abs().sum().item() == 0.0
    c = f1.update_com(pred, lab, n_base, mean, std).clone()
    assert torch.equal(c, a) and torch.equal(f1.epoch[:20], a[:20] + a[:20])
    f1.reset()
    assert f1.epoch.abs().sum().item() == 0.0


def _grf_inputs(B, dtype, gen):
    pred = torch.randn(B, 12, generator=gen) * 40.0
    lab = (pred.double() + 5.0 * torch.randn(B, 12, generator=gen, dtype=torch.float64)).to(dtype)
    q = (torch.randn(B, 4, generator=gen, dtype=torch.float64) * 1.7).to(dtype)     # not normalised
    return pred, lab, q


@pytest.mark.gpu
@pytest.mark.parametrize("z_only", [False, True])
@pytest.mark.parametrize("dtype", [torch.float32, torch.float64])
def test_grf_world_fused_equals_op_by_op(dtype, z_only):
    from ms_hgnn.lightning_py import customMetrics as CM
    from ms_hgnn.lightning_py.gnnLightning import HGNN_C2_Lightning_Reg
    helper = HGNN_C2_Lightning_Reg.__new__(HGNN_C2_Lightning_Reg)
    gen = torch.Generator().manual_seed(21 + int(z_only))
    fused = CM.FusedStepMetrics()
    body = [CM.MeanSquaredError(), CM.MeanSquaredError(squared=False), CM.MeanAbsoluteError()]
    world = [CM.MeanSquaredError(), CM.MeanSquaredError(squared=False), CM.MeanAbsoluteError()]
    for B in BATCHES:
        pred, lab, q = _grf_inputs(B, dtype, gen)
        b = fused.update_grf_world(pred.to(DEV), lab.to(DEV), q.to(DEV), z_only).cpu()
        pd, yd = pred.double(), lab.double()
        ref = [m(pd, yd) for m in body]
        yw = HGNN_C2_Lightning_Reg.body_frame_to_world_frame(helper, q.double(), yd)
        pw = HGNN_C2_Lightning_Reg.body_frame_to_world_frame(helper, q.double(), pd)
        if z_only:
            yw, pw = yw[:, [2, 5, 8, 11]], pw[:, [2, 5, 8, 11]]
        ref += [m(pw, yw) for m in world]
        for slot, r in zip(range(N.GRF_MSE, N.GRF_L1_WORLD + 1), ref):
            assert _close(b[slot], r), (B, slot, b[slot].item(), r.item())
        assert b[N.GRF_N].item() == 12 * B and b[N.GRF_N_WORLD].item() == (4 if z_only else 12) * B
    e = fused.epoch.cpu()
    derived = [e[0] / e[2], torch.sqrt(e[0] / e[2]), e[1] / e[2], e[3] / e[5], torch.sqrt(e[3] / e[5]), e[4] / e[5]]
    for d, m in zip(derived, body + world):
        assert _close(d, m.compute()), (d.item(), m.compute().item())
    # same inputs twice: identical bits
    pred, lab, q = (t.to(DEV) for t in _grf_inputs(16384, dtype, gen))
    a = fused.update_grf_world(pred, lab, q, z_only).clone()
    assert torch.equal(a, fused.update_grf_world(pred, lab, q, z_only))


# ---------------------------------------------------------------- Lightning modules (GPU) ----------------------------------------

def _stats_dir(tmp_path, y_mean, y_std):
    d = tmp_path / "data"
    (d / "processed").mkdir(parents=True)
    np.savez(d / "processed" / "rss_stats.npz", x_mean=np.zeros(24), x_std=np.ones(24), y_mean=np.asarray(y_mean), y_std=np.asarray(y_std))
    return d


def _logged(mod):
    return {k: float(v) for k, v in mod.logged.items()}


def _compare_logs(a, b):
    assert a.keys() == b.keys()
    for k in a:
        assert _close(a[k], b[k]), (k, a[k], b[k])


def _run_both(monkeypatch, make, step, epoch, batches, extra=()):
    """Step and epoch logs of ``step`` over ``batches``: fused (CUDA tensors) and CPU fallback (the same tensors in fp64 on the host;
    the gradient-carrying native loss, which needs the device, is replayed from the fused run)."""
    from ms_hgnn.lightning_py import gnnLightning, gnnLightning_com
    gpu, cpu = make(), make()
    logs_gpu, logs_cpu, losses, tensors = [], [], [], []
    gpu.reset_all_metrics() if not hasattr(gpu, "reset_all_metrics_worldframe") else gpu.reset_all_metrics_worldframe()
    with torch.no_grad():
        for i, b in enumerate(batches):
            y, y_pred = gpu.step_helper_function(b.to(DEV))
            ex = [e[i].to(DEV) for e in extra]
            step(gpu, y, y_pred, *ex)
            losses.append(gpu.mse_loss.detach().cpu().double())
            logs_gpu.append(_logged(gpu))
            tensors.append((y.cpu().double(), y_pred.cpu().double(), [e.cpu() for e in ex]))
        epoch(gpu)
        logs_gpu.append(_logged(gpu))
    it = iter(losses)
    stub = lambda model, y_pred, y, kind: next(it)
    monkeypatch.setattr(gnnLightning, "native_loss", stub)
    monkeypatch.setattr(gnnLightning_com, "native_loss", stub)
    cpu.reset_all_metrics() if not hasattr(cpu, "reset_all_metrics_worldframe") else cpu.reset_all_metrics_worldframe()
    with torch.no_grad():
        for y, y_pred, ex in tensors:
            step(cpu, y, y_pred, *ex)
            logs_cpu.append(_logged(cpu))
        epoch(cpu)
        logs_cpu.append(_logged(cpu))
    for a, b in zip(logs_gpu, logs_cpu):
        _compare_logs(a, b)
    return logs_gpu


@pytest.mark.gpu
@pytest.mark.parametrize("model_type,group,n_base", COM_TYPES)
def test_com_module_logs_the_fallback_values(tmp_path, monkeypatch, model_type, group, n_base):
    from ms_hgnn.lightning_py.gnnLightning_com import COM_HGNN_SYM_Lightning
    from ms_hgnn.synthetic import CONFIGS, make_batch
    cfg = CONFIGS[{"heterogeneous_gnn_k4_com": "solo12-k4-com", "heterogeneous_gnn_c2_com": "solo-c2-com",
                   "heterogeneous_gnn_s4_com": "mi-com"}[model_type]]
    tpl = M.TEMPLATES[cfg.template]
    data = _stats_dir(tmp_path, [0.3, -1.1, 0.02, 2.5, -0.7, 0.9], [1.7, 0.4, 2.2, 0.05, 1.3, 0.8])
    batches = [make_batch(cfg, B, seed=s) for s, B in ((1, 63), (2, 129), (3, 1))]
    kw = dict(symmetry_mode="MorphSym", group_operator_path=M.cfg_path(group)) if group else {}
    torch.manual_seed(4)

    def make():
        torch.manual_seed(4)
        return COM_HGNN_SYM_Lightning(16, 2, tpl.metadata, batches[0], "adam", 1e-3, model_type=model_type, data_path=str(data), **kw).to(DEV)

    def step(m, y, y_pred):
        m.calculate_losses_step(y, y_pred)
        m.log_losses("train", on_step=True)

    def epoch(m):
        m.calculate_losses_epoch()
        m.log_losses("val", on_step=False)

    logs = _run_both(monkeypatch, make, step, epoch, batches)
    assert {"train_cos_sim_lin", "train_avg_cos_sim", "val_MSE_loss_ang", "val_RMSE_loss"} <= set(logs[-1])


@pytest.mark.gpu
@pytest.mark.parametrize("z_only", [False, True])
def test_worldframe_module_logs_the_fallback_values(monkeypatch, z_only):
    from ms_hgnn.lightning_py.gnnLightning import HGNN_C2_Lightning_Reg
    from ms_hgnn.synthetic import CONFIGS, make_batch
    cfg = CONFIGS["a1-c2-grf"]
    tpl = M.TEMPLATES[cfg.template]
    Bs = (63, 129, 1)
    batches = [make_batch(cfg, B, seed=s) for s, B in zip((1, 2, 3), Bs)]
    gen = torch.Generator().manual_seed(8)
    quats = [(torch.randn(B, 4, generator=gen) * 0.8) for B in Bs]

    def make():
        torch.manual_seed(5)
        return HGNN_C2_Lightning_Reg(16, 2, tpl.metadata, batches[0], "adam", 1e-3, regression=True, symmetry_mode="MorphSym",
                                     group_operator_path=M.cfg_path("a1-c2"), grf_body_to_world_frame=True, grf_dimension=3).to(DEV)

    def step(m, y, y_pred, q):
        m.calculate_losses_step_worldframe(y, y_pred, q, z_only)
        m.log_losses_worldframe("train", on_step=True)

    def epoch(m):
        m.calculate_losses_epoch_worldframe()
        m.log_losses_worldframe("val", on_step=False)

    logs = _run_both(monkeypatch, make, step, epoch, batches, extra=(quats,))
    assert {"train_L1_loss_WorldFrame", "val_RMSE_loss_WorldFrame", "val_L1_loss"} <= set(logs[-1])


# ---------------------------------------------------------------- train_model / evaluate_model (GPU) ------------------------------

@pytest.mark.gpu
@pytest.mark.parametrize("model_type,group,n_base", COM_TYPES)
def test_train_and_evaluate_com_models(tmp_path, monkeypatch, model_type, group, n_base):
    import window_oracle as WO
    from ms_hgnn.lightning_py.gnnLightning import WindowSubset, evaluate_model, train_model
    from ms_hgnn.lightning_py.gnnLightning_com import COM_HGNN_SYM_Lightning
    from ms_hgnn.windows import DeviceSequence, WindowSpec
    monkeypatch.chdir(tmp_path)
    mat = WO.synthetic_solo_mat(1500, seed=31)
    data = _stats_dir(tmp_path, mat["y_mean"], mat["y_std"])
    ds = DeviceSequence(mat, WindowSpec(model_type, 1, True, dataset="solo12"), DEV, torch.float32)
    n = len(ds)
    tr, va, te = WindowSubset(ds, torch.arange(0, 1000)), WindowSubset(ds, torch.arange(1000, 1250)), WindowSubset(ds, torch.arange(1250, n))
    sym = dict(symmetry_mode="MorphSym", group_operator_path=M.cfg_path(group)) if group else {}
    kw = dict(normalize=True, testing_mode=True, disable_logger=True, batch_size=64, num_layers=2, optimizer="adam", lr=1e-3,
              hidden_size=16, seed=2, data_path=data, **sym)
    path = train_model(tr, va, te, epochs=3, **kw)
    names = sorted(c for c in os.listdir(path) if c.endswith(".ckpt"))
    pat = re.compile(r"^epoch=(\d+)-val_MSE_loss=\d+\.\d{5}\.ckpt$")
    assert len(names) == 3 and all(pat.match(c) for c in names), names
    rows = [json.loads(l) for l in open(os.path.join(path, "metrics.jsonl"))]
    val = [r for r in rows if "epoch" in r]
    assert [r["epoch"] for r in val] == [0, 1, 2] and val[-1]["global_step"] == 30
    assert all(np.isfinite(r[k]) for r in val for k in ("val_MSE_loss", "val_cos_sim_lin", "val_cos_sim_ang", "val_MSE_loss_lin"))
    assert "test_MSE_loss" in rows[-1]
    last = os.path.join(path, [c for c in names if c.startswith("epoch=2-")][0])
    ck = torch.load(last, weights_only=False)
    assert ck["epoch"] == 2 and ck["global_step"] == 30 and ck["hyper_parameters"]["model_type"] == model_type
    # resume
    path2 = train_model(tr, va, te, epochs=5, ckpt_path=last, **kw)
    rows2 = [json.loads(l) for l in open(os.path.join(path2, "metrics.jsonl")) if "epoch" in l]
    assert [r["epoch"] for r in rows2 if "val_MSE_loss" in r] == [3, 4] and rows2[-1]["global_step"] == 50
    # evaluate_model: predictions of a direct forward, metrics recomputed op by op from them
    res = evaluate_model(last, te, data_path=data, batch_size=100, **sym)
    assert len(res) == 8
    pred, lab, mse, rmse, mse_lin, mse_ang, cos_lin, cos_ang = res
    mod = COM_HGNN_SYM_Lightning.load_from_checkpoint(last, strict=False, data_path=data, **sym).to(DEV)
    with torch.no_grad():
        direct = torch.cat([mod.step_helper_function(ds.batch(idx))[1] for idx in torch.split(te.indices, 100)])
    assert torch.equal(pred, direct)
    w = n_base * 6
    assert pred.shape == lab.shape == (len(te), w)
    pd, yd = pred.double().cpu(), lab.double().cpu()
    pv, yv = pd.view(-1, n_base, 6), yd.view(-1, n_base, 6)
    ym, ys = torch.as_tensor(mat["y_mean"], dtype=torch.float64), torch.as_tensor(mat["y_std"], dtype=torch.float64)
    pu, yu = pv * ys + ym, yv * ys + ym
    cs = torch.nn.functional.cosine_similarity
    ref = [((pd - yd) ** 2).mean(), ((pd - yd) ** 2).mean().sqrt(), ((pv - yv)[:, :, :3] ** 2).mean(), ((pv - yv)[:, :, 3:] ** 2).mean(),
           cs(pu[:, 0, :3], yu[:, 0, :3], dim=1).mean(), cs(pu[:, 0, 3:], yu[:, 0, 3:], dim=1).mean()]
    for got, r in zip((mse, rmse, mse_lin, mse_ang, cos_lin, cos_ang), ref):
        assert _close(got.cpu(), r), (got.item(), r.item())
