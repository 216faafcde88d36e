"""Model batches of different hidden widths and learning rates on the GPU: every model of a mixed batch must get bit for bit
what the single-model calls on a plan of its own width give it - predictions, loss, gradients, and after training steps
with its own learning rate, parameters and optimizer state."""
import os

import numpy as np
import pytest
import torch

from ms_hgnn import _native as N
from ms_hgnn import morphology as M_
from ms_hgnn.engine import Engine
from ms_hgnn.model_batch import ModelBatch, ModelBatchTrainer
from ms_hgnn.synthetic import CONFIGS, build_model, make_batch
from ms_hgnn.train import FusedTrainer
from test_gpu_model_batch import CFGS, _kind
from test_gpu_train_models import _same_runs

pytestmark = pytest.mark.gpu

DEV = torch.device("cuda:0") if torch.cuda.is_available() else None
WIDTHS = [128, 64, 37, 10, 1]


def setup(name, widths, B, layers=4, mode="tc"):
    """One seeded model per width, one batch each; every model's own engine, and the engine of the batch's plan."""
    cfg = CONFIGS[name]
    models = [build_model(cfg, hidden=h, layers=layers, seed=10 + m).to(DEV).set_mode(mode) for m, h in enumerate(widths)]
    batches = [make_batch(cfg, B, seed=20 + m).to(DEV) for m in range(len(widths))]
    engs = []
    for nm, b in zip(models, batches):
        eng, _ = nm._engine_for(b.x_dict, b.edge_index_dict)
        nm._ensure_flat(DEV)
        engs.append(eng)
    mixed = Engine(dict(engs[0].spec, widths=list(widths)), engs[0].mode)
    return cfg, models, batches, engs, mixed


def singles(cfg, models, batches, engs, train=True):
    res = []
    for nm, b, eng in zip(models, batches, engs):
        xs = [b.x_dict[t] for t in nm.node_types]
        out = eng.forward(xs, nm._flat, train=train)
        if not train:
            res.append((out.clone(), None, None))
            continue
        loss, dout = eng.loss(out, b.y, _kind(cfg))
        g = eng.backward(dout, nm._flat)
        res.append((out.clone(), loss.clone(), g.clone()))
    return res


def _inputs(models, batches):
    nt = models[0].node_types
    xs = [torch.cat([b.x_dict[t] for b in batches]) for t in nt]
    y = torch.cat([b.y.reshape(-1) for b in batches])
    return xs, y


def batched(cfg, models, batches, eng, train=True):
    xs, y = _inputs(models, batches)
    flat = torch.cat([nm._flat for nm in models])
    out = eng.forward(xs, flat, train=train, n_models=len(models))
    if not train:
        return out, None, None
    loss, dout = eng.loss(out, y, _kind(cfg), n_models=len(models))
    return out, loss, eng.backward(dout, flat)


def check(cfg, models, batches, engs, mixed, train=True, tag=""):
    ref = singles(cfg, models, batches, engs, train)
    out, loss, g = batched(cfg, models, batches, mixed, train)
    torch.cuda.synchronize()
    rows = out.shape[0] // len(models)
    offs = mixed.model_offsets()
    for m, (o, l, gg) in enumerate(ref):
        assert torch.equal(out[m * rows:(m + 1) * rows], o), f"{tag} model {m}: predictions differ"
        if train:
            assert torch.equal(loss[m:m + 1], l), f"{tag} model {m}: loss {loss[m].item()} != {l.item()}"
            gm = g[offs[m]:offs[m + 1]]
            assert torch.equal(gm, gg), f"{tag} model {m}: gradients differ in {(gm != gg).sum().item()} elements"


@pytest.mark.parametrize("B", [1, 100, 2048])
@pytest.mark.parametrize("name", CFGS)
def test_mixed_widths_are_bit_identical_to_single_models(name, B):
    """Five models at 2048 graphs (10 240 in all) also cross the CTA-pair stack kernel's 6144-graph threshold."""
    check(*setup(name, WIDTHS, B), tag=f"{name} B={B}")


@pytest.mark.parametrize("name", CFGS)
def test_mixed_widths_inference(name):
    check(*setup(name, WIDTHS, 100), train=False, tag=f"{name} inference")


@pytest.mark.parametrize("width", [10, 128])
@pytest.mark.parametrize("name", ["mini_cheetah-k4-contact", "solo12-k4-com"])
def test_equal_widths_give_the_uniform_batch(name, width):
    """A plan of three equal widths gives what a plain plan's model batch of the same three models gives."""
    cfg, models, batches, engs, mixed = setup(name, [width] * 3, 129)
    xs, y = _inputs(models, batches)
    flat = torch.stack([nm._flat for nm in models])
    res = []
    for eng, f in ((engs[0], flat), (mixed, flat.reshape(-1))):
        out = eng.forward(xs, f, train=True, n_models=3)
        loss, dout = eng.loss(out, y, _kind(cfg), n_models=3)
        res.append((out.clone(), loss.clone(), eng.backward(dout, f).reshape(-1).clone()))
    torch.cuda.synchronize()
    for a, b in zip(*res):
        assert torch.equal(a, b)


@pytest.mark.parametrize("optimizer", ["adam", "sgd"])
def test_trainer_with_per_model_learning_rates(optimizer):
    name, widths, lrs = "mini_cheetah-k4-contact", [16, 128, 37], [1e-3, 1e-4, 3e-3]
    cfg = CONFIGS[name]
    models = [build_model(cfg, hidden=h, layers=4, seed=10 + m).to(DEV).set_mode("tc") for m, h in enumerate(widths)]
    twins = [build_model(cfg, hidden=h, layers=4, seed=10 + m).to(DEV).set_mode("tc") for m, h in enumerate(widths)]
    batches = [make_batch(cfg, 129, seed=20 + m).to(DEV) for m in range(3)]
    tr = ModelBatchTrainer(ModelBatch(models, mixed_hidden=True), optimizer=optimizer, lr=lrs)
    fts = [FusedTrainer(t, optimizer=optimizer, lr=l) for t, l in zip(twins, lrs)]
    for step in range(5):
        active = [True, step < 3, True]                 # model 1 stops after three steps: its state must freeze
        losses = tr.train_step(batches, active=active)
        for m in range(3):
            if active[m]:
                lm = fts[m].train_step(batches[m])
                assert torch.equal(losses[m:m + 1], lm), f"step {step} model {m}: loss"
    torch.cuda.synchronize()
    for m in range(3):
        for (n, p), (n2, p2) in zip(models[m].named_parameters(), twins[m].named_parameters()):
            assert n == n2 and torch.equal(p, p2), f"model {m}: {n}"
        if optimizer == "adam":
            assert torch.equal(tr.exp_avg[m], fts[m].exp_avg) and torch.equal(tr.exp_avg_sq[m], fts[m].exp_avg_sq), f"model {m}: moments"
        assert tr.step_count[m] == fts[m].step_count
    assert models[2]._flat.data_ptr() == tr.mb.flat[2].data_ptr()
    b = batches[2]
    preds = tr.infer(batches)
    with torch.no_grad():
        assert torch.equal(preds[2], models[2](b.x_dict, b.edge_index_dict))


def test_adam_models_equals_grouped_launches():
    """One adam_step_models launch with one lr equals today's launches per run of models with one step count."""
    g = torch.Generator(device=DEV).manual_seed(3)
    sizes = [1000, 4097, 3, 70001, 256]
    offs = [0]
    for s in sizes:
        offs.append(offs[-1] + s)
    n = offs[-1]
    p0, grads = torch.randn(n, device=DEV, generator=g), torch.randn(n, device=DEV, generator=g)
    m0, v0 = torch.randn(n, device=DEV, generator=g) * 0.1, torch.rand(n, device=DEV, generator=g) * 0.1
    steps = [3, 3, 0, 7, 1]
    stream = torch.cuda.current_stream(DEV).cuda_stream
    for wd in (0.0, 0.01):
        a = [t.clone() for t in (p0, m0, v0)]
        b = [t.clone() for t in (p0, m0, v0)]
        N.adam_step_models(a[0].data_ptr(), grads.data_ptr(), a[1].data_ptr(), a[2].data_ptr(), offs, steps, [1e-3] * 5, 0.9, 0.999, 1e-8,
                           wd, stream)
        for i, st in enumerate(steps):
            if st:
                o, k = offs[i], sizes[i]
                N.adam_step(b[0][o:].data_ptr(), grads[o:].data_ptr(), b[1][o:].data_ptr(), b[2][o:].data_ptr(), k, st, 1e-3, 0.9, 0.999,
                            1e-8, wd, stream)
        torch.cuda.synchronize()
        for x, y in zip(a, b):
            assert torch.equal(x, y)
        assert torch.equal(a[0][offs[2]:offs[3]], p0[offs[2]:offs[3]])      # step 0: untouched
    a, b = p0.clone(), p0.clone()
    N.sgd_step_models(a.data_ptr(), grads.data_ptr(), offs, [0.1, 0.2, 0.3, 0.4, 0.5], [True, False, True, True, True], stream)
    for i, l in enumerate([0.1, 0.2, 0.3, 0.4, 0.5]):
        if i != 1:
            N.sgd_step(b[offs[i]:].data_ptr(), grads[offs[i]:].data_ptr(), sizes[i], l, stream)
    torch.cuda.synchronize()
    assert torch.equal(a, b)


def test_mixed_batch_in_a_cuda_graph():
    """Forward + loss + backward of a mixed batch captured once, replayed on new inputs copied into the captured buffers."""
    cfg, models, batches, engs, mixed = setup("a1-c2-grf", WIDTHS, 100)
    xs, y = _inputs(models, batches)
    flat = torch.cat([nm._flat for nm in models])
    grads = torch.empty_like(flat)
    kind = _kind(cfg)

    def step():
        out = mixed.forward(xs, flat, train=True, n_models=len(models))
        loss, dout = mixed.loss(out, y, kind, n_models=len(models))
        mixed.backward(dout, flat, grads=grads)
        return out, loss

    step()                                        # eager call first: uploads the plan tables, sizes the workspace
    torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        g_out, g_loss = step()
    new = [make_batch(cfg, 100, seed=90 + m).to(DEV) for m in range(len(models))]
    nxs, ny = _inputs(models, new)
    for dst, src in zip(xs, nxs):
        dst.copy_(src)
    y.copy_(ny)
    with torch.no_grad():
        flat.mul_(0.5)
    graph.replay()
    torch.cuda.synchronize()
    r_out, r_loss, r_grads = g_out.clone(), g_loss.clone(), grads.clone()
    e_out, e_loss = step()
    torch.cuda.synchronize()
    assert torch.equal(r_out, e_out) and torch.equal(r_loss, e_loss) and torch.equal(r_grads, grads)


KW_SWEEP = dict(seeds=[0, 0, 5], hidden_size=[16, 8, 32], lr=[1e-3, 1e-4, 1e-3])


def _sweep(tmp_path, monkeypatch, tr, va, te, kw):
    from ms_hgnn.lightning_py.gnnLightning import train_model, train_models
    monkeypatch.chdir(tmp_path)
    paths = train_models(tr, va, te, mode="tc", **KW_SWEEP, **kw)
    assert len(paths) == 3 and len(set(paths)) == 3
    for seed, h, lr, p in zip(KW_SWEEP["seeds"], KW_SWEEP["hidden_size"], KW_SWEEP["lr"], paths):
        ref = train_model(tr, va, te, seed=seed, hidden_size=h, lr=lr, mode="tc", **kw)
        _same_runs(p, ref)
        ck = sorted(c for c in os.listdir(p) if c.endswith(".ckpt"))[0]
        assert torch.load(os.path.join(p, ck), weights_only=False)["optimizer_states"][0]["param_groups"][0]["lr"] == lr


def test_train_models_sweep_mini_cheetah_contact(tmp_path, monkeypatch):
    import window_oracle as WO
    from ms_hgnn.lightning_py.gnnLightning import WindowSubset
    from ms_hgnn.windows import DeviceSequence, WindowSpec
    mat = WO.synthetic_mat(800, seed=21, dtype=np.float32)
    mat["contacts"] = (mat["qd"][:, [2, 5, 8, 11]] > 0).astype(np.float32)
    ds = DeviceSequence(mat, WindowSpec("heterogeneous_gnn_k4", 150, True), DEV, torch.float32)
    tr, va, te = WindowSubset(ds, torch.arange(0, 400)), WindowSubset(ds, torch.arange(400, 520)), WindowSubset(ds, torch.arange(520, len(ds)))
    kw = dict(normalize=True, testing_mode=True, disable_logger=True, batch_size=64, num_layers=2, optimizer="adam",
              regression=False, epochs=3, symmetry_mode="MorphSym", group_operator_path=M_.cfg_path("mini_cheetah-k4"))
    _sweep(tmp_path, monkeypatch, tr, va, te, kw)


def test_train_models_sweep_com(tmp_path, monkeypatch):
    import window_oracle as WO
    from ms_hgnn.lightning_py.gnnLightning import WindowSubset
    from ms_hgnn.windows import DeviceSequence, WindowSpec
    from test_com_grf_metrics import _stats_dir
    mat = WO.synthetic_solo_mat(1200, seed=31)
    data = _stats_dir(tmp_path, mat["y_mean"], mat["y_std"])
    ds = DeviceSequence(mat, WindowSpec("heterogeneous_gnn_k4_com", 1, True, dataset="solo12"), DEV, torch.float32)
    tr, va, te = WindowSubset(ds, torch.arange(0, 800)), WindowSubset(ds, torch.arange(800, 1000)), WindowSubset(ds, torch.arange(1000, len(ds)))
    kw = dict(normalize=True, testing_mode=True, disable_logger=True, batch_size=64, num_layers=2, optimizer="adam",
              epochs=3, data_path=data, symmetry_mode="MorphSym", group_operator_path=M_.cfg_path("solo12-k4"))
    _sweep(tmp_path, monkeypatch, tr, va, te, kw)
