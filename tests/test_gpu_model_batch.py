"""Model batches on the GPU: M models in one native step must give every model bit for bit what M separate single-model
calls give it - predictions, loss, every gradient row, and the parameters and Adam moments after training steps."""
import pytest
import torch

from ms_hgnn import _native as N
from ms_hgnn.model_batch import ModelBatch, ModelBatchTrainer
from ms_hgnn.synthetic import CONFIGS, build_model, make_batch
from ms_hgnn.train import FusedTrainer

pytestmark = pytest.mark.gpu

DEV = torch.device("cuda:0") if torch.cuda.is_available() else None
CFGS = ["mini_cheetah-k4-contact", "a1-c2-grf", "solo12-k4-com", "mi-com", "mi-grf"]


@pytest.fixture
def restore_options():
    saved = {k: N.get_option(k) for k in ("stack", "stack_pair")}
    yield
    for k, v in saved.items():
        N.set_option(k, v)


def _kind(cfg):
    return N.LOSS_CE2 if cfg.loss == "ce" else N.LOSS_MSE


def setup(name, M, B, hidden=128, layers=4, mode="tc", xdtype=torch.float32):
    """M seeded models of one config, one batch each; the engine of model 0 and every model's flat parameters."""
    cfg = CONFIGS[name]
    models = [build_model(cfg, hidden=hidden, layers=layers, seed=10 + m).to(DEV).set_mode(mode) for m in range(M)]
    batches = []
    for m in range(M):
        b = make_batch(cfg, B, seed=20 + m).to(DEV)
        if xdtype != torch.float32:
            b._x = {k: v.to(xdtype) for k, v in b.x_dict.items()}
        batches.append(b)
    engs = []
    for nm, b in zip(models, batches):
        eng, _ = nm._engine_for(b.x_dict, b.edge_index_dict)
        nm._ensure_flat(DEV)
        engs.append(eng)
    return cfg, models, batches, engs[0]


def singles(cfg, models, batches, eng, train=True):
    res = []
    for nm, b in zip(models, batches):
        xs = [b.x_dict[t] for t in nm.node_types]
        out = eng.forward(xs, nm._flat, train=train)
        if not train:
            res.append((out.clone(), None, None))
            continue
        loss, dout = eng.loss(out, b.y, _kind(cfg))
        g = eng.backward(dout, nm._flat)
        res.append((out.clone(), loss.clone(), g.clone()))
    return res


def batched(cfg, models, batches, eng, train=True):
    M = len(models)
    nt = models[0].node_types
    xs = [torch.cat([b.x_dict[t] for b in batches]) for t in nt]
    flat = torch.stack([nm._flat for nm in models])
    out = eng.forward(xs, flat, train=train, n_models=M)
    if not train:
        return out, None, None
    y = torch.cat([b.y.reshape(-1) for b in batches])
    loss, dout = eng.loss(out, y, _kind(cfg), n_models=M)
    g = eng.backward(dout, flat)
    return out, loss, g.view(M, -1)


def check(cfg, models, batches, eng, train=True, tag=""):
    ref = singles(cfg, models, batches, eng, train)
    out, loss, g = batched(cfg, models, batches, eng, train)
    torch.cuda.synchronize()
    rows = out.shape[0] // len(models)
    for m, (o, l, gg) in enumerate(ref):
        assert torch.equal(out[m * rows:(m + 1) * rows], o), f"{tag} model {m}: predictions differ"
        if train:
            assert torch.equal(loss[m:m + 1], l), f"{tag} model {m}: loss {loss[m].item()} != {l.item()}"
            assert torch.equal(g[m], gg), f"{tag} model {m}: gradients differ in {(g[m] != gg).sum().item()} elements"


@pytest.mark.parametrize("M", [1, 2, 5])
@pytest.mark.parametrize("B", [1, 64, 100, 129, 2048])
@pytest.mark.parametrize("name", CFGS)
def test_model_batch_is_bit_identical(name, B, M):
    check(*setup(name, M, B), tag=f"{name} M={M} B={B}")


@pytest.mark.parametrize("name", CFGS)
def test_model_batch_cta_pair_kernel(name):
    """M = 4 x 2048 graphs cross the CTA-pair threshold (6144 graphs) while each model stays below it."""
    check(*setup(name, 4, 2048, layers=8), tag=f"{name} M=4 B=2048")


@pytest.mark.parametrize("B", [1, 100])
@pytest.mark.parametrize("name", CFGS)
def test_model_batch_narrow_hidden(name, B):
    check(*setup(name, 3, B, hidden=10), tag=f"{name} hidden 10")


@pytest.mark.parametrize("xdtype", [torch.float16, torch.float64])
@pytest.mark.parametrize("name", CFGS)
def test_model_batch_feature_dtypes(name, xdtype):
    check(*setup(name, 2, 129, xdtype=xdtype), tag=f"{name} {xdtype}")


@pytest.mark.parametrize("name", CFGS)
def test_model_batch_tc1x_forward(name):
    check(*setup(name, 3, 100, mode="tc1x"), train=False, tag="tc1x")
    check(*setup(name, 3, 100, mode="tc"), train=False, tag="tc inference")


def test_model_batch_trainer_matches_fused_trainers():
    name, M, B = "mini_cheetah-k4-contact", 3, 129
    cfg, models, batches, _ = setup(name, M, B)
    twins = [build_model(cfg, hidden=128, layers=4, seed=10 + m).to(DEV).set_mode("tc") for m in range(M)]
    tr = ModelBatchTrainer(ModelBatch(models), optimizer="adam", lr=1e-3)
    fts = [FusedTrainer(t, optimizer="adam", lr=1e-3) for t in twins]
    for step in range(5):
        active = [True, step < 3, True]                 # model 1 stops after three steps: its state must freeze
        losses = tr.train_step(batches, active=active)
        for m in range(M):
            if active[m]:
                lm = fts[m].train_step(batches[m])
                assert torch.equal(losses[m:m + 1], lm), f"step {step} model {m}: loss"
    torch.cuda.synchronize()
    for m in range(M):
        for (n, p), (n2, p2) in zip(models[m].named_parameters(), twins[m].named_parameters()):
            assert n == n2 and torch.equal(p, p2), f"model {m}: {n}"
        assert torch.equal(tr.exp_avg[m], fts[m].exp_avg) and torch.equal(tr.exp_avg_sq[m], fts[m].exp_avg_sq), f"model {m}: moments"
        assert tr.step_count[m] == fts[m].step_count
    # the parameters stay the models' own: a single-model forward reads row m of the batch buffer
    b = batches[1]
    assert models[1]._flat.data_ptr() == tr.mb.flat[1].data_ptr()
    preds = tr.infer(batches)
    with torch.no_grad():
        assert torch.equal(preds[1], models[1](b.x_dict, b.edge_index_dict))


def test_model_batch_rejections(restore_options):
    cfg, models, batches, eng = setup("mini_cheetah-k4-contact", 2, 64)
    nt = models[0].node_types
    xs = [torch.cat([b.x_dict[t] for b in batches]) for t in nt]
    flat = torch.stack([nm._flat for nm in models])
    eng.mode = N.MODE_FP32
    with pytest.raises(RuntimeError):
        eng.forward(xs, flat, train=True, n_models=2)
    eng.mode = N.MODE_TC
    N.set_option("stack", 0)
    with pytest.raises(RuntimeError):
        eng.forward(xs, flat, train=True, n_models=2)
    N.set_option("stack", 1)
    out = eng.forward(xs, flat, train=True, n_models=2)
    loss, dout = eng.loss(out, torch.cat([b.y for b in batches]), N.LOSS_CE2, n_models=2)
    eng.backward(dout, flat)
    with pytest.raises(ValueError, match="model batch"):
        eng.input_grad([True] * len(nt), flat)
    with pytest.raises(ValueError, match="process group"):
        ModelBatchTrainer(ModelBatch(models), process_group=object())
