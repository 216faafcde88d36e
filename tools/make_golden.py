"""Generates tests/golden/* from a checkout of the reference repository (MSHGNN_REFERENCE=<its directory>).

1. mi_grf_ckpt.pt  - from the reference's shipped checkpoint tests/test_models/epoch=48-val_MSE_loss=6.33834.ckpt:
   its embedded 20-graph batch (x, edge_index, y), the weights rounded to float32 (5.3 MB instead of 10.6 MB),
   the fp64 oracle output on exactly those numbers, and the pinned metrics.
2. seeded.pt       - oracle outputs / losses / gradient norms of every model class on seeded synthetic batches
   (weights and inputs are regenerated from the seeds by the tests; only the expected numbers are stored).
3. reference_models.pt - outputs, loss and per-tensor gradient digests of the reference's UNMODIFIED model files
   (src/ms_hgnn/lightning_py/hgnn*.py, imported against oracle/pyg_shim by oracle/reference_pin.py) for
   every CONFIGS entry at L = 8 on a seeded 5-graph batch with seeded weights - the pin of the MS-HGNN-specific oracle
   semantics (sign tables, base_transform + residual, mean relations, output decoders) and of all gradients.
4. reference_cfg.json - the reference's group tables (cfg/*.yaml), parsed.
"""
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in ("morphsym-hgnn_b200", "oracle", "tests"):
    sys.path.insert(0, os.path.join(ROOT, p))
import mshgnn_oracle as O  # noqa: E402
import reference_pin as RP  # noqa: E402
from helpers import oracle_model, oracle_run  # noqa: E402
from ms_hgnn.synthetic import CONFIGS, make_batch  # noqa: E402

GOLD = os.path.join(ROOT, "tests", "golden")
CKPT = os.path.join(RP.REF_ROOT, "tests", "test_models", "epoch=48-val_MSE_loss=6.33834.ckpt")
SEEDED_CASES = [(n, 3, 2) for n in CONFIGS]   # (config, B, layers)
RP_B, RP_LAYERS, RP_BATCH_SEED, RP_WEIGHT_SEED = 5, 8, 11, 4


def main():
    if not RP.available():
        raise SystemExit("set MSHGNN_REFERENCE to the directory of a checkout of the reference repository")
    os.makedirs(GOLD, exist_ok=True)
    torch.set_default_dtype(torch.float64)
    sd, hp, batch = O.load_reference_checkpoint(CKPT)
    md = (list(hp["data_metadata"][0]), [tuple(e) for e in hp["data_metadata"][1]])
    m = O.GRF_HGNN(hp["hidden_channels"], hp["num_layers"], md, regression=True, in_dims={t: v.shape[1] for t, v in batch["x"].items()})
    m.load_state_dict(sd)
    B = batch["x"]["base"].shape[0]
    out64 = m(batch["x"], batch["edge_index"]).detach()
    y = batch["y"].reshape(B, 4)
    pins64 = [O.mse_loss(out64.reshape(B, 4), y).item(), O.rmse_loss(out64.reshape(B, 4), y).item(), O.l1_loss(out64.reshape(B, 4), y).item()]
    print("fp64 checkpoint pins", pins64)
    sd32 = {k: v.float() for k, v in sd.items()}
    m.load_state_dict({k: v.double() for k, v in sd32.items()})
    out = m(batch["x"], batch["edge_index"]).detach()
    torch.save({"metadata": md, "hidden": hp["hidden_channels"], "layers": hp["num_layers"], "state_dict_f32": sd32,
                "x": batch["x"], "edge_index": batch["edge_index"], "y": batch["y"], "oracle_out": out,
                "pins_fp64_weights": pins64, "reference_pins": [6.33834, 2.51761, 2.31058],
                "source": "tests/test_models/epoch=48-val_MSE_loss=6.33834.ckpt; pins tests/testGnnLightning.py:L214-216"},
               os.path.join(GOLD, "mi_grf_ckpt.pt"))
    seeded = {}
    torch.set_default_dtype(torch.float32)
    for name, Bs, layers in SEEDED_CASES:
        cfg = CONFIGS[name]
        b = make_batch(cfg, Bs, seed=11)
        om = oracle_model(cfg, layers=layers, seed=5)
        o, l, g = oracle_run(cfg, om, b)
        seeded[name] = {"B": Bs, "layers": layers, "batch_seed": 11, "model_seed": 5, "out": o, "loss": l,
                        "grad_norms": {k: v.norm().item() for k, v in g.items()},
                        "x_checksum": {k: v.double().sum().item() for k, v in b.x_dict.items()},
                        "w_checksum": sum(p.double().sum().item() for p in om.parameters())}
    torch.save(seeded, os.path.join(GOLD, "seeded.pt"))
    from helpers import oracle_loss
    ref = {}
    for name, cfg in CONFIGS.items():
        b = make_batch(cfg, RP_B, seed=RP_BATCH_SEED)
        rm = RP.build_reference_model(cfg, RP_LAYERS, 1)
        RP.materialize(rm, b)
        rm.load_state_dict(RP.seeded_state_dict(rm, RP_WEIGHT_SEED))
        o, l, g = RP.reference_run(cfg, rm, b, oracle_loss)
        ref[name] = {"B": RP_B, "layers": RP_LAYERS, "batch_seed": RP_BATCH_SEED, "weight_seed": RP_WEIGHT_SEED,
                     "keys": list(rm.state_dict().keys()), "shapes": [tuple(v.shape) for v in rm.state_dict().values()],
                     "out": o, "loss": l, "grad_digest": RP.grad_digest(g),
                     "grad_is_none": sorted(n for n, p in rm.named_parameters() if p.grad is None)}
        print("reference", name, tuple(o.shape), float(l))
    torch.save({"cases": ref, "source": "unmodified src/ms_hgnn/lightning_py/hgnn*.py of the reference @ 9e55c68 run against "
                "oracle/pyg_shim (torch_geometric 2.5.0 semantics), fp64, CPU"}, os.path.join(GOLD, "reference_models.pt"))
    import glob
    import json
    import yaml
    tables = {os.path.basename(p)[:-5]: yaml.safe_load(open(p)) for p in sorted(glob.glob(os.path.join(RP.REF_ROOT, "cfg", "*.yaml")))}
    with open(os.path.join(GOLD, "reference_cfg.json"), "w") as f:
        f.write(json.dumps(tables, sort_keys=True) + "\n")
    for f in os.listdir(GOLD):
        print(f, os.path.getsize(os.path.join(GOLD, f)))


if __name__ == "__main__":
    main()
