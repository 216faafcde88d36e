"""Model batches against sequential single-model steps: K4 Mini Cheetah contact, H = 128, L = 8, tc mode.

For M in {1, 4, 16} models and B in {64, 256, 1024} graphs per model, one training step (forward + loss + backward + Adam)
of all M models is timed four ways:
  * batch_eager:  ModelBatchTrainer.train_step (one native step for all M models);
  * seq_eager:    M FusedTrainer.train_step calls, one per model;
  * batch_graph:  forward + loss + backward of the model batch replayed from one CUDA graph, then the optimizer launch;
  * seq_graph:    M FusedTrainer.train_step_graphed calls.
Reported per configuration: CUDA-event time per step of all M models (ms), graphs/s (M x B per step), native launches per
step (mshgnn_launch_count; a graph replay counts only the launches made outside the graph), and the bytes of (hi, lo) weight
images the step writes and reads back, counted from the plan (they grow with M).  GPU name, power limit and SM clock are read
in the same run.  Weight-image bytes are a count, not a measurement, and are filled in without a GPU as well (--count-only).

usage: python tools/model_batch_bench.py [--out profiles/r3_model_batch.json] [--steps 20] [--warmup 3] [--count-only]
"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "morphsym-hgnn_b200"))

import torch  # noqa: E402

from ms_hgnn import _native as N  # noqa: E402
from ms_hgnn import morphology as M_  # noqa: E402
from ms_hgnn.engine import build_spec  # noqa: E402
from ms_hgnn.model_batch import ModelBatch, ModelBatchTrainer  # noqa: E402
from ms_hgnn.synthetic import CONFIGS, build_model, make_batch  # noqa: E402
from ms_hgnn.train import FusedTrainer  # noqa: E402

CFG = "mini_cheetah-k4-contact"
MS, BS = (1, 4, 16), (64, 256, 1024)


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm,clocks.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    name, power, max_clock, clock = [s.strip() for s in q.stdout.strip().splitlines()[0].split(",")]
    return {"name": name, "power_limit": power, "max_sm_clock": max_clock, "sm_clock_at_start": clock}


def image_bytes_per_model():
    """(hi, lo) fp16 images of one model: the 128 x 128 layer weight images and the encoder weight image (k_fwd_prologue writes them,
    the stack / encoder kernels read them)."""
    cfg = CONFIGS[CFG]
    nm = build_model(cfg, hidden=128, layers=8)
    tpl = M_.TEMPLATES[cfg.template]
    spec = build_spec(nm.node_types, tpl.nodes_per_graph, cfg.in_width, nm.edge_types, tpl.edges, nm.mean_relations, 128, 8,
                      nm.morph_sym, "base" if nm.morph_sym else None, nm.decode_node, nm._out_channels, nm._in_sign(dict(cfg.in_width)),
                      nm._out_sign(), pad_hidden=True)
    d = N.NativePlan(spec).describe()
    return 2 * 2 * (d["n_mats16"] * 128 * 128 + d["n_types"] * 128 * d["enc_kmax"]), 4 * N.NativePlan(spec).n_params


def timed(fn, steps, warmup):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    n0 = N.launch_count()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(steps):
        fn()
    b.record()
    b.synchronize()
    return a.elapsed_time(b) / steps, (N.launch_count() - n0) / steps


def run_config(Mn, B, steps, warmup, dev):
    cfg = CONFIGS[CFG]
    models = [build_model(cfg, hidden=128, layers=8, seed=m).to(dev).set_mode("tc") for m in range(Mn)]
    twins = [build_model(cfg, hidden=128, layers=8, seed=m).to(dev).set_mode("tc") for m in range(Mn)]
    batches = [make_batch(cfg, B, seed=m).to(dev) for m in range(Mn)]
    tr = ModelBatchTrainer(ModelBatch(models), optimizer="adam", lr=1e-4)
    fts = [FusedTrainer(t, optimizer="adam", lr=1e-4) for t in twins]
    res = {}
    res["batch_eager"] = timed(lambda: tr.train_step(batches), steps, warmup)
    res["seq_eager"] = timed(lambda: [ft.train_step(b) for ft, b in zip(fts, batches)], steps, warmup)
    # model batch in a CUDA graph: forward + loss + backward captured once, the optimizer launched per step (as train_step_graphed)
    tr.train_step(batches)
    eng, Bm, xs, flat, _ = tr._prepare(batches)
    y = torch.cat([b.y.reshape(-1) for b in batches]) if Mn > 1 else batches[0].y
    g = torch.cuda.CUDAGraph()
    torch.cuda.synchronize()
    with torch.cuda.graph(g):
        out = eng.forward(xs, flat, train=True, n_models=Mn)
        _, dout = eng.loss(out, y, tr._loss_kind(), want_grad=True, n_models=Mn)
        eng.backward(dout, flat, grads=tr.grads)

    def batch_graph():
        g.replay()
        tr._optimizer_step(None, dev)
    res["batch_graph"] = timed(batch_graph, steps, warmup)
    res["seq_graph"] = timed(lambda: [ft.train_step_graphed(b) for ft, b in zip(fts, batches)], steps, warmup)
    out = {}
    for k, (ms, launches) in res.items():
        out[k] = {"ms_per_step": round(ms, 4), "graphs_per_s": round(Mn * B / (ms * 1e-3)), "native_launches_per_step": launches}
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r3_model_batch.json"))
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--count-only", action="store_true", help="no GPU: write the counted weight-image bytes only")
    args = ap.parse_args()
    img, par = image_bytes_per_model()
    result = {"workload": "K4 Mini Cheetah contact, H=128, L=8, tc mode, train step (forward + loss + backward + Adam) of all M models",
              "weight_image_bytes_per_model": img, "fp32_parameter_bytes_per_model": par, "configs": []}
    if not args.count_only:
        assert torch.cuda.is_available(), "timing needs a CUDA device (--count-only counts bytes without one)"
        result["gpu"] = gpu_info()
    dev = torch.device("cuda:0") if not args.count_only else None
    for Mn in MS:
        for B in BS:
            row = {"M": Mn, "B": B, "graphs_per_step": Mn * B,
                   "weight_image_bytes_per_step": {"model_batch": Mn * img, "sequential": Mn * img}}
            row.update(run_config(Mn, B, args.steps, args.warmup, dev) if not args.count_only else
                       {k: "not measured" for k in ("batch_eager", "seq_eager", "batch_graph", "seq_graph")})
            result["configs"].append(row)
            print(json.dumps(row), flush=True)
    if not args.count_only:
        result["gpu_at_end"] = gpu_info()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(result, f, indent=1)


if __name__ == "__main__":
    main()
