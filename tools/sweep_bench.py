"""Hyperparameter sweeps as one model batch: K4 Mini Cheetah contact, L = 8, tc mode, 8 models = widths {16, 32, 64, 128} x
learning rates {1e-4, 1e-3}, at B graphs per model (64 and 1024).

Three comparisons per B, every arm timed with CUDA events after a warm-up, the arms alternated over --rounds rounds (the
median round is reported, with the spread):
  * sweep:    the mixed batch (forward + loss + backward replayed from one CUDA graph, then the optimizer launch, as in
              tools/model_batch_bench.py) against 8 sequential FusedTrainer.train_step_graphed steps;
  * mixing:   the same mixed batch against a uniform batch of 8 models of width 128 (same lrs): what mixing costs is the pad
              and compaction launches of the narrower models;
  * optimizer: one adam_step_models launch for the 8 models against the launches a model batch needed before, one per run of
              consecutive models with one step count and one lr (here 8, since neighbouring models differ in lr).
GPU name, power limit and SM clock are read in the same run.

usage: python tools/sweep_bench.py [--out profiles/r3_sweep.json] [--steps 20] [--warmup 3] [--rounds 5]
"""
import argparse
import json
import os
import statistics
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "morphsym-hgnn_b200"))
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))

import torch  # noqa: E402

from model_batch_bench import gpu_info, timed  # noqa: E402
from ms_hgnn import _native as N  # noqa: E402
from ms_hgnn.model_batch import ModelBatch, ModelBatchTrainer  # noqa: E402
from ms_hgnn.synthetic import CONFIGS, build_model, make_batch  # noqa: E402
from ms_hgnn.train import FusedTrainer  # noqa: E402

CFG, LAYERS = "mini_cheetah-k4-contact", 8
WIDTHS = [16, 16, 32, 32, 64, 64, 128, 128]
LRS = [1e-4, 1e-3] * 4
BS = (64, 1024)


def graphed_batch(tr, batches, dev):
    """A ModelBatchTrainer step with forward + loss + backward in one CUDA graph and the optimizer launched after it."""
    M = len(batches)
    tr.train_step(batches)
    eng, _, xs, flat, _ = tr._prepare(batches)
    y = torch.cat([b.y.reshape(-1) for b in batches])
    g = torch.cuda.CUDAGraph()
    torch.cuda.synchronize()
    with torch.cuda.graph(g):
        out = eng.forward(xs, flat, train=True, n_models=M)
        _, dout = eng.loss(out, y, tr._loss_kind(), want_grad=True, n_models=M)
        eng.backward(dout, flat, grads=tr.grads)
    captured = (xs, y, flat)         # the graph reads these addresses: they must outlive it (torch.cuda.graph empties the cache)

    def step():
        g.replay()
        tr._optimizer_step(None, dev)
    step.captured = captured
    return step


def optimizer_arms(tr, dev):
    """(one per-model launch, the grouped launches) on the trainer's buffers; both leave the same values."""
    buf, offs, M = tr.mb.buffer, tr.mb.offsets, len(tr.mb)
    mom = tr._moments
    stream = torch.cuda.current_stream(dev).cuda_stream
    steps = [1] * M

    def one():
        N.adam_step_models(buf.data_ptr(), tr.grads.data_ptr(), mom[0].data_ptr(), mom[1].data_ptr(), offs, steps, tr.lr, 0.9, 0.999, 1e-8,
                           0.0, stream)

    groups, m = [], 0
    while m < M:                          # runs of consecutive models with one step count and one lr
        e = m + 1
        while e < M and tr.lr[e] == tr.lr[m]:
            e += 1
        groups.append((offs[m], offs[e] - offs[m], tr.lr[m]))
        m = e

    def grouped():
        for o, n, lr in groups:
            N.adam_step(buf[o:].data_ptr(), tr.grads[o:].data_ptr(), mom[0, o:].data_ptr(), mom[1, o:].data_ptr(), n, 1, lr, 0.9, 0.999,
                        1e-8, 0.0, stream)
    return one, grouped, len(groups)


def run_B(B, steps, warmup, rounds, dev):
    cfg = CONFIGS[CFG]
    batches = [make_batch(cfg, B, seed=m).to(dev) for m in range(len(WIDTHS))]

    def models(widths):
        return [build_model(cfg, hidden=h, layers=LAYERS, seed=m).to(dev).set_mode("tc") for m, h in enumerate(widths)]
    mixed = ModelBatchTrainer(ModelBatch(models(WIDTHS), mixed_hidden=True), optimizer="adam", lr=LRS)
    uniform = ModelBatchTrainer(ModelBatch(models([128] * len(WIDTHS))), optimizer="adam", lr=LRS)
    fts = [FusedTrainer(t, optimizer="adam", lr=lr) for t, lr in zip(models(WIDTHS), LRS)]
    mixed_step = graphed_batch(mixed, batches, dev)
    opt_one, opt_grouped, n_groups = optimizer_arms(mixed, dev)
    arms = {
        "mixed_batch_graph": mixed_step,
        "sequential_graph": lambda: [ft.train_step_graphed(b) for ft, b in zip(fts, batches)],
        "uniform_128_batch_graph": graphed_batch(uniform, batches, dev),
        "adam_step_models": opt_one,
        "adam_grouped": opt_grouped,
    }
    times = {k: [] for k in arms}
    launches = {}
    for _ in range(rounds):
        for k, fn in arms.items():
            ms, nl = timed(fn, steps, warmup)
            times[k].append(ms)
            launches[k] = nl
    res = {k: {"ms_per_step_median": round(statistics.median(v), 4), "ms_per_step_min": round(min(v), 4), "ms_per_step_max": round(max(v), 4),
               "native_launches_per_step": launches[k]} for k, v in times.items()}
    med = {k: res[k]["ms_per_step_median"] for k in res}
    return {
        "B": B, "graphs_per_step": B * len(WIDTHS), "arms": res,
        "sweep": {"mixed_batch_ms": med["mixed_batch_graph"], "sequential_ms": med["sequential_graph"],
                  "speedup": round(med["sequential_graph"] / med["mixed_batch_graph"], 3)},
        "mixing": {"mixed_batch_ms": med["mixed_batch_graph"], "uniform_128_batch_ms": med["uniform_128_batch_graph"],
                   "mixed_over_uniform": round(med["mixed_batch_graph"] / med["uniform_128_batch_graph"], 3)},
        "optimizer": {"one_launch_ms": med["adam_step_models"], "grouped_ms": med["adam_grouped"], "grouped_launches": n_groups,
                      "grouped_over_one": round(med["adam_grouped"] / med["adam_step_models"], 3)},
    }


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r3_sweep.json"))
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--rounds", type=int, default=5)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "timing needs a CUDA device"
    dev = torch.device("cuda:0")
    result = {"workload": f"K4 Mini Cheetah contact, L={LAYERS}, tc mode, train step of {len(WIDTHS)} models",
              "widths": WIDTHS, "lrs": LRS, "gpu": gpu_info(), "configs": []}
    for B in BS:
        row = run_B(B, args.steps, args.warmup, args.rounds, dev)
        result["configs"].append(row)
        print(json.dumps(row), flush=True)
    result["gpu_at_end"] = gpu_info()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(result, f, indent=1)


if __name__ == "__main__":
    main()
