"""Cost of hidden widths below 128 (zero-padded into the 128-channel kernels): 16384 K4 Mini Cheetah contact graphs, tc mode.

For H in {10, 64, 128} reports, with the GPU name, power limit and clocks read in the same run:
  * train step time (FusedTrainer.train_step with Adam: forward, loss, backward, optimizer) and inference time (no-grad
    forward), CUDA events over --steps steps after warm-up; the widths are measured in alternating rounds and the median round
    is reported;
  * the pad_params profile kind per train step (k_pad_params in the forward + the two k_compact_grads launches of the
    backward), from the library's per-kernel event profiling in a separate pass, and its algorithmic bytes.

usage: python tools/hidden_width_bench.py [--out profiles/r3_hidden_width.json] [--batch 16384] [--steps 50] [--rounds 3]
"""
import argparse
import json
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "morphsym-hgnn_b200"))

import torch  # noqa: E402

from ms_hgnn import _native as N  # noqa: E402
from ms_hgnn.synthetic import CONFIGS, build_model, make_batch  # noqa: E402
from ms_hgnn.train import FusedTrainer  # noqa: E402

WIDTHS = (10, 64, 128)


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm,clocks.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    name, power, max_clock, clock = [s.strip() for s in q.stdout.strip().splitlines()[0].split(",")]
    return {"name": name, "power_limit": power, "max_sm_clock": max_clock, "sm_clock_at_start": clock}


def timed(fn, iters):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(iters):
        fn()
    b.record()
    b.synchronize()
    return a.elapsed_time(b) / iters


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r3_hidden_width.json"))
    ap.add_argument("--batch", type=int, default=16384)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--rounds", type=int, default=3)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("hidden_width_bench needs a CUDA device")
    info = gpu_info()
    dev = torch.device("cuda:0")
    cfg = CONFIGS["mini_cheetah-k4-contact"]
    B = args.batch
    b = make_batch(cfg, B, seed=1).to(dev)
    runs = {}
    for H in WIDTHS:
        nm = build_model(cfg, hidden=H, layers=8, seed=2).set_mode("tc").to(dev)
        nm.validate_edges = "cached"
        tr = FusedTrainer(nm, optimizer="adam", lr=1e-4)
        for _ in range(5):
            tr.train_step(b)
        eng = nm._last_engine
        xs = [b.x_dict[t].contiguous() for t in nm.node_types]

        def infer(eng=eng, nm=nm, xs=xs):
            eng.forward(xs, nm.flat_parameters, train=False)

        for _ in range(5):
            infer()
        torch.cuda.synchronize()
        runs[H] = {"trainer": tr, "infer": infer, "eng": eng, "train_ms": [], "infer_ms": []}
    for _ in range(args.rounds):
        for H in WIDTHS:
            r = runs[H]
            r["train_ms"].append(timed(lambda: r["trainer"].train_step(b), args.steps))
            r["infer_ms"].append(timed(r["infer"], args.steps))
    res = {"gpu": info, "batch": B, "mode": "tc", "config": cfg.name, "layers": 8, "steps_per_round": args.steps,
           "rounds": args.rounds, "widths": {}}
    for H in WIDTHS:
        r = runs[H]
        N.profile_enable(True)
        try:
            N.profile_read()
            for _ in range(10):
                r["trainer"].train_step(b)
            prof = N.profile_read()
        finally:
            N.profile_enable(False)
        pad_ms, pad_launches = prof.get("pad_params", (0.0, 0))
        eng = r["eng"]
        n_ext = eng.n_params
        internal = 0 if H == 128 else N.NativePlan(dict(eng.spec, hidden=128, pad_hidden=False)).n_params
        t_train, t_infer = statistics.median(r["train_ms"]), statistics.median(r["infer_ms"])
        res["widths"][str(H)] = {
            "params": n_ext, "train_step_ms": round(t_train, 4), "train_step_ms_rounds": [round(v, 4) for v in r["train_ms"]],
            "train_graphs_per_s": round(B / (t_train * 1e-3)), "inference_ms": round(t_infer, 4),
            "inference_ms_rounds": [round(v, 4) for v in r["infer_ms"]], "inference_graphs_per_s": round(B / (t_infer * 1e-3)),
            "pad_params_ms_per_step": round(pad_ms / 10, 4), "pad_params_launches_per_step": pad_launches / 10,
            # pad: external read + internal written; compact: internal read (the block that is kept) + external written
            "pad_params_bytes_per_step": 4 * (n_ext + internal) + 8 * n_ext if H != 128 else 0,
        }
    res["note"] = ("train_step: FusedTrainer.train_step (Adam), CUDA events over steps_per_round steps, median of the rounds, widths "
                   "alternated within each round; inference: no-grad forward; pad_params: the library's event profiling in a separate "
                   "pass of 10 train steps (k_pad_params + 2 x k_compact_grads per step)")
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res))


if __name__ == "__main__":
    main()
