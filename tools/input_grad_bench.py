"""Input-gradient timing at the flagship size: 16384 K4 Mini Cheetah contact graphs, tensor-core mode.

Reports, with the GPU name and power limit read in the same run:
  * the dx_encoder kernel (k_tc_encoder_dx) time: CUDA events around many launches of mshgnn_input_grad on the workspace a
    backward left, after warm-up; its algorithmic bytes (dx written + dpre0 (hi, lo) read), GB/s and share of the HBM bandwidth
    (MEASURED_PEAKS.json when present, as bench.py does);
  * backward time (CUDA events, forward excluded) with parameter gradients only, parameter + input gradients, and input only.

usage: python tools/input_grad_bench.py [--out profiles/r3_input_grad.json] [--batch 16384] [--iters 200]
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
from ms_hgnn.synthetic import CONFIGS, build_model, make_batch  # noqa: E402


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    name, power, clock = [s.strip() for s in q.stdout.strip().splitlines()[0].split(",")]
    return {"name": name, "power_limit": power, "max_sm_clock": clock}


def hbm_gbs():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        return json.load(open(p))["hbm_gbs"], "measured"
    return 6650.0, "fallback"


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
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r3_input_grad.json"))
    ap.add_argument("--batch", type=int, default=16384)
    ap.add_argument("--iters", type=int, default=200)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("input_grad_bench needs a CUDA device")
    dev = torch.device("cuda:0")
    cfg = CONFIGS["mini_cheetah-k4-contact"]
    B = args.batch
    b = make_batch(cfg, B, seed=1).to(dev)
    nm = build_model(cfg, layers=8, seed=2).set_mode("tc").to(dev)
    nm.validate_edges = "cached"
    xs = [b.x_dict[t].contiguous() for t in nm.node_types]
    out = nm(b.x_dict, b.edge_index_dict)           # builds the engine and the flat parameter buffer
    eng, flat = nm._last_engine, nm.flat_parameters
    eng.forward(xs, flat, train=True)
    _, dout = eng.loss(out.detach().contiguous(), b.y, N.LOSS_CE2)
    grads = torch.empty(eng.n_params, device=dev)
    dx = [torch.empty_like(x) for x in xs]
    ws = eng._ws
    stream = torch.cuda.current_stream().cuda_stream

    def bwd(param_grads):
        eng.backward(dout, flat, grads if param_grads else None, param_grads=param_grads)

    def igrad():
        eng.plan.input_grad(B, flat.data_ptr(), [t.data_ptr() for t in dx], ws.data_ptr(), ws.numel(), eng.mode, stream)

    bwd(True)
    for _ in range(10):
        igrad()
    torch.cuda.synchronize()
    t_dx = timed(igrad, args.iters)

    def igrad_1x():       # same workspace layout: the dpre0 hi images only and one MMA per product (what the operand side costs)
        eng.plan.input_grad(B, flat.data_ptr(), [t.data_ptr() for t in dx], ws.data_ptr(), ws.numel(), N.MODE_TC_1X, stream)

    igrad_1x()
    t_dx_1x = timed(igrad_1x, args.iters)

    # backward variants: a forward before each backward (the backward needs the forward's workspace), timed apart
    def variant(param_grads, inputs, n=30):
        ta, tb = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        tot = 0.0
        for i in range(n + 5):
            eng.forward(xs, flat, train=True)
            ta.record()
            bwd(param_grads)
            if inputs:
                igrad()
            tb.record()
            tb.synchronize()
            if i >= 5:
                tot += ta.elapsed_time(tb)
        return tot / n

    t_p = variant(True, False)
    t_pi = variant(True, True)
    t_i = variant(False, True)

    nodes = eng.spec["nodes_per_graph"]
    widths = eng.spec["in_width"]
    live = sum(eng.plan.describe()["need"][0])
    written = 4 * sum(n * k for n, k in zip(nodes, widths))               # fp32 dx rows per graph
    read = live * 128 * 2 * 2                                              # dpre0 (hi, lo) fp16 per live slot
    total = (written + read) * B
    peak, src = hbm_gbs()
    gbs = total / (t_dx * 1e-3) / 1e9
    res = {
        "gpu": gpu_info(), "batch": B, "mode": "tc", "config": cfg.name, "iters": args.iters,
        "dx_encoder_ms": round(t_dx, 4), "dx_encoder_hi_only_1_mma_ms": round(t_dx_1x, 4),
        "bytes_per_graph": {"dx_written": written, "dpre0_read": read}, "bytes_per_batch": total,
        "achieved_gbs": round(gbs, 1), "hbm_gbs": peak, "hbm_gbs_source": src, "share_of_hbm": round(gbs / peak, 3),
        "bound_ms": round(total / (peak * 1e9) * 1e3, 4),
        "backward_ms": {"param_grads": round(t_p, 4), "param_and_input_grads": round(t_pi, 4), "input_only": round(t_i, 4)},
        "note": "dx_encoder: CUDA events around many mshgnn_input_grad calls on one backward's workspace (dx ~700 MB per batch, "
                "larger than L2); backward_ms: events around backward (+ input_grad), forward excluded",
    }
    os.makedirs(os.path.dirname(args.out), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res))


if __name__ == "__main__":
    main()
