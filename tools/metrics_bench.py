"""Metric side of a step: the op-by-op torch path against one mshgnn_step_metrics_ex call.

Two steps of the paper's regression tasks, at B = 64 (the reference's batch sizes) and 16384 graphs:
  * COM K4 (Solo12, COM_HGNN_SYM_Lightning): ``_metrics_step_op_by_op`` (six metric objects, reshapes, un-standardisation,
    two cosine similarities) against ``_metrics_step_fused`` (METRIC_COM);
  * A1 world-frame GRF (HGNN_C2_Lightning_Reg, grf_body_to_world_frame=True): the previous CUDA path (the fused MSE call for
    the body frame, then quaternion normalisation, rotation matrices, two batched matmuls and three metric objects) against
    ``_worldframe_metrics_fused`` (METRIC_GRF_WORLD).
The gradient-carrying loss is the same native launch on both paths and is left out.  Reported per step, with the GPU name,
power limit and SM clock read in the same run:
  * time: CUDA events over --iters steps, old and new alternated in --rounds rounds, median round;
  * device work: kernels and memcpy / memset operations per step, from torch.profiler (CUDA activity) in a separate pass;
  * the largest relative difference between the two paths' batch values on the timed inputs.

usage: python tools/metrics_bench.py [--out profiles/r3_metrics.json] [--iters 200] [--rounds 5]
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
from ms_hgnn import morphology as M  # noqa: E402
from ms_hgnn.lightning_py.gnnLightning import HGNN_C2_Lightning_Reg  # noqa: E402
from ms_hgnn.lightning_py.gnnLightning_com import COM_HGNN_SYM_Lightning, Standarizer  # noqa: E402
from ms_hgnn.synthetic import CONFIGS, make_batch  # noqa: E402

DEV = torch.device("cuda:0")


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


def device_ops(fn, steps=10):
    """(kernels, memcpy + memset operations) per step seen by torch.profiler's CUDA activity."""
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(steps):
            fn()
        torch.cuda.synchronize()
    kernels = copies = 0
    for e in prof.events():
        if e.device_type != torch.autograd.DeviceType.CUDA:
            continue
        if e.name.startswith(("Memcpy", "Memset")):
            copies += 1
        else:
            kernels += 1
    return kernels / steps, copies / steps


def com_case(B, gen):
    cfg = CONFIGS["solo12-k4-com"]
    tpl = M.TEMPLATES[cfg.template]
    m = COM_HGNN_SYM_Lightning(128, 8, tpl.metadata, make_batch(cfg, 2), "adam", 1e-3, model_type="heterogeneous_gnn_k4_com",
                               symmetry_mode="MorphSym", group_operator_path=M.cfg_path(cfg.group))
    m.standarizer = Standarizer(None, None, torch.randn(6, generator=gen).numpy(), (torch.rand(6, generator=gen) + 0.5).numpy())
    pred = torch.randn(B, 24, generator=gen).to(DEV)
    y = (pred.cpu() + 0.5 * torch.randn(B, 24, generator=gen)).to(DEV)
    old = lambda: m._metrics_step_op_by_op(y, pred)
    new = lambda: m._metrics_step_fused(y, pred)
    names = ("rmse_loss", "mse_loss_lin", "mse_loss_ang", "cos_sim_lin", "cos_sim_ang", "avg_cos_sim")
    return old, new, lambda: [getattr(m, k) for k in names], m.reset_all_metrics


def grf_case(B, gen):
    cfg = CONFIGS["a1-c2-grf"]
    tpl = M.TEMPLATES[cfg.template]
    m = HGNN_C2_Lightning_Reg(128, 8, tpl.metadata, make_batch(cfg, 2), "adam", 1e-3, regression=True, symmetry_mode="MorphSym",
                              group_operator_path=M.cfg_path(cfg.group), grf_body_to_world_frame=True, grf_dimension=3)
    pred = (torch.randn(B, 12, generator=gen) * 40).to(DEV)
    y = (pred.cpu() + 5 * torch.randn(B, 12, generator=gen)).to(DEV)
    q = torch.randn(B, 4, generator=gen).to(DEV)

    def old():      # the CUDA path before METRIC_GRF_WORLD: Base_Lightning's fused MSE call, then the world frame op by op
        b = m._fused.update(N.LOSS_MSE, pred.reshape(-1), y, pred.numel(), 1)
        b = b[21:23].clone()
        m.rmse_loss, m.l1_loss = b[0], b[1]
        m._worldframe_metrics_op_by_op(y, pred, q, False)

    new = lambda: m._worldframe_metrics_fused(y, pred, q, False)
    names = ("rmse_loss", "l1_loss", "mse_loss_worldframe", "rmse_loss_worldframe", "l1_loss_worldframe")
    return old, new, lambda: [getattr(m, k) for k in names], m.reset_all_metrics_worldframe


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r3_metrics.json"))
    ap.add_argument("--iters", type=int, default=200)
    ap.add_argument("--rounds", type=int, default=5)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("metrics_bench needs a CUDA device")
    info = gpu_info()
    gen = torch.Generator().manual_seed(0)
    res = {"gpu": info, "iters": args.iters, "rounds": args.rounds, "cases": []}
    for case, make in (("com_k4_step", com_case), ("a1_worldframe_grf_step", grf_case)):
        for B in (64, 16384):
            old, new, values, reset = make(B, gen)
            reset(); old(); v_old = [float(v) for v in values()]
            reset(); new(); v_new = [float(v) for v in values()]
            diff = max(abs(a - b) / abs(b) for a, b in zip(v_new, v_old))
            for fn in (old, new):                       # warm-up: module load, caching allocator, cuBLAS handles
                for _ in range(20):
                    fn()
            torch.cuda.synchronize()
            t_old, t_new = [], []
            for _ in range(args.rounds):
                t_old.append(timed(old, args.iters))
                t_new.append(timed(new, args.iters))
            k_old, c_old = device_ops(old)
            k_new, c_new = device_ops(new)
            row = {"case": case, "B": B,
                   "old": {"ms_per_step": statistics.median(t_old), "ms_rounds": t_old, "kernels_per_step": k_old,
                           "memcpy_memset_per_step": c_old},
                   "fused": {"ms_per_step": statistics.median(t_new), "ms_rounds": t_new, "kernels_per_step": k_new,
                             "memcpy_memset_per_step": c_new},
                   "max_rel_diff_of_batch_values": diff}
            print(json.dumps(row), flush=True)
            res["cases"].append(row)
    res["gpu_after"] = gpu_info()
    res["note"] = ("metric side of one step only (the gradient-carrying native loss is the same launch on both paths); fp32 "
                   "predictions and labels resident on the device; old = the op-by-op torch path the modules ran on CUDA batches "
                   "before the fused kinds, fused = one mshgnn_step_metrics_ex call + the clone of the logged values")
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
    print("wrote", args.out)


if __name__ == "__main__":
    main()
