#!/usr/bin/env python
"""bench.py - graphs/s of the MS-HGNN train step (and inference) on N B200s.

Contract (one JSON line on rank 0):
  value      train-step graphs/s, whole job, inputs resident in HBM (fused native step: forward ->
             loss head -> backward -> [all-reduce of the flat gradient] -> Adam), CUDA events, max over ranks
  e2e        the same metric through the public API with HOST (pinned) buffers: per step H2D of the
             batch (features, edge_index, labels), the train step, D2H of the loss
  inference  no-grad forward graphs/s (device resident)
  roofline   dominant kernel: algorithmic FLOPs (SURVEY 8d) / measured kernel time vs measured peak
  cpu_baseline  the oracle (CPU restatement of the reference's PyG op sequence) timed on host cores
`--impl reference` times that oracle alone (the reference's own code cannot be installed: it needs
torch_geometric / lightning, which are not in this image and there is no network).
"""
import argparse
import atexit
import json
import os
import statistics
import subprocess
import sys
import tempfile
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
for _p in (os.path.join(ROOT, "morphsym-hgnn_b200"), os.path.join(ROOT, "oracle"), os.path.join(ROOT, "tests")):
    if _p not in sys.path:
        sys.path.insert(0, _p)

import torch  # noqa: E402

WORKLOAD = "mini_cheetah-k4-contact"      # BASELINE.json configs[2]: MS-HGNN K4 Mini Cheetah contact, batch 16384 per GPU
PER_GPU_BATCH = 16384
REFERENCE_SAMPLE = 4096                    # graphs per step of the CPU arm (bounded sample, see run_reference)
METRIC = "train-step graphs/s (MS-HGNN K4 Mini Cheetah contact, H=128, L=8, fwd+loss+bwd+allreduce+Adam)"

# Algorithmic work per graph, SURVEY 8d (minimum: zero aggregates skipped, roots pre-summed, dead last layer):
#   MAC: encoder sum n_t*in_t*H ; layers (R*(L-1)+R_last)*H^2 with R=64, R_last=8 ; decoder n_out*H*C
_ENC_MAC = (4 * 900 + 12 * 300 + 4 * 900) * 128
_LAY_MAC = (64 * 7 + 8) * 128 * 128
_DEC_MAC = 4 * 128 * 2
ALG = {
    "fwd_flop": 2 * (_ENC_MAC + _LAY_MAC + _DEC_MAC),                      # 17.71 MFLOP
    "train_flop": 2 * (2 * _ENC_MAC + 3 * _LAY_MAC + 3 * _DEC_MAC),        # 50.36 MFLOP
    "in_bytes": 43200,                                                     # fp32 features per graph
    # per kernel kind (names from mshgnn_kernel_kind_name)
    "encoder_fwd": 2 * _ENC_MAC,
    "conv_fwd": 2 * (_LAY_MAC - 8 * 7 * 128 * 128),             # layer rows minus the base-MLP rows
    "base_mlp_fwd": 2 * (8 * 7 * 128 * 128),
    "dx_bwd": 2 * (_LAY_MAC - 8 * 7 * 128 * 128),
    "base_mlp_bwd": 2 * (8 * 7 * 128 * 128),
    "stack_fwd": 2 * _LAY_MAC,                                  # cross-layer kernel: conv + chained base MLP of all layers
    "stack_bwd": 2 * _LAY_MAC,                                  # dX chain + chained base MLP backward of all layers
    "dw_layers": 2 * _LAY_MAC,
    "dw_encoder": 2 * _ENC_MAC,
}


DUMP_LIMIT = 64 << 20                      # bytes written by --dump-outputs at most

TRAFFIC_FILE = "r2_dominant_traffic.json"   # ncu DRAM bytes of THIS round's kernels (tools/launch_traffic.py); keyed by kernel kind


KERNEL_SWITCHES = ("MSHGNN_STACK", "MSHGNN_STACK_2CTA", "MSHGNN_ROWGEMM", "MSHGNN_ENCODER", "MSHGNN_ENC_TPI", "MSHGNN_ENC_DW", "MSHGNN_ENC_PF",
                   "MSHGNN_ENC_DEBUG", "MSHGNN_STACK_DEBUG")


def recorded_traffic():
    """DRAM bytes from the committed ncu captures (profiles/): per launch of the dominant kernels and per train step.  The capture belongs
    to the DEFAULT kernel selection of this round: when a kernel switch of the library is set in the environment another kernel runs and
    the recorded bytes are not its bytes - no traffic is reported then (stderr says why)."""
    p = os.path.join(ROOT, "profiles", TRAFFIC_FILE)
    if not os.path.exists(p):
        return {}
    overridden = [k for k in KERNEL_SWITCHES if os.environ.get(k) not in (None, "")]
    if overridden:
        print(f"bench.py: {', '.join(overridden)} set - profiles/{TRAFFIC_FILE} was captured on the default kernels, roofline.traffic / hbm_step omitted",
              file=sys.stderr)
        return {}
    return json.load(open(p))


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return {"hbm_gbs": d["hbm_gbs"], "tflops": d.get("bf16_tflops_sustained", d["bf16_tflops"]), "src": "measured"}
    return {"hbm_gbs": 6650.0, "tflops": 1400.0, "src": "fallback"}


class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        self.p = None
        try:
            self.p = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "20",
                                       "-i", str(gpu_index)], stdout=self.f, stderr=subprocess.DEVNULL)
            atexit.register(self.p.kill)              # a run that fails before stop() must not leave the sampler running
        except Exception:
            self.p = None

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        if self.p is None:
            return out
        self.p.terminate()
        try:
            self.p.wait(timeout=5)
        except Exception:
            self.p.kill()
        self.f.flush()
        rows = [r.strip().split(", ") for r in open(self.f.name).read().strip().splitlines() if r.strip()]
        os.unlink(self.f.name)
        sm, reasons, mx = [], set(), None
        for r in rows:
            if len(r) < 9:
                continue
            try:
                sm.append(float(r[1])); mx = float(r[2])
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[5:9]):
                if v.strip().lower() == "active":
                    reasons.add(name)
        if sm:
            out.update(sm_mhz=statistics.median(sm), sm_max_mhz=mx, reasons=sorted(reasons), samples=len(sm))
        return out


def dump_outputs(path, arrays):
    """Writes each tensor as <path>/<name>.npy (float64 stays float64, everything else becomes float32).  Above DUMP_LIMIT
    bytes in all, every array is replaced by the same share of its elements at fixed, seeded positions (flattened)."""
    import numpy as np
    os.makedirs(path, exist_ok=True)
    arrays = {k: v.detach().cpu() if v.dtype == torch.float64 else v.detach().float().cpu() for k, v in arrays.items()}
    total = sum(v.numel() * v.element_size() for v in arrays.values())
    for i, (name, v) in enumerate(arrays.items()):
        if total > DUMP_LIMIT:
            keep = max(1, v.numel() * DUMP_LIMIT // total)
            idx = torch.randperm(v.numel(), generator=torch.Generator().manual_seed(i))[:keep].sort().values
            v = v.reshape(-1)[idx]
        np.save(os.path.join(path, name + ".npy"), v.numpy())


def oracle_train_rate(B, steps, warmup, dtype=torch.float64, threads=None):
    """graphs/s of the CPU oracle train step (fwd + loss + bwd + torch.optim.Adam) on the host cores."""
    import mshgnn_oracle as O
    from helpers import oracle_loss
    from ms_hgnn.synthetic import CONFIGS, build_model, make_batch
    if threads:
        torch.set_num_threads(threads)
    cfg = CONFIGS[WORKLOAD]
    prev = torch.get_default_dtype()
    torch.set_default_dtype(dtype)
    try:
        model = build_model(cfg, 128, 8, 0, module=O)
        batch = make_batch(cfg, B, seed=1, dtype=dtype)
        opt = torch.optim.Adam(model.parameters(), lr=1e-4)
        ts = []
        for i in range(warmup + steps):
            t0 = time.perf_counter()
            opt.zero_grad()
            out = model(batch.x_dict, batch.edge_index_dict)
            loss = oracle_loss(cfg, out, batch.y, B)
            loss.backward()
            opt.step()
            if i >= warmup:
                ts.append(time.perf_counter() - t0)
    finally:
        torch.set_default_dtype(prev)
    return B / (sum(ts) / len(ts)), B / min(ts)


def run_reference(args, rank):
    if rank != 0:
        return
    cores = os.cpu_count()
    torch.set_num_threads(cores)
    # bounded sample of the 16384-graph step: 4096 graphs per CPU step (8.7 GB of fp64 autograd state, ~1 s per step on 16
    # cores; the full 16384 would need ~35 GB and 25 x 3.5 s).  Throughput is per graph, so the sample size only matters
    # through cache effects: 1024 / 4096 graphs per step measured within 10 % of each other.
    B = REFERENCE_SAMPLE
    mean_rate, best_rate = oracle_train_rate(B, args.steps, args.warmup)
    ms = 1e3 * B / mean_rate
    line = {
        "impl": "reference", "metric": METRIC, "value": mean_rate, "unit": "graphs/s", "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f64", "data": "synthetic",
        "config": {"workload": WORKLOAD, "per_gpu_batch": PER_GPU_BATCH, "global_batch": PER_GPU_BATCH * max(args.gpus, 1), "hidden": 128, "layers": 8,
                   "sample_graphs_per_step": B,
                   "note": "CPU oracle = pure-PyTorch restatement of the reference's torch_geometric op sequence, pinned to the reference's "
                           "unmodified model files (tests/test_reference_pin.py); the reference itself is not installable offline.  fp64 like "
                           "the reference.  Each step is a bounded 4096-graph sample of the 16384-graph batch (graphs/s is per graph)"},
        "cpu_baseline": {"value": mean_rate, "unit": "graphs/s", "cores": torch.get_num_threads(), "kind": "port",
                         "sample": f"{args.steps} train steps of {B} graphs (of the 16384-graph batch), fp64, torch threads={torch.get_num_threads()}"},
        "e2e": {"value": mean_rate, "unit": "graphs/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="native", choices=["native", "reference"])
    ap.add_argument("--batch", type=int, default=PER_GPU_BATCH, help="graphs per GPU per step")
    ap.add_argument("--mode", default="tc", choices=["fp32", "tc", "tc1x"], help="arithmetic mode of the native kernels")
    ap.add_argument("--skip-cpu", action="store_true")
    ap.add_argument("--skip-e2e", action="store_true")
    ap.add_argument("--skip-extra", action="store_true", help="skip the short runs of the other BASELINE.json configs")
    ap.add_argument("--skip-strong", action="store_true", help="skip the strong-scaling block (16384 graphs global)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what the last timed train step and the last timed inference "
                    "step returned to the caller as DIR/<name>.npy (same arguments -> same inputs: compares two builds)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "native":
        ap.error("--dump-outputs applies to the native implementation")
    if args.warmup < 3:
        args.warmup = 3

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank)
        return

    import torch.distributed as dist
    from ms_hgnn import _native as N
    from ms_hgnn import morphology as M
    from ms_hgnn.lightning_py.gnnLightning import HGNN_K4_Lightning
    from ms_hgnn.synthetic import CONFIGS, HeteroBatch, make_batch
    from ms_hgnn.train import FusedTrainer

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (no CPU fallback); use --impl reference for the CPU arm")
    dev = torch.device("cuda", local_rank)
    torch.cuda.set_device(dev)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)
    assert world == args.gpus or world == 1, f"--gpus {args.gpus} but WORLD_SIZE={world}"

    cfg = CONFIGS[WORKLOAD]
    B = args.batch
    K, W = args.steps, args.warmup
    host = make_batch(cfg, B, seed=100 + rank).pin_memory()
    torch.manual_seed(2024)
    module = HGNN_K4_Lightning(128, 8, M.K4_MINI_CHEETAH.metadata, host, "adam", 1e-4, regression=False,
                               symmetry_mode="MorphSym", group_operator_path=M.cfg_path(cfg.group)).to(dev)
    module.model.validate_edges = "cached"
    module.model.set_mode(args.mode)
    trainer = FusedTrainer(module)
    resident = host.to(dev)
    h2d_bytes = sum(v.numel() * v.element_size() for v in host._x.values()) + \
        sum(v.numel() * v.element_size() for v in host._edge_index.values()) + host.y.numel() * host.y.element_size()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    def max_over_ranks(ms):
        if world == 1:
            return ms
        t = torch.tensor([ms], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def timed(fn, steps):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            fn()
        e1.record()
        barrier()
        return max_over_ranks(e0.elapsed_time(e1))

    # ---------------- train step, device resident ----------------
    for _ in range(W):
        trainer.train_step(resident)
    sampler = ClockSampler(local_rank) if rank == 0 else None
    last = {}

    def train_step():
        last["loss"] = trainer.train_step(resident)

    n0 = N.launch_count()
    train_ms = timed(train_step, K)
    launches = N.launch_count() - n0
    # after the last timed step its caller holds the returned loss and the parameters it updated in place (views of the flat
    # buffer); the flat gradient that update used is kept as well.  Copied now: the steps below change all three.
    dumped = {"train_loss": last["loss"].clone(), "train_params": trainer.model._flat.clone(),
              "train_grads": trainer.grads.clone()} if args.dump_outputs else None

    # ---------------- per-kernel times (same steps, events around every launch) ----------------
    N.profile_enable(True)
    prof_ms = timed(lambda: trainer.train_step(resident), K)
    prof = N.profile_read()
    N.profile_enable(False)

    # ---------------- inference, device resident ----------------
    for _ in range(W):
        trainer.infer(resident)

    def infer_step():
        last["infer"] = trainer.infer(resident)

    infer_ms = timed(infer_step, K)
    if dumped is not None:
        dumped["infer_out"] = last["infer"].clone()
    clocks = sampler.stop() if sampler else {}          # sampled across the three device-resident timed regions above

    # ---------------- strong scaling: BASELINE.json configs[2] as written = 16384 graphs GLOBAL over the N GPUs ----------------
    # Every rank trains PER_GPU_BATCH / N graphs per step (eager launches, and with the forward + loss + backward replayed from
    # one CUDA graph: at 2048 graphs per GPU the step is launch bound).  Efficiency = T(16384 on one GPU, no collective) /
    # (N x T(16384 / N per GPU, with the all-reduce)), both measured in THIS run on the same GPUs.
    strong = None
    if B == PER_GPU_BATCH and not args.skip_strong:
        trainer.skip_allreduce = True
        for _ in range(W):
            trainer.train_step(resident)
        t1_ms = timed(lambda: trainer.train_step(resident), K) / K        # one GPU's 16384-graph step without the collective
        trainer.skip_allreduce = False

        def small(bs):
            hb = make_batch(cfg, bs, seed=300 + rank).to(dev)
            for _ in range(W):
                trainer.train_step(hb)
            eager = timed(lambda: trainer.train_step(hb), K) / K
            for _ in range(W):
                trainer.train_step_graphed(hb)
            graphed = timed(lambda: trainer.train_step_graphed(hb), K) / K
            return eager, graphed

        if world > 1:
            bs = PER_GPU_BATCH // world
            eager, graphed = small(bs)
            best = min(eager, graphed)
            strong = {"global_batch": PER_GPU_BATCH, "per_gpu_batch": bs, "n_gpus": world, "ms_per_step": eager, "ms_per_step_cuda_graph": graphed,
                      "value": PER_GPU_BATCH / (best * 1e-3), "unit": "graphs/s", "single_gpu_ms_per_step": t1_ms,
                      "efficiency": t1_ms / (world * best), "efficiency_eager": t1_ms / (world * eager),
                      "note": "16384 graphs global; efficiency = T1 / (N x TN) with T1 = this run's 16384-graph step on one GPU without the collective"}
        else:
            # one GPU: what each rank of an N-GPU strong-scaling run computes (no collective here, so an upper bound on the
            # N-GPU efficiency; the N-GPU runs of this script report the measured one)
            rows = []
            for n in (2, 4, 8):
                eager, graphed = small(PER_GPU_BATCH // n)
                rows.append({"n_gpus_emulated": n, "per_gpu_batch": PER_GPU_BATCH // n, "ms_per_step": eager, "ms_per_step_cuda_graph": graphed,
                             "compute_efficiency_bound": t1_ms / (n * min(eager, graphed))})
            strong = {"global_batch": PER_GPU_BATCH, "n_gpus": 1, "single_gpu_ms_per_step": t1_ms, "efficiency": 1.0,
                      "per_rank_compute_at_n_gpus": rows,
                      "note": "per-rank compute of a 16384-graph global batch split over N GPUs, measured on this one GPU (no collective)"}

    # ---------------- end to end: pinned host buffers -> H2D -> train step -> D2H loss ----------------
    def e2e_leg(hb):
        """ms for K steps: per step the pinned host batch `hb` -> H2D on a copy stream (double-buffered) -> train step -> D2H loss."""
        copy_stream = torch.cuda.Stream(dev)
        bufs = [hb.to(dev), hb.to(dev)]
        ready = [torch.cuda.Event(), torch.cuda.Event()]
        done = [torch.cuda.Event(), torch.cuda.Event()]
        loss_host = torch.empty(K + W, dtype=torch.float32).pin_memory()

        def upload(i):
            b = bufs[i % 2]
            with torch.cuda.stream(copy_stream):
                copy_stream.wait_event(done[i % 2])          # the step that last read this buffer has finished
                for k, v in hb._x.items():
                    b._x[k].copy_(v, non_blocking=True)
                for k, v in hb._edge_index.items():
                    b._edge_index[k].copy_(v, non_blocking=True)
                b.y.copy_(hb.y, non_blocking=True)
                ready[i % 2].record(copy_stream)

        def e2e_loop(steps, base):
            upload(base)
            for i in range(base, base + steps):
                if i + 1 < base + steps:
                    upload(i + 1)
                torch.cuda.current_stream(dev).wait_event(ready[i % 2])
                loss = trainer.train_step(bufs[i % 2])
                done[i % 2].record(torch.cuda.current_stream(dev))
                loss_host[i:i + 1].copy_(loss, non_blocking=True)

        for e in done:
            e.record(torch.cuda.current_stream(dev))
        e2e_loop(W, 0)
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        e2e_loop(K, W)
        e1.record()
        barrier()
        return max_over_ranks(e0.elapsed_time(e1))

    e2e_ms = e2e_h_ms = None
    h2d_bytes_h = None
    if not args.skip_e2e:
        e2e_ms = e2e_leg(host)
        # the same leg with the node features stored as fp16 on the host (MSHGNN_F16, an input FORMAT: the kernels widen on load,
        # results stay fp32; labels and edge_index unchanged) - half the bytes over PCIe.  Not the credited `e2e`: extra key.
        host_h = type(host)({k: v.to(torch.float16) for k, v in host._x.items()}, dict(host._edge_index), host.y, host.batch_size).pin_memory()
        h2d_bytes_h = sum(v.numel() * v.element_size() for v in host_h._x.values()) + \
            sum(v.numel() * v.element_size() for v in host_h._edge_index.values()) + host_h.y.numel() * host_h.y.element_size()
        e2e_h_ms = e2e_leg(host_h)
        del host_h

    # ---------------- end to end through the device-side dataset (SURVEY 8f-3) ----------------
    # The raw sequence (what the reference keeps in host RAM as data.mat) is uploaded once; per step the host sends the
    # shuffled window indices, the window builder writes the collated batch in HBM, then the same train step runs.
    win_ms, win_info = None, None
    if not args.skip_e2e:
        import numpy as np
        from ms_hgnn.windows import DeviceSequence, WindowSpec
        n_rows = 1_000_000                                   # ~ the size of the Mini Cheetah contact dataset
        rng = np.random.default_rng(7 + rank)
        mat = {k: rng.standard_normal((n_rows, w), dtype=np.float32) for k, w in
               (("imu_acc", 3), ("imu_omega", 3), ("q", 12), ("qd", 12), ("p", 12), ("v", 12))}
        mat["contacts"] = (rng.random((n_rows, 4)) < 0.5).astype(np.float32)
        ds = DeviceSequence(mat, WindowSpec("heterogeneous_gnn_k4", 150, True), dev, torch.float32)
        idx_host = torch.from_numpy(rng.integers(0, len(ds), size=(K + W, B))).pin_memory()
        # double-buffered: the window builder of step i + 1 runs on a side stream while step i trains (same pattern as the
        # host-collated e2e leg above, with the H2D copy shrunk to the index vector)
        side = torch.cuda.Stream(dev)
        idx_dev = [torch.empty(B, dtype=torch.int64, device=dev) for _ in range(2)]
        wbufs = [ds.batch(idx_host[0]), ds.batch(idx_host[0])]
        w_ready = [torch.cuda.Event(), torch.cuda.Event()]
        w_done = [torch.cuda.Event(), torch.cuda.Event()]
        wloss = torch.empty(K + W, dtype=torch.float32).pin_memory()
        torch.cuda.synchronize(dev)

        def build(i):
            with torch.cuda.stream(side):
                side.wait_event(w_done[i % 2])               # the step that last read this buffer has finished
                idx_dev[i % 2].copy_(idx_host[i], non_blocking=True)
                ds.batch(idx_dev[i % 2], out=wbufs[i % 2])
                w_ready[i % 2].record(side)

        def win_loop(i0, i1):
            cur = torch.cuda.current_stream(dev)
            build(i0)
            for i in range(i0, i1):
                if i + 1 < i1:
                    build(i + 1)
                cur.wait_event(w_ready[i % 2])
                loss = trainer.train_step(wbufs[i % 2])
                w_done[i % 2].record(cur)
                wloss[i:i + 1].copy_(loss, non_blocking=True)

        for e in w_done:
            e.record(torch.cuda.current_stream(dev))
        win_loop(0, W)
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        win_loop(W, W + K)
        e1.record()
        barrier()
        win_ms = max_over_ranks(e0.elapsed_time(e1))
        N.profile_enable(True)
        ds.batch(idx_dev[0], out=wbufs[0])
        torch.cuda.synchronize(dev)
        wb_ms = N.profile_read().get("window_builder", (0.0, 1))[0]
        N.profile_enable(False)
        win_info = {"sequence_rows": n_rows, "sequence_bytes_resident": int(ds.seq.numel() * 4 + ds.labels.numel() * 4),
                    "window_builder_ms": wb_ms,
                    "window_builder_gbs": (150 * 54 * 4 + 43200 + 16) * B / (wb_ms * 1e-3) / 1e9 if wb_ms else None}

    # ---------------- the other BASELINE.json configs, briefly (rank 0, device resident; not the headline) ----------------
    extra = None
    if not args.skip_extra and world == 1 and B == PER_GPU_BATCH and args.mode == "tc":
        from ms_hgnn.synthetic import build_model
        extra = {}

        def quick(fn, steps=10, warm=3):
            for _ in range(warm):
                fn()
            torch.cuda.synchronize(dev)
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            for _ in range(steps):
                fn()
            b.record()
            torch.cuda.synchronize(dev)
            return a.elapsed_time(b) / steps

        # configs[1]: MS-HGNN C2 Mini Cheetah contact, batch 4096, train step
        c2 = CONFIGS["mini_cheetah-c2-contact"]
        m2 = build_model(c2, 128, 8, 1).set_mode(args.mode).to(dev)
        m2.validate_edges = "cached"
        b2 = make_batch(c2, 4096, seed=5).to(dev)
        t2 = FusedTrainer(m2, optimizer="adam", lr=1e-4, process_group=None)
        t2.world = 1
        ms = quick(lambda: t2.train_step(b2))
        extra["mini_cheetah-c2-contact_train_b4096"] = {"graphs_per_s": 4096 / (ms * 1e-3), "ms_per_step": ms}
        del m2, b2, t2
        # configs[4]: MS-HGNN K4 Solo12 COM, inference sweep
        c5 = CONFIGS["solo12-k4-com"]
        m5 = build_model(c5, 128, 8, 2).set_mode(args.mode).to(dev)
        m5.validate_edges = "cached"
        sweep = []
        for nb in (1 << 10, 1 << 14, 1 << 17, 1 << 20):
            b5 = make_batch(c5, nb, seed=6).to(dev)
            with torch.no_grad():
                ms = quick(lambda: m5(b5.x_dict, b5.edge_index_dict), steps=5 if nb >= (1 << 17) else 20)
            sweep.append({"graphs": nb, "graphs_per_s": nb / (ms * 1e-3), "ms": ms})
            del b5
        extra["solo12-k4-com_inference_sweep"] = sweep
        del m5
        torch.cuda.empty_cache()

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    if dumped is not None:
        dump_outputs(args.dump_outputs, dumped)

    # ---------------- roofline of the dominant kernel ----------------
    pk = peaks()
    per_kind = []
    for name, (ms, cnt) in prof.items():
        per_step_ms = ms / K
        flop = ALG.get(name)
        ent = {"kernel": name, "ms_per_step": per_step_ms, "launches_per_step": cnt / K, "share": ms / (prof_ms if prof_ms else 1)}
        if flop:
            ent["achieved_tflops"] = flop * B / (per_step_ms * 1e-3) / 1e12
            ent["frac_tensor_peak"] = ent["achieved_tflops"] / pk["tflops"]
        if name.startswith("encoder_fwd") or name.startswith("dw_encoder"):
            ent["achieved_gbs"] = ALG["in_bytes"] * B / (per_step_ms * 1e-3) / 1e9
            ent["frac_hbm_peak"] = ent["achieved_gbs"] / pk["hbm_gbs"]
        per_kind.append(ent)
    per_kind.sort(key=lambda e: -e["ms_per_step"])
    dom = next((e for e in per_kind if "achieved_tflops" in e), None)
    roofline = None
    traffic = recorded_traffic()
    if dom:
        t_dom = traffic.get(dom["kernel"], {}).get("dram_bytes_per_launch") if B == PER_GPU_BATCH and args.mode == "tc" else None
        ms_launch = dom["ms_per_step"] / max(dom["launches_per_step"], 1)
        roofline = {"kernel": dom["kernel"], "bound": "tensor", "achieved": dom["achieved_tflops"], "peak": pk["tflops"],
                    "unit": "TFLOP/s", "frac": dom["frac_tensor_peak"], "traffic": t_dom,
                    "traffic_view": None if not t_dom else {
                        "dram_gbs": t_dom / (ms_launch * 1e-3) / 1e9, "frac_hbm_peak": t_dom / (ms_launch * 1e-3) / 1e9 / pk["hbm_gbs"],
                        "note": "ncu DRAM bytes of this kernel's launch (profiles/" + TRAFFIC_FILE + ") / measured launch time.  The cross-layer "
                                "stack kernel keeps a row chunk's slabs in L2 between layers; what still reaches DRAM in a TRAINING launch is "
                                "what the other pass needs (forward: h_l written once per layer; backward: h_l / masks read, dc_l written for "
                                "the weight-gradient launch, dh_l of the residual chain written back although dead) - SURVEY 8d counts zero "
                                "mandatory bytes for the layer stack of an inference forward"},
                    "peak_source": pk["src"] + " (bf16 dense, sustained)",
                    "launches_per_step": dom["launches_per_step"], "ms_per_launch": dom["ms_per_step"] / max(dom["launches_per_step"], 1),
                    "note": "algorithmic FLOPs per SURVEY 8d (one MAC per product; the fp32-class mode issues 3 fp16 MMAs per product, "
                            "so tensor-pipe occupancy is ~3x this fraction)"}

    # ---------------- CPU baseline (oracle on host cores), bounded sample ----------------
    cpu = None
    if not args.skip_cpu and world == 1:
        cores = os.cpu_count()
        torch.set_num_threads(cores)
        r64, _ = oracle_train_rate(64, 40, 3)             # the reference's own batch size
        r1k, _ = oracle_train_rate(1024, 6, 1)
        best = max(r64, r1k)
        cpu = {"value": best, "unit": "graphs/s", "cores": torch.get_num_threads(), "kind": "port",
               "sample": f"oracle train step fp64: 40 steps of 64 graphs ({r64:.0f} graphs/s), 6 steps of 1024 graphs ({r1k:.0f} graphs/s); best reported"}

    total_graphs = B * world * K
    line = {
        "metric": METRIC, "value": total_graphs / (train_ms * 1e-3), "unit": "graphs/s", "n_gpus": world, "steps": K, "warmup": W,
        "ms_per_step": train_ms / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": {"fp32": "f32", "tc": "f16x2-split (f32 accumulate)", "tc1x": "f16 (f32 accumulate)"}[args.mode],
        "data": "synthetic",
        "config": {"workload": WORKLOAD, "per_gpu_batch": B, "global_batch": B * world, "hidden": 128, "layers": 8,
                   "parallelism": f"dp{world}", "mode": {"fp32": "fp32 SIMT FMA", "tc": "tcgen05 split-fp16 x3 (fp32-class accuracy): encoder, layers, dX, dW all on tensor cores", "tc1x": "tcgen05 fp16 x1"}[args.mode], "l2": "inputs (708 MB/step/GPU) exceed the 126 MB L2; no flush needed"},
        "inference": {"value": total_graphs / (infer_ms * 1e-3), "unit": "graphs/s", "ms_per_step": infer_ms / K},
        "strong": strong,
        "allreduce": None if world == 1 else {"overlapped": bool(trainer.overlap_allreduce), "skipped": bool(trainer.skip_allreduce),
                                              "note": "two buckets: layer-stack gradients on a side stream under the encoder weight gradient, encoder block at the end"},
        "e2e": None if e2e_ms is None else {"value": total_graphs / (e2e_ms * 1e-3), "unit": "graphs/s", "ms_per_step": e2e_ms / K,
                                            "h2d_bytes_per_step": h2d_bytes, "d2h_bytes_per_step": 4,
                                            "note": "pinned host batch -> H2D (copy stream, double-buffered) -> train step -> D2H loss"},
        "e2e_fp16_features": None if e2e_h_ms is None else {"value": total_graphs / (e2e_h_ms * 1e-3), "unit": "graphs/s", "ms_per_step": e2e_h_ms / K,
                                                             "h2d_bytes_per_step": h2d_bytes_h, "d2h_bytes_per_step": 4,
                                                             "note": "as e2e, host node features stored as fp16 (x_dtype MSHGNN_F16; lossy input format, arithmetic unchanged)"},
        "e2e_windowed": None if win_ms is None else dict(
            {"value": total_graphs / (win_ms * 1e-3), "unit": "graphs/s", "ms_per_step": win_ms / K, "h2d_bytes_per_step": B * 8,
             "d2h_bytes_per_step": 4,
             "note": "device-side dataset (ms_hgnn.windows, SURVEY 8f-3): raw sequence uploaded once, per step pinned shuffled window "
                     "indices -> H2D -> mshgnn_build_windows (z-score, URDF order, collate; side stream, double-buffered) -> train step -> D2H loss"}, **win_info),
        "gpu_launches": launches,
        "clocks": clocks,
        "roofline": roofline,
        "kernels": per_kind,
        "model_flops": {"train_mflop_per_graph": ALG["train_flop"] / 1e6, "fwd_mflop_per_graph": ALG["fwd_flop"] / 1e6,
                        "train_tflops": ALG["train_flop"] * B * world / (train_ms / K * 1e-3) / 1e12,
                        "infer_tflops": ALG["fwd_flop"] * B * world / (infer_ms / K * 1e-3) / 1e12},
        "cpu_baseline": cpu,
        "hbm_step": None if not (traffic.get("step") and B == PER_GPU_BATCH and args.mode == "tc") else {
            "dram_bytes_per_step": traffic["step"]["dram_bytes"], "achieved_gbs": traffic["step"]["dram_bytes"] / (train_ms / K * 1e-3) / 1e9,
            "peak_gbs": pk["hbm_gbs"], "frac": traffic["step"]["dram_bytes"] / (train_ms / K * 1e-3) / 1e9 / pk["hbm_gbs"],
            "source": "profiles/" + TRAFFIC_FILE + " (ncu DRAM counters of one step) / this run's step time"},
        "profiled_ms_per_step": prof_ms / K,
        "other_configs": extra,
    }
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
