"""Worker of tests/test_gpu_hidden_width.py::test_nccl_reduced_gradients_at_width_10 (one process per GPU, launched with
torch.distributed.run): a width-10 model's NCCL-reduced flat gradient of the sharded batch equals the single-rank gradient of
the whole batch, and the overlapped all-reduce (started at layers_ready, in the model's own parameter layout) equals the plain one."""
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (os.path.join(ROOT, "morphsym-hgnn_b200"), os.path.join(ROOT, "oracle"), os.path.join(ROOT, "tests")):
    sys.path.insert(0, p)

import torch  # noqa: E402
import torch.distributed as dist  # noqa: E402

from ms_hgnn.synthetic import CONFIGS, build_model, make_batch  # noqa: E402
from ms_hgnn.train import FusedTrainer  # noqa: E402


def main():
    rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
    dev = torch.device("cuda", local)
    torch.cuda.set_device(dev)
    dist.init_process_group("nccl", device_id=dev)
    cfg = CONFIGS["mini_cheetah-k4-contact"]
    full = make_batch(cfg, 256 * world, seed=5)
    out = {"rank": rank, "world": world}
    for mode in ("tc", "fp32"):
        nm = build_model(cfg, hidden=10, layers=8, seed=10).set_mode(mode).to(dev)
        nm.validate_edges = "cached"
        tr = FusedTrainer(nm, optimizer="sgd", lr=0.0)
        shard = full.shard(rank, world).to(dev)
        tr.overlap_allreduce = True
        tr.train_step(shard)
        g_overlap = tr.grads.clone()
        tr.overlap_allreduce = False
        tr.train_step(shard)
        out[f"{mode}_overlap_equals_plain"] = bool(torch.equal(g_overlap, tr.grads))
        solo = FusedTrainer(nm, optimizer="sgd", lr=0.0, process_group=None)
        solo.world = 1
        solo._synced_params = True
        solo.train_step(full.to(dev))
        out[f"{mode}_err"] = ((g_overlap.double() - solo.grads.double()).norm() / solo.grads.double().norm()).item()
    gathered = [None] * world
    dist.all_gather_object(gathered, out)
    if rank == 0:
        print("DPRESULT " + json.dumps(gathered), flush=True)
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
