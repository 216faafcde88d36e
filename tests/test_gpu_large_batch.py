"""Every graph of production-size batches against the fp64 oracle, at the batch sizes where the library's kernel selection changes.

The oracle runs on the GPU in chunks of graphs (helpers.oracle_run with ``device`` / ``chunk``; test_oracle_chunks.py ties it to the
pinned host oracle).  Bounds are those of test_gpu_parity.check_gradients: outputs and loss within 1e-4 norm-wise, every parameter
gradient and every x.grad within 1e-4 norm-wise under the ReLU sign pattern the native forward took (which may differ from the
oracle's own only at numerically ambiguous pre-activations), oracle gradients that are exactly zero exactly zero natively.  A norm
over tens of thousands of graphs dilutes one wrong row tile, so every row tile of 128 graphs of the outputs and of each x.grad tensor
is also held on its own to TILE_TOL.

The sizes are derived at run time from the selection rules (cited below) and the device's SM count.
"""
import time

import pytest
import torch

from helpers import (TOL_FP32, gradient_check_under_native_pattern, graph_slice, in_x_grad_dtype, oracle_model, oracle_outputs,
                     oracle_run, rel_err)
from ms_hgnn import _native as N
from ms_hgnn import morphology as M
from ms_hgnn.synthetic import CONFIGS, HeteroBatch, build_model

TILE = 128                   # graphs per row tile (TILE_M of the kernels)
TILE_TOL = 1e-3              # per row tile, relative; 10 x the norm-wise bound
PLAIN_GRAD_BOUND = 1e-1      # as test_gpu_parity: plain (unforced) error when a pre-activation flipped
ORACLE_CHUNK = 16384         # graphs per oracle chunk in training
INFER_CHUNK = 65536          # graphs per oracle chunk in inference

# selection rules of the library, restated
STACK_PAIR_MIN_GRAPHS = 6144                 # plan.cu ws_layout: CTA-pair stack kernel from this many graphs (STACK_PAIR_MIN_GRAPHS)
STACK_L2_CHUNK_BYTES = 84 * 1024 * 1024      # api.cu stack_rows_per_chunk: a chunk's slabs of one layer fit 84 MB of L2


def round_up(a, b):
    return (a + b - 1) // b * b


def padded_rows(B, pair):
    return round_up(B, 2 * TILE if pair else TILE)           # plan.cu ws_layout: Bp rounds to 256 for the CTA-pair kernel


def stack_chunk_row_tiles(S, pair):
    """api.cu stack_rows_per_chunk (clamped to 16..64 row tiles); the CTA-pair kernel walks rc / 2 pairs per chunk (launch_stack)."""
    rc = min(max(STACK_L2_CHUNK_BYTES // (2 * S * TILE * 128 * 4), 16), 64)
    return 2 * max(rc // 2, 1) if pair else rc


def encoder_tiles_per_item(B, n_enc, n_sm, pair):
    """api.cu launch_tc_encoder: two row tiles per item of k_tc_encoder_stream once L.count * ceil(n_row_tiles / 2) >= 4 * n_sm."""
    nt = padded_rows(B, pair) // TILE
    return 2 if n_enc * ((nt + 1) // 2) >= 4 * n_sm else 1


def plan_facts(nm, batch):
    """Plan of the native model (built by a one-graph forward): slots, live encoder slots, SM count."""
    one = graph_slice(batch, 0, 1)
    with torch.no_grad():
        nm(one.x_dict, one.edge_index_dict)
    d = nm._last_engine.plan.describe()
    return {"S": d["S"], "n_enc": sum(d["need"][0]), "n_sm": torch.cuda.get_device_properties(0).multi_processor_count}


def batch_size_for(rule, f):
    """Batch size of a named case, from the selection rules and the plan / device facts ``f``."""
    if isinstance(rule, int):
        return rule
    P = STACK_PAIR_MIN_GRAPHS
    if rule in ("pair_min-1", "pair_min", "pair_min+1"):
        return P + {"pair_min-1": -1, "pair_min": 0, "pair_min+1": 1}[rule]
    if rule == "second_chunk":
        # one-CTA kernel: the first graph of the second L2 chunk, so the last chunk is one row tile holding one graph
        B = stack_chunk_row_tiles(f["S"], False) * TILE + 1
        assert B < P, "the second chunk of the one-CTA kernel starts above the CTA-pair threshold"
        return B
    if rule == "pair_last_chunk_one_pair":
        # CTA-pair kernel: the last chunk is one row-tile pair, whose first tile holds one graph and whose second is empty
        per = stack_chunk_row_tiles(f["S"], True) * TILE
        k = -(-(P - 1) // per)
        return k * per + 1
    if rule in ("tpi1_last", "tpi2_first"):
        lo, hi = 1, 1 << 22                                                       # tpi(hi) == 2; monotone in B
        assert encoder_tiles_per_item(hi, f["n_enc"], f["n_sm"], True) == 2
        while hi - lo > 1:
            mid = (lo + hi) // 2
            if encoder_tiles_per_item(mid, f["n_enc"], f["n_sm"], mid >= P) == 2:
                hi = mid
            else:
                lo = mid
        return hi if rule == "tpi2_first" else lo
    raise ValueError(rule)


def selection(nm, B, mode, f, train=True):
    """What the library selects for this batch: CTA-pair kernel, padded rows, stack chunks, encoder tpi, weight-gradient splits."""
    eng = nm._last_engine
    tc = mode != "fp32"
    pair = tc and B >= STACK_PAIR_MIN_GRAPHS
    Bp = padded_rows(B, pair)
    _, _, bp = eng.plan.relu_mask_offset(B, eng.mode, -1)
    assert bp == Bp, f"padded rows {bp}, expected {Bp} from the selection rule (pair kernel {pair})"
    splits = sorted({ns for _, ns, _, _ in eng.plan.dw_layout(B, eng.mode)})
    rows = sorted({r for _, _, r, _ in eng.plan.dw_layout(B, eng.mode)})
    s = {"Bp": Bp, "dw_splits": splits, "dw_rows_per_split": rows} if train else {"Bp": Bp}
    if tc:
        ct = stack_chunk_row_tiles(f["S"], pair)
        nt = Bp // TILE
        s.update({"stack": "CTA-pair" if pair else "one-CTA", "stack_chunks": -(-nt // ct), "last_chunk_row_tiles": nt - (-(-nt // ct) - 1) * ct,
                  "encoder_tpi": encoder_tiles_per_item(B, f["n_enc"], f["n_sm"], pair), "last_tile_graphs": B - (B - 1) // TILE * TILE})
    return s


def device_batch(cfg, B, seed, device="cuda:0"):
    """Seeded synthetic batch built on the device, in make_batch's formats: z-scored 150-sample windows (Bessel std), the 900-wide
    IMU window tiled over the base nodes, zero COM base inputs, the constant A1 foot feature; labels of the config's loss."""
    tpl = M.TEMPLATES[cfg.template]
    gen = torch.Generator(device=device).manual_seed(1000 + seed)

    def windows(rows, w):
        x = torch.randn(rows, w, generator=gen, device=device)
        if cfg.zscore and w % 150 == 0:
            v = x.view(rows, w // 150, 150)
            x = ((v - v.mean(-1, keepdim=True)) / v.std(-1, keepdim=True)).reshape(rows, w)
        return x

    x = {}
    for t in tpl.node_types:
        n, w = tpl.nodes_per_graph[t], cfg.in_width[t]
        if t == "base" and w == 900:
            x[t] = windows(B, w).repeat_interleave(n, dim=0)
        elif t == "base" and cfg.model.startswith("COM"):
            x[t] = torch.zeros(B * n, w, device=device)
        elif t == "foot" and w == 1:
            x[t] = torch.ones(B * n, 1, device=device)
        else:
            x[t] = windows(B * n, w)
    if cfg.loss == "ce":
        y = (torch.rand(B * cfg.label_width, generator=gen, device=device) > 0.5).float()
    elif cfg.model.startswith("COM"):
        y = torch.randn(B, 6, generator=gen, device=device).repeat(1, tpl.nodes_per_graph["base"]).reshape(-1)
    else:
        y = torch.rand(B * cfg.label_width, generator=gen, device=device) * 70.0
    return HeteroBatch(x, tpl.edge_index_dict(B, device), y, B)


def tile_errors(a, b, B):
    """Relative error of every row tile of TILE graphs (a: native, b: oracle, both graph-major over B graphs), computed in fp64 where
    b lives.  A tile whose oracle values are all zero must be exactly zero (error inf otherwise)."""
    b = b.detach().double().reshape(B, -1)
    a = a.detach().to(b.device, torch.float64).reshape(B, -1)
    nt = -(-B // TILE)
    d = torch.zeros(nt * TILE, dtype=torch.float64, device=b.device)
    r = torch.zeros_like(d)
    d[:B] = (a - b).pow(2).sum(1)
    r[:B] = b.pow(2).sum(1)
    d, r = d.view(nt, TILE).sum(1), r.view(nt, TILE).sum(1)
    zero = r == 0
    e = (d / torch.where(zero, 1.0, r)).sqrt()
    return torch.where(zero & (d > 0), float("inf"), torch.where(zero, 0.0, e))


def worst_tile(tensors, B):
    """(worst tile error, tile index, tensor name) over {name: (native, oracle)}."""
    best = (0.0, -1, None)
    for k, (a, b) in tensors.items():
        e = tile_errors(a, b, B)
        i = int(e.argmax())
        if e[i].item() > best[0]:
            best = (e[i].item(), i, k)
    return best


def native_train_step(cfg, nm, batch):
    """Forward, native loss and backward through the module's autograd path, with x.requires_grad (as test_gpu_input_grad)."""
    x = {k: v.detach().requires_grad_() for k, v in batch.x_dict.items()}
    nm.zero_grad(set_to_none=True)
    out = nm(x, batch.edge_index_dict)
    eng = nm._last_engine
    C = eng.spec["out_channels"]
    loss, dout = eng.loss(out.detach().float().reshape(-1, C).contiguous(), batch.y, N.LOSS_CE2 if cfg.loss == "ce" else N.LOSS_MSE)
    out.backward(dout.view_as(out).to(out.dtype))
    grads = {n: (p.grad.clone() if p.grad is not None else torch.zeros_like(p)) for n, p in nm.named_parameters()}
    return out.detach(), loss.detach(), grads, {k: v.grad for k, v in x.items()}


def check_training_batch(cfg, nm, om, batch, mode, label, sel=None, t0=None):
    """Native training step of ``nm`` on ``batch`` against the chunked device oracle ``om``: the norm-wise, per-tile and exact-zero
    checks of this module.  Returns the measured numbers."""
    t0 = time.time() if t0 is None else t0
    B = batch.batch_size
    out_n, loss_n, g_n, dx_n = native_train_step(cfg, nm, batch)
    out_o, loss_o, g_o, dx_plain = oracle_run(cfg, om, batch, device=out_n.device, chunk=ORACLE_CHUNK, x_grad=True)
    e_out = rel_err(out_n, out_o)
    e_loss = abs(loss_n.item() - loss_o.item()) / abs(loss_o.item())
    ok, info = gradient_check_under_native_pattern(cfg, om, batch, nm, g_n, e_out, plain_grads=g_o, device=out_n.device,
                                                   chunk=ORACLE_CHUNK, native_dx=dx_n, plain_dx=dx_plain)
    dx_o = info.pop("forced_dx", None)
    tiles = {"out": (out_n, out_o)}
    if dx_o is not None:
        tiles.update({f"x.grad[{k}]": (dx_n[k], in_x_grad_dtype(dx_o[k], dx_n[k])) for k in dx_o})
    wt = worst_tile(tiles, B)
    torch.cuda.synchronize()
    res = {"B": B, "mode": mode, "out": e_out, "loss": e_loss, "grad": info.get("err"), "grad_tensor": info.get("tensor"),
           "x.grad": info.get("dx_err"), "x.grad_type": info.get("dx_type"), "plain_grad": info.get("plain_err"),
           "plain_x.grad": info.get("dx_plain_err"), "flips": info.get("flips"), "worst_tile": wt, "seconds": time.time() - t0}
    print(f"\nlarge batch [{label} {mode} B={B}] selection {sel}\n"
          f"  out {e_out:.2e}  loss {e_loss:.2e}  grad worst (native ReLU pattern) {res['grad']:.2e} [{res['grad_tensor']}]  "
          f"x.grad worst {res['x.grad']:.2e} [{res['x.grad_type']}]\n"
          f"  plain (unforced): grad {res['plain_grad']:.2e}  x.grad {res['plain_x.grad']:.2e}  flipped pre-activations {res['flips']}  "
          f"worst ReLU |x| / threshold {info.get('worst |x| / threshold', 0.0):.2f}\n"
          f"  worst row tile {wt[0]:.2e} (tile {wt[1]} of {-(-B // TILE)}, {wt[2]})  time {res['seconds']:.1f} s"
          if "error" not in info else f"\nlarge batch [{label} {mode} B={B}] selection {sel}: {info}")
    assert tuple(out_n.reshape(B, -1).shape) == tuple(out_o.reshape(B, -1).shape)
    assert e_out <= TOL_FP32 and e_loss <= TOL_FP32, res
    assert ok, info
    assert res["plain_grad"] <= (PLAIN_GRAD_BOUND if res["flips"] else TOL_FP32), res
    assert res["plain_x.grad"] <= (PLAIN_GRAD_BOUND if res["flips"] else TOL_FP32), res
    assert wt[0] <= TILE_TOL, res
    return res


def models(cfg):
    om = oracle_model(cfg, layers=8, seed=1)
    nm = build_model(cfg, layers=8, seed=2)
    nm.load_state_dict({k: v.float() for k, v in om.state_dict().items()})
    return om, nm


K4 = "mini_cheetah-k4-contact"
TRAIN_CASES = [
    (K4, "tc", "pair_min-1"), (K4, "tc", "pair_min"), (K4, "tc", "pair_min+1"),     # one-CTA / CTA-pair stack kernel; half-empty last pair
    (K4, "tc", "second_chunk"), (K4, "tc", "pair_last_chunk_one_pair"),             # chunked item order, one-tile / one-pair last chunk
    (K4, "tc", "tpi1_last"), (K4, "tc", "tpi2_first"),                              # k_tc_encoder_stream, one / two row tiles per item
    (K4, "tc", 16384), (K4, "fp32", 16384),                                         # bench.py's training batch
    (K4, "tc", 70001), (K4, "fp32", 70001),     # > 64 x 1024 graphs: tcgen05 splits of > 1024 rows, fp32 SIMT splits of > 512 rows
    ("mini_cheetah-c2-contact", "tc", 8193), ("a1-c2-grf", "tc", 16384), ("solo12-k4-com", "tc", 16384), ("mi-contact", "tc", 16384),
]


@pytest.mark.gpu
@pytest.mark.parametrize("name,mode,rule", TRAIN_CASES)
def test_training_batch_matches_oracle_on_every_graph(name, mode, rule):
    t0 = time.time()
    cfg = CONFIGS[name]
    om, nm = models(cfg)
    nm = nm.set_mode(mode).to("cuda:0")
    probe = device_batch(cfg, 1, seed=0)
    f = plan_facts(nm, probe)
    B = batch_size_for(rule, f)
    need = nm._last_engine.plan.workspace_bytes(B, True, nm._last_engine.mode)
    free, _ = torch.cuda.mem_get_info()
    assert need < free // 2, f"workspace of {need / 2**30:.1f} GiB for {B} graphs does not fit beside the oracle ({free / 2**30:.1f} GiB free)"
    batch = device_batch(cfg, B, seed=B)
    sel = selection(nm, B, mode, f)
    if rule in ("pair_min-1", "second_chunk"):
        assert sel["stack"] == "one-CTA"
    if rule in ("pair_min", "pair_min+1", "pair_last_chunk_one_pair"):
        assert sel["stack"] == "CTA-pair"
    if rule == "second_chunk":
        assert sel["stack_chunks"] == 2 and sel["last_chunk_row_tiles"] == 1 and sel["last_tile_graphs"] == 1
    if rule == "pair_last_chunk_one_pair":
        assert sel["last_chunk_row_tiles"] == 2 and sel["last_tile_graphs"] == 1 and sel["Bp"] - B == 2 * TILE - 1
    if rule in ("tpi1_last", "tpi2_first"):
        assert sel["encoder_tpi"] == (1 if rule == "tpi1_last" else 2)
    check_training_batch(cfg, nm, om, batch, mode, f"{name} {rule}", sel, t0)


@pytest.mark.gpu
def test_solo12_com_inference_of_2_20_graphs_matches_oracle_on_every_graph():
    """The 2^20-graph Solo12 K4 COM inference of bench.py's sweep, tensor-core mode: outputs of every graph against the oracle."""
    t0 = time.time()
    cfg = CONFIGS["solo12-k4-com"]
    B = 1 << 20
    om, nm = models(cfg)
    nm = nm.set_mode("tc").to("cuda:0")
    nm.validate_edges = "cached"
    batch = device_batch(cfg, B, seed=3)
    f = plan_facts(nm, batch)
    with torch.no_grad():
        out_n = nm(batch.x_dict, batch.edge_index_dict)
    sel = selection(nm, B, "tc", f, train=False)
    out_o = oracle_outputs(om, batch, device="cuda:0", chunk=INFER_CHUNK)
    e_out = rel_err(out_n, out_o)
    wt = worst_tile({"out": (out_n, out_o)}, B)
    torch.cuda.synchronize()
    print(f"\nlarge batch [solo12-k4-com inference tc B={B}] selection {sel}\n  out {e_out:.2e}  worst row tile {wt[0]:.2e} "
          f"(tile {wt[1]} of {B // TILE})  time {time.time() - t0:.1f} s")
    assert e_out <= TOL_FP32
    assert wt[0] <= TILE_TOL


def test_size_rules_give_the_intended_boundaries():
    """The derived sizes sit on the two sides of each rule (host arithmetic; 148 and 132 SMs as examples of a device)."""
    for n_sm in (148, 132):
        f = {"S": 20, "n_enc": 20, "n_sm": n_sm}
        lo, hi = batch_size_for("tpi1_last", f), batch_size_for("tpi2_first", f)
        assert hi == lo + 1
        assert encoder_tiles_per_item(lo, 20, n_sm, lo >= STACK_PAIR_MIN_GRAPHS) == 1
        assert encoder_tiles_per_item(hi, 20, n_sm, hi >= STACK_PAIR_MIN_GRAPHS) == 2
        B = batch_size_for("second_chunk", f)
        assert (B - 1) % TILE == 0 and (B - 1) // TILE == stack_chunk_row_tiles(20, False)
        B = batch_size_for("pair_last_chunk_one_pair", f)
        per = stack_chunk_row_tiles(20, True) * TILE
        assert B >= STACK_PAIR_MIN_GRAPHS and (B - 1) % per == 0 and padded_rows(B, True) - (B - 1) == 2 * TILE


def test_per_tile_check_finds_what_the_norm_misses():
    """One wrong last row tile among 70001 graphs (547 tiles): a 2e-3 relative error there is below the 1e-4 norm-wise bound over the
    batch, and the per-tile check reports it with its index."""
    gen = torch.Generator().manual_seed(0)
    B = 70001
    ref = torch.randn(B * 4, 2, generator=gen, dtype=torch.float64)
    out = ref * (1 + 1e-7 * torch.randn(ref.shape, generator=gen, dtype=torch.float64))
    first = (B - 1) // TILE * TILE                                   # first graph of the last (short) tile
    out.view(B, -1)[first:] *= 1 + 2e-3
    assert rel_err(out, ref) <= TOL_FP32
    e, i, name = worst_tile({"out": (out, ref)}, B)
    assert e > TILE_TOL and i == (B - 1) // TILE and name == "out"
    # a tile whose reference is exactly zero must be exactly zero
    z = torch.zeros(300, 3, dtype=torch.float64)
    bad = z.clone(); bad[299, 0] = 1e-30
    assert tile_errors(z, z, 300).max().item() == 0.0
    assert tile_errors(bad, z, 300)[2].item() == float("inf")
