"""Shared helpers of the parity tests: the oracle is the checker, the native path the thing checked."""
import contextlib

import torch

import mshgnn_oracle as O
from ms_hgnn.synthetic import CONFIGS, build_model, make_batch

TOL_FP32 = 1e-4      # north_star: within 1e-4 relative (norm-wise, per tensor) in fp32 against the fp64 oracle


def in_x_grad_dtype(ref: torch.Tensor, native: torch.Tensor) -> torch.Tensor:
    """The oracle's input gradient as the native path delivers it: the x.grad of fp16 features is the fp32 input gradient
    rounded to fp16 (test_gpu_input_grad.test_float64_and_float16_features), so it is compared with the oracle's rounded the
    same way; every other dtype is compared with the oracle's fp64 values."""
    return ref.half() if native.dtype == torch.float16 else ref


def rel_err(a: torch.Tensor, b: torch.Tensor) -> float:
    """||a - b|| / ||b|| in fp64 (||a - b|| when b is zero), computed where b lives."""
    b = b.detach().double().flatten(); a = a.detach().to(b.device, torch.float64).flatten()
    nb = b.norm().item()
    if nb == 0.0:
        return (a - b).norm().item()
    return ((a - b).norm() / nb).item()


def oracle_model(cfg, hidden=128, layers=8, seed=0):
    """fp64 oracle whose weights are exactly representable in fp32 (so both sides see the same numbers)."""
    prev = torch.get_default_dtype()
    torch.set_default_dtype(torch.float64)
    try:
        m = build_model(cfg, hidden, layers, seed, module=O)
        with torch.no_grad():
            for p in m.parameters():
                p.copy_(p.float().double())
    finally:
        torch.set_default_dtype(prev)
    return m


def oracle_loss(cfg, out, y, B):
    if cfg.loss == "ce":
        return O.contact_ce_loss_exact(out.reshape(B, 8), y.reshape(B, 4))
    return O.mse_loss(out.reshape(B, -1), y.reshape(B, -1))


def graph_slice(batch, g0, g1, device=None):
    """Graphs [g0, g1) of a collated batch, as a batch of g1 - g0 graphs (optionally moved to ``device``).  Every node tensor is
    graph-major and every edge_index is the template tiled from offset 0, so the first (g1 - g0) graphs' edges serve any slice."""
    from ms_hgnn.synthetic import HeteroBatch
    B, nb = batch.batch_size, g1 - g0
    x = {k: v[g0 * (v.shape[0] // B):g1 * (v.shape[0] // B)] for k, v in batch.x_dict.items()}
    ei = {k: v[:, :(v.shape[1] // B) * nb] for k, v in batch.edge_index_dict.items()}
    w = batch.y.numel() // B
    out = HeteroBatch(x, ei, batch.y.reshape(-1)[g0 * w:g1 * w], nb)
    return out.to(device) if device is not None else out


def graph_chunks(B, chunk):
    """[g0, g1) ranges of at most ``chunk`` graphs covering B graphs (one range when chunk is None)."""
    step = B if not chunk else int(chunk)
    return [(g0, min(g0 + step, B)) for g0 in range(0, B, step)]


def slice_forced(forced, rows_per_graph, g0, g1, device="cpu"):
    """The part of a forced ReLU pattern ({call i: (flat index into [B * n_i, 128], values)}) that falls in graphs [g0, g1),
    re-indexed to the chunk's own [(g1 - g0) * n_i, 128] tensor and moved to ``device`` (ReluTap writes it into the mask there)."""
    out = {}
    for i, (idx, val) in forced.items():
        per = rows_per_graph[i] * 128
        keep = (idx >= g0 * per) & (idx < g1 * per)
        if keep.any():
            out[i] = ((idx[keep] - g0 * per).to(device), val[keep].to(device))
    return out


def _oracle_pass(cfg, model, batch, forced=None, device="cpu", chunk=None, x_grad=False):
    """fp64 forward + loss + backward of the oracle, on ``device``, in chunks of at most ``chunk`` graphs.

    Graphs are independent and the loss is a mean, so a chunk of n_c graphs contributes (n_c / B) x its own mean loss: parameter
    gradients accumulate those weighted chunk gradients in fp64, the input gradient of a chunk's rows is its weighted chunk
    gradient, and the outputs are the chunks' outputs concatenated.  One chunk (the default) is the plain whole-batch run.
    ``forced`` ({ReLU call: (flat index, value)} over the whole batch) is sliced to each chunk's graphs."""
    device = torch.device(device)
    if next(model.parameters()).device != device:
        import copy
        model = copy.deepcopy(model).to(device)
    B = batch.batch_size
    rows_per_graph = None
    if forced:
        with torch.no_grad(), O.ReluTap(record=True) as tap:       # which node type (rows per graph) each ReLU call runs on
            one = graph_slice(batch, 0, 1, device)
            model({k: v.double() for k, v in one.x_dict.items()}, one.edge_index_dict)
        rows_per_graph = [p.shape[0] for p in tap.pre]
    model.zero_grad()
    outs, dx, loss = [], {k: [] for k in batch.x_dict}, torch.zeros((), dtype=torch.float64, device=device)
    for g0, g1 in graph_chunks(B, chunk):
        part = graph_slice(batch, g0, g1, device)
        x = {k: v.double().detach().requires_grad_(x_grad) for k, v in part.x_dict.items()}
        f = slice_forced(forced, rows_per_graph, g0, g1, device) if forced else None
        with O.ReluTap(forced=f) if f is not None else contextlib.nullcontext():
            out = model(dict(x), part.edge_index_dict)
            l_c = oracle_loss(cfg, out, part.y.double(), g1 - g0)
            if g1 - g0 != B:
                l_c = l_c * ((g1 - g0) / B)
            l_c.backward()
        outs.append(out.detach())
        loss = loss + l_c.detach()
        for k, v in x.items():
            dx[k].append(v.grad if v.grad is not None else torch.zeros_like(v))
    grads = {n: (p.grad.clone() if p.grad is not None else torch.zeros_like(p)) for n, p in model.named_parameters()}
    return torch.cat(outs), loss, grads, ({k: torch.cat(v) for k, v in dx.items()} if x_grad else None)


def oracle_run(cfg, model, batch, device="cpu", chunk=None, x_grad=False):
    """fp64 forward + loss + backward of the oracle; returns out, loss, {name: grad} (and {type: x.grad} when x_grad).
    Runs on the host in one piece by default; on ``device`` in chunks of ``chunk`` graphs otherwise (_oracle_pass)."""
    out, loss, grads, dx = _oracle_pass(cfg, model, batch, None, device, chunk, x_grad)
    return (out, loss, grads, dx) if x_grad else (out, loss, grads)


def oracle_outputs(model, batch, device="cpu", chunk=None):
    """fp64 forward only (inference), on ``device`` in chunks of ``chunk`` graphs; the chunks' outputs concatenated."""
    device = torch.device(device)
    if next(model.parameters()).device != device:
        import copy
        model = copy.deepcopy(model).to(device)
    outs = []
    with torch.no_grad():
        for g0, g1 in graph_chunks(batch.batch_size, chunk):
            part = graph_slice(batch, g0, g1, device)
            outs.append(model({k: v.double() for k, v in part.x_dict.items()}, part.edge_index_dict))
    return torch.cat(outs)


def oracle_fp32_floor(cfg, model, batch, ref_out, ref_grads):
    """Error of the SAME oracle op sequence run in plain PyTorch float32 against its float64 self.

    ReLU makes the gradient discontinuous in the forward numerics: an fp32 rounding that flips the sign
    of one pre-activation changes a whole gradient row.  No fp32 implementation (including the
    reference's own ops in fp32) can be closer to the fp64 oracle than this floor, so the parity bound
    for gradients is max(1e-4, 2 x floor) per tensor."""
    import copy
    m32 = copy.deepcopy(model).float()
    x = {k: v.float() for k, v in batch.x_dict.items()}
    m32.zero_grad()
    out = m32(x, batch.edge_index_dict)
    loss = oracle_loss(cfg, out, batch.y.float(), batch.batch_size)
    loss.backward()
    floor = {n: (rel_err(p.grad, ref_grads[n]) if p.grad is not None else 0.0) for n, p in m32.named_parameters()}
    return rel_err(out, ref_out), floor


# ------------------------------------------------------------------------------------------------
# oracle backward under a forced ReLU sign pattern
# ------------------------------------------------------------------------------------------------
def oracle_grads_with_forced(cfg, model, batch, forced, device="cpu", chunk=None, x_grad=False):
    """{name: grad} of the oracle under a forced ReLU sign pattern (and {type: x.grad} when x_grad); device / chunk as oracle_run."""
    _, _, grads, dx = _oracle_pass(cfg, model, batch, forced, device, chunk, x_grad)
    return (grads, dx) if x_grad else grads


# ------------------------------------------------------------------------------------------------
# Gradient comparison under the ReLU sign pattern the native forward actually took
# ------------------------------------------------------------------------------------------------
def native_relu_pattern(model, B, device="cpu"):
    """{oracle tap tag: (BoolTensor [B * nodes_of_type, 128], live BoolTensor [B * nodes_of_type])} read back from the native
    training workspace (mshgnn_relu_mask_offset) and the plan's liveness table, rows re-ordered to the oracle's graph-major layout.
    The bits are expanded on the workspace's device one layer at a time and the result is left on ``device``."""
    eng = next(iter(model._engines.values()))
    spec, plan = eng.spec, eng.plan
    types, npg = spec["node_types"], spec["nodes_per_graph"]
    base = [sum(npg[:i]) for i in range(len(types))]
    S = sum(npg)
    need = plan.describe()["need"]                       # need[l][slot], l = 0..L
    torch.cuda.synchronize()
    ws = eng._ws
    shifts = torch.arange(32, device=ws.device, dtype=torch.int32)

    def read(layer):                                     # -> [slot][graph][channel] bool, on the workspace's device
        off, ns, bp = plan.relu_mask_offset(B, eng.mode, layer)
        words = ws[off:off + ns * bp * 16].view(torch.int32).view(ns, bp, 4)[:, :B]
        return ((words.unsqueeze(-1) >> shifts) & 1).bool().reshape(ns, B, 128)

    def rows_of(bits, first_slot, n):                    # -> [B * n, 128], row = graph * n + local node
        return bits[first_slot:first_slot + n].permute(1, 0, 2).reshape(B * n, 128).to(device)

    def live_of(l, first_slot, n):                       # [B * n] bool
        return torch.tensor([bool(need[l][first_slot + j]) for j in range(n)], device=device).repeat(B)

    out = {}
    enc = read(-1)
    for t, name in enumerate(types):
        out[("enc", name)] = (rows_of(enc, base[t], npg[t]), live_of(0, base[t], npg[t]))
    del enc
    mlp_t = spec["mlp_type"]
    for l in range(spec["num_layers"]):
        bits = read(l)
        for t, name in enumerate(types):
            if spec["morph_sym"] and t == mlp_t:
                out[("mlp", l, name)] = (rows_of(bits, S, npg[t]), live_of(l + 1, base[t], npg[t]))
            else:
                out[("conv", l, name)] = (rows_of(bits, base[t], npg[t]), live_of(l + 1, base[t], npg[t]))
        del bits
    return out


def forced_native_pattern(model, batch, pattern, fwd_rel_err, device="cpu", chunk=None):
    """The native forward's ReLU signs (``pattern``, from native_relu_pattern) where they differ from the oracle's own, in the
    form O.ReluTap(forced=...) takes.  Returns (forced, flips, worst ratio, error or None): the ratio is the largest |x| among
    the differing pre-activations over 16 * max(forward error, 1e-7) * rms(x) of that ReLU call, so <= 1 means every difference
    is numerically ambiguous.  The oracle's pre-activations are recorded chunk by chunk on ``device``."""
    device = torch.device(device)
    if next(model.parameters()).device != device:
        import copy
        model = copy.deepcopy(model).to(device)
    B = batch.batch_size
    sumsq, count, worst_abs, idx_parts, val_parts, tags = {}, {}, {}, {}, {}, {}
    for g0, g1 in graph_chunks(B, chunk):
        part = graph_slice(batch, g0, g1, device)
        with torch.no_grad(), O.ReluTap(record=True) as tap:
            model({k: v.double() for k, v in part.x_dict.items()}, part.edge_index_dict)
        for i, (pre, tag) in enumerate(zip(tap.pre, tap.tags)):
            if tag not in pattern:
                return None, 0, 0.0, f"no native pattern for oracle ReLU {tag}"
            bits, live = pattern[tag]
            n = pre.shape[0] // (g1 - g0)
            if tuple(bits.shape) != (B * n, pre.shape[1]):
                return None, 0, 0.0, f"shape mismatch at {tag}: {tuple(bits.shape)} vs {(B * n, pre.shape[1])}"
            tags[i] = tag
            v = pre.detach()
            sumsq[i] = sumsq.get(i, 0.0) + v.pow(2).sum().item()
            count[i] = count.get(i, 0) + v.numel()
            diff = ((v > 0) != bits[g0 * n:g1 * n].to(v.device)) & live[g0 * n:g1 * n].to(v.device)[:, None]
            if diff.any():
                worst_abs[i] = max(worst_abs.get(i, 0.0), v.abs()[diff].max().item())
                idx = torch.nonzero(diff.reshape(-1)).reshape(-1)
                idx_parts.setdefault(i, []).append(idx + g0 * n * v.shape[1])
                val_parts.setdefault(i, []).append(bits[g0 * n:g1 * n].reshape(-1).to(v.device)[idx])
    forced, flips, worst_ratio = {}, 0, 0.0
    for i in idx_parts:
        thr = 16.0 * max(fwd_rel_err, 1e-7) * (sumsq[i] / count[i]) ** 0.5
        worst_ratio = max(worst_ratio, (worst_abs[i] / thr) if thr > 0 else float("inf"))
        forced[i] = (torch.cat(idx_parts[i]), torch.cat(val_parts[i]))
        flips += int(forced[i][0].numel())
    return forced, flips, worst_ratio, None


def gradient_check_under_native_pattern(cfg, model, batch, native_model, native_grads, fwd_rel_err, tol=TOL_FP32, plain_grads=None,
                                        device="cpu", chunk=None, native_dx=None, plain_dx=None):
    """Returns (ok, info).  ReLU makes d(loss)/d(params) discontinuous in the forward numerics: an implementation whose
    forward is accurate to 1e-6 may put a pre-activation of +-1e-7 on the other side of zero, which moves whole gradient
    tensors by 1e-4..1e-2 (plain PyTorch fp32 does the same against fp64).  So the native gradient is compared, strictly
    (``tol`` per tensor, norm-wise), with the oracle's fp64 gradient under the sign pattern the native forward took, after
    checking that this pattern differs from the oracle's own ONLY at numerically ambiguous pre-activations:
    |x| < 16 * max(forward error, 1e-7) * rms(x).

    ``device`` / ``chunk``: where and in how many graphs at a time the oracle runs (oracle_run).  ``native_dx`` ({type: x.grad}):
    the input gradients are held to the same bound under the same pattern; the oracle's are then returned as info["forced_dx"]."""
    names = [n for n, _ in model.named_parameters()]
    B = batch.batch_size
    pattern = native_relu_pattern(native_model, B, device)
    forced, flips, worst_ratio, error = forced_native_pattern(model, batch, pattern, fwd_rel_err, device, chunk)
    del pattern
    if error is not None:
        return False, {"error": error}
    if worst_ratio > 1.0:
        return False, {"error": "native ReLU pattern differs from the oracle at a NON-ambiguous pre-activation",
                       "worst |x| / threshold": worst_ratio, "flips": flips}
    g, dx = oracle_grads_with_forced(cfg, model, batch, forced, device, chunk, x_grad=True)
    worst, worst_name = 0.0, None
    for n in names:
        if g[n].norm().item() == 0.0:
            if native_grads[n].abs().max().item() != 0.0:
                return False, {"error": f"{n}: oracle gradient is exactly zero, native is not"}
            continue
        e = rel_err(native_grads[n], g[n])
        if e > worst:
            worst, worst_name = e, n
    info = {"flips": flips, "err": worst, "tensor": worst_name, "worst |x| / threshold": worst_ratio}
    if plain_grads is not None:
        # the PLAIN error too (oracle's own ReLU pattern, nothing forced): reported next to the forced one so that the
        # size of the sign-flip effect is visible; it equals the forced error when no pre-activation flipped
        pw, pn = 0.0, None
        for n in names:
            if plain_grads[n].norm().item() == 0.0:
                continue
            e = rel_err(native_grads[n], plain_grads[n])
            if e > pw:
                pw, pn = e, n
        info["plain_err"], info["plain_tensor"] = pw, pn
    ok = worst <= tol
    if native_dx is not None:
        dw, dn, dp = 0.0, None, 0.0
        for k in dx:
            if dx[k].norm().item() == 0.0:
                if native_dx[k].abs().max().item() != 0.0:
                    return False, {"error": f"x.grad[{k}]: oracle gradient is exactly zero, native is not"}
                continue
            e = rel_err(native_dx[k], in_x_grad_dtype(dx[k], native_dx[k]))
            if e > dw:
                dw, dn = e, k
            if plain_dx is not None:
                dp = max(dp, rel_err(native_dx[k], in_x_grad_dtype(plain_dx[k], native_dx[k])))
        info["dx_err"], info["dx_type"], info["forced_dx"] = dw, dn, dx
        if plain_dx is not None:
            info["dx_plain_err"] = dp
        ok = ok and dw <= tol
    return ok, info
