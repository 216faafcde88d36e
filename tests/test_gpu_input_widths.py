"""Oracle parity at the input widths and depths a user can reach, beyond the BASELINE shapes.

The library takes any input width K >= 1 per node type and 1..15 layers; the BASELINE datasets only give K = 900 / 450 / 300 / 6 /
3 / 2 / 1 at 1..8 layers.  Other history lengths of the window builder (ms_hgnn.windows.WindowSpec) give other widths, and the
encoder kernels depend on K in several places: the persistent encoder's 64-column TMA box (wider than the row at K < 64), the
192-column units and 64-column blocks of the encoder weight gradient, the vector width of the register-staged loads (parity of K,
node offset and base pointer), the input gradient's tensor-map store (32-column box) and the zero-padded encoder weight image
[n_types * 128][enc_kmax], which a narrow type shares with its widest sibling.

Every case is a training step on random features of every node type (make_batch / device_batch give the COM models all-zero base
features, which leaves that encoder's weight gradient exactly zero) checked against the chunked fp64 oracle with
test_gpu_large_batch.check_training_batch: outputs and loss within 1e-4 norm-wise, every row tile within 1e-3, every parameter
gradient and every x.grad within 1e-4 under the native ReLU pattern.  In tensor-core mode every encoder variant must give the same
bits, and a profiler trace of each variant's step shows which encoder kernels ran; the selection rule they must match is restated
below (expected_kernels) and checked on the host over the whole width grid.
"""
import dataclasses
import re
import time

import pytest
import torch

from helpers import native_relu_pattern, oracle_model
from ms_hgnn import _native as N
from ms_hgnn import morphology as M
from ms_hgnn.engine import build_spec
from ms_hgnn.synthetic import CONFIGS, HeteroBatch, build_model
from test_gpu_large_batch import STACK_PAIR_MIN_GRAPHS, check_training_batch, native_train_step, plan_facts, selection

B = 300                      # three row tiles of 128 graphs: a partial last tile, a half-empty last row-tile pair
MI, K4C, C2C = "mi-grf", "solo12-k4-com", "solo-c2-com"

# (config, widths in the config's node-type order).  MI-HGNN (GRF_HGNN) has three free widths; the COM models two, the K4 joint
# width carrying a +-1 sign table.  Every width of the window builder at history lengths 1 / 2 / 3 / 8 is here (window_widths());
# the A1 and Mini Cheetah ones run on MI-HGNN, since the K4 / C2 GRF models fix the history at 150 steps (hgnn_k4.py, hgnn_c2.py).
WIDTH_CASES = [
    (MI, (6, 2, 6)), (MI, (12, 4, 12)), (MI, (18, 6, 18)), (MI, (48, 16, 48)),      # Mini Cheetah MI-HGNN at h = 1 / 2 / 3 / 8
    (MI, (1, 3, 5)), (MI, (7, 8, 60)), (MI, (63, 64, 65)), (MI, (68, 127, 128)),
    (MI, (129, 191, 192)), (MI, (193, 196, 256)), (MI, (257, 388, 9)),
    (MI, (4, 1988, 24)),     # K = 4 beside K = 1988 = 4 + 31 x 64: the weight image is 2048 columns wide for both
    (MI, (1999, 4, 2)),      # the same image with an odd wide type (register-staged loads, one-item-per-CTA encoder)
    (K4C, (12, 4)), (K4C, (18, 6)), (K4C, (48, 16)),                                # Solo12 K4 COM at h = 2 / 3 / 8
    (K4C, (1988, 4)), (K4C, (192, 8)),
    (C2C, (193, 12)),
]
REQUIRED_WIDTHS = set(range(1, 9)) | {12, 60, 63, 64, 65, 68, 127, 128, 129, 191, 192, 193, 196, 256, 257, 388}

# encoder run-time options (encoder, encoder_tpi, encoder_dw_tma); the library's default first
DEFAULT = (-1, 0, -1)
VARIANTS = [DEFAULT, (0, 1, 0), (0, 2, 0), (1, 0, 0), (2, 0, 0), (0, 0, 1)]


def cfg_with(name, widths):
    cfg = CONFIGS[name]
    w = dict(zip(cfg.in_width, widths))
    return dataclasses.replace(cfg, name=f"{name} " + "/".join(str(v) for v in widths), in_width=w)


def case_id(c):
    return f"{c[0]}-" + "-".join(str(v) for v in c[1])


def window_widths():
    """Every input width the window builder gives at history lengths 1, 2, 3 and 8."""
    from ms_hgnn import windows as W
    out = set()
    for h in (1, 2, 3, 8):
        specs = [W.WindowSpec(mt, h, normalize=False) for mt in W._MODEL_TYPES]
        specs += [W.WindowSpec(mt, h, normalize=False, dataset="solo12") for mt in W._SOLO_MODEL_TYPES]
        specs.append(W.WindowSpec("heterogeneous_gnn_c2", h, normalize=False, dataset="a1"))
        for s in specs:
            out |= set(s.widths.values())
    return out


# ---- the library's encoder kernel selection, restated ----------------------------------------------------------------------
ENQ_MAX_SLOTS = 32           # kernels_enc.cuh: node slots the persistent encoder's slot table holds


def rows_ok(K, misalign=0):
    """kernels_enc.cuh enq_rows_ok: fp32 rows of a 16-byte multiple on a 16-byte aligned base.  (Its sign-offset condition always
    holds: plan.cu pads every slot's sign vector to a multiple of 4.)"""
    return misalign % 16 == 0 and K % 4 == 0 and K >= 4


def expected_kernels(widths, live, mode, variant=DEFAULT, x_dtype=torch.float32, misalign=0, n_models=1):
    """Encoder kernels of a training step.  widths {type: K}; live {type: encoder slots live at layer 0 (plan need[0])};
    misalign: byte offset of every feature tensor's base pointer modulo 16.

      forward      (api.cu launch_tc_encoder): a model batch takes k_tc_encoder_pair; option encoder 1 / 2 takes k_tc_encoder /
                   k_tc_encoder_pair; otherwise k_tc_encoder_stream when every live type is fp32 with rows_ok and at most
                   ENQ_MAX_SLOTS slots are live, else k_tc_encoder_pair;
      weight grad  (api.cu launch_tc_encoder_dw): k_tc_encoder_dw<true> (x rows by TMA) only with option encoder_dw_tma 1, one
                   model, fp32 features and rows_ok for every live type; k_tc_encoder_dw<false> otherwise;
      input grad   (api.cu mshgnn_input_grad): k_tc_encoder_dx, storing through a tensor map for the types whose (freshly
                   allocated, so aligned) x.grad rows are rows_ok; fp32 mode: k_encoder_dx.
    The fp32 (SIMT) mode runs the encoder forward and weight gradient in the row-GEMM kernels it uses for every layer."""
    if mode == "fp32":
        return {"fwd": None, "dw": None, "dx": "k_encoder_dx", "dx_tma": []}
    enc = variant[0]
    used = [t for t in widths if live[t]]
    f32 = x_dtype == torch.float32
    stream_ok = f32 and sum(live.values()) <= ENQ_MAX_SLOTS and all(rows_ok(widths[t], misalign) for t in used)
    which = 2 if n_models > 1 else (enc if enc >= 0 else 0)
    fwd = "k_tc_encoder" if which == 1 else ("k_tc_encoder_pair" if which == 2 or not stream_ok else "k_tc_encoder_stream")
    xt = f32 and n_models == 1 and variant[2] > 0 and all(rows_ok(widths[t], misalign) for t in used)
    return {"fwd": fwd, "dw": f"k_tc_encoder_dw<{'true' if xt else 'false'}>", "dx": "k_tc_encoder_dx",
            "dx_tma": [t for t in widths if rows_ok(widths[t])]}


ENCODER_FWD = {"k_tc_encoder", "k_tc_encoder_pair", "k_tc_encoder_stream"}
ENCODER_DW = {"k_tc_encoder_dw<true>", "k_tc_encoder_dw<false>"}


def live_slots(plan, spec):
    need0 = plan.describe()["need"][0]
    out, first = {}, 0
    for t, n in zip(spec["node_types"], spec["nodes_per_graph"]):
        out[t] = sum(need0[first:first + n])
        first += n
    return out


def host_plan(cfg, layers=8):
    """The native plan of cfg's model, built on the host (the liveness it needs does not depend on the sign tables)."""
    tpl = M.TEMPLATES[cfg.template]
    morph = cfg.group is not None
    com = cfg.model.startswith("COM")
    spec = build_spec(tpl.node_types, tpl.nodes_per_graph, cfg.in_width, tpl.edge_types, tpl.edges, ("gt", "gs", "center_bb"), 128,
                      layers, morph, "base" if morph else None, "base" if com else "foot", 6 if com else 1, {}, None)
    return N.NativePlan(spec), spec


# ---- profiler: which of the library's kernels ran ---------------------------------------------------------------------------
_DEMANGLED = re.compile(r"mshgnn::(k_\w+)(?:<\s*(true|false)\s*>)?")
_MANGLED = re.compile(r"6mshgnn(\d+)")


def kernel_name(s):
    """'k_tc_encoder_dw<true>' from a demangled or mangled kernel name of the library (None for other kernels)."""
    m = _DEMANGLED.search(s)
    if m:
        return m.group(1) + (f"<{m.group(2)}>" if m.group(2) else "")
    m = _MANGLED.search(s)
    if m:
        end = m.end() + int(m.group(1))
        name, rest = s[m.end():end], s[end:]
        if name.startswith("k_"):
            return name + ("<true>" if rest.startswith("ILb1E") else ("<false>" if rest.startswith("ILb0E") else ""))
    return None


def profiled(fn):
    """(fn(), set of the library's kernel names the profiler saw while fn ran)."""
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
        res = fn()
        torch.cuda.synchronize()
    names = {kernel_name(e.name) for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA}
    names.discard(None)
    return res, names


def check_kernels(names, exp, tag, input_grad=True):
    if exp["fwd"] is None:                                   # fp32 mode: no tensor-core encoder kernel at all
        assert not {n for n in names if n.startswith("k_tc_")}, (tag, sorted(names))
    else:
        assert exp["fwd"] in names and not (ENCODER_FWD - {exp["fwd"]}) & names, (tag, exp, sorted(names))
        assert exp["dw"] in names and not (ENCODER_DW - {exp["dw"]}) & names, (tag, exp, sorted(names))
    if input_grad:
        assert exp["dx"] in names, (tag, exp, sorted(names))


# ---- inputs and models ------------------------------------------------------------------------------------------------------
def random_batch(cfg, B, seed, dtype=torch.float32, device="cuda:0"):
    """Seeded batch with random features for EVERY node type (fp64 features are drawn in fp64, fp16 ones rounded from fp32) and the
    labels of device_batch; labels stay fp32 whatever the feature dtype."""
    tpl = M.TEMPLATES[cfg.template]
    gen = torch.Generator(device=device).manual_seed(7000 + seed)
    x = {}
    for t in tpl.node_types:
        shape = (B * tpl.nodes_per_graph[t], cfg.in_width[t])
        x[t] = torch.randn(shape, generator=gen, device=device, dtype=torch.float64 if dtype == torch.float64 else torch.float32).to(dtype)
    if cfg.loss == "ce":
        y = (torch.rand(B * cfg.label_width, generator=gen, device=device) > 0.5).float()
    elif cfg.model.startswith("COM"):
        y = torch.randn(B, 6, generator=gen, device=device).repeat(1, tpl.nodes_per_graph["base"]).reshape(-1)
    else:
        y = torch.rand(B * cfg.label_width, generator=gen, device=device) * 70.0
    return HeteroBatch(x, tpl.edge_index_dict(B, device), y, B)


def misaligned(batch, offset_bytes):
    """The same batch with every feature tensor a contiguous view whose base pointer sits offset_bytes past a 16-byte boundary."""
    x = {}
    for k, v in batch.x_dict.items():
        e = offset_bytes // v.element_size()
        buf = torch.zeros(v.numel() + e + 16, dtype=v.dtype, device=v.device)
        x[k] = buf[e:e + v.numel()].view_as(v)
        x[k].copy_(v)
        assert x[k].is_contiguous() and x[k].data_ptr() % 16 == offset_bytes
    return HeteroBatch(x, batch.edge_index_dict, batch.y, batch.batch_size)


def models(cfg, layers, seed=0):
    om = oracle_model(cfg, layers=layers, seed=1 + seed)
    nm = build_model(cfg, layers=layers, seed=2 + seed)
    nm.load_state_dict({k: v.float() for k, v in om.state_dict().items()})
    return om, nm


def engine_facts(nm):
    eng = nm._last_engine
    spec = eng.spec
    return dict(zip(spec["node_types"], spec["in_width"])), live_slots(eng.plan, spec)


@pytest.fixture
def restore_encoder_options():
    yield
    N.set_option("encoder", DEFAULT[0]); N.set_option("encoder_tpi", DEFAULT[1]); N.set_option("encoder_dw_tma", DEFAULT[2])


def set_variant(v):
    N.set_option("encoder", v[0]); N.set_option("encoder_tpi", v[1]); N.set_option("encoder_dw_tma", v[2])


# ---- 1 + 2: width sweep, tensor-core mode, every encoder variant ------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("name,widths", WIDTH_CASES, ids=[case_id(c) for c in WIDTH_CASES])
def test_encoder_variants_at_input_width(name, widths, restore_encoder_options):
    t0 = time.time()
    cfg = cfg_with(name, widths)
    om, nm = models(cfg, 8)
    nm = nm.set_mode("tc").to("cuda:0")
    batch = random_batch(cfg, B, seed=sum(widths))
    ref, seen = None, {}
    for v in VARIANTS:
        set_variant(v)
        (out, loss, g, dx), names = profiled(lambda: native_train_step(cfg, nm, batch))
        w, live = engine_facts(nm)
        exp = expected_kernels(w, live, "tc", v)
        check_kernels(names, exp, (cfg.name, v))
        seen[v] = sorted(n for n in names if n in ENCODER_FWD | ENCODER_DW | {"k_tc_encoder_dx"})
        if ref is None:
            ref = (out.clone(), loss.clone(), {k: t.clone() for k, t in g.items()}, {k: t.clone() for k, t in dx.items()})
            continue
        assert torch.equal(out, ref[0]) and torch.equal(loss, ref[1]), (cfg.name, v)
        for k in g:
            assert torch.equal(g[k], ref[2][k]), (cfg.name, v, k)
        for k in dx:
            assert torch.equal(dx[k], ref[3][k]), (cfg.name, v, f"x.grad[{k}]")
    print(f"\ninput widths [{cfg.name}] live encoder slots {live}; tensor-map x.grad store for {exp['dx_tma']}")
    for v, n in seen.items():
        print(f"  encoder / tpi / dw_tma {v}: {n}")
    set_variant(DEFAULT)
    check_training_batch(cfg, nm, om, batch, "tc", cfg.name, {"kernels": seen[DEFAULT]}, t0)


# ---- 3: the same widths in fp32 (SIMT) mode ---------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("name,widths", WIDTH_CASES, ids=[case_id(c) for c in WIDTH_CASES])
def test_fp32_mode_at_input_width(name, widths):
    t0 = time.time()
    cfg = cfg_with(name, widths)
    om, nm = models(cfg, 8)
    nm = nm.set_mode("fp32").to("cuda:0")
    batch = random_batch(cfg, B, seed=sum(widths))
    _, names = profiled(lambda: native_train_step(cfg, nm, batch))
    w, live = engine_facts(nm)
    check_kernels(names, expected_kernels(w, live, "fp32"), cfg.name)
    check_training_batch(cfg, nm, om, batch, "fp32", cfg.name, {"kernels": sorted(names)}, t0)


# ---- 4: feature formats: fp16 / fp64 features, fp32 views on a base pointer 4 or 8 bytes past a 16-byte boundary -------------
FORMAT_CASES = [(MI, (12, 9, 6)), (MI, (388, 65, 130)), (K4C, (48, 18))]       # multiple of 4 / odd / even (not a multiple of 4)


@pytest.mark.gpu
@pytest.mark.parametrize("mode", ["tc", "fp32"])
@pytest.mark.parametrize("dtype", [torch.float16, torch.float64], ids=["fp16", "fp64"])
@pytest.mark.parametrize("name,widths", FORMAT_CASES, ids=[case_id(c) for c in FORMAT_CASES])
def test_feature_dtypes_at_input_width(name, widths, dtype, mode):
    t0 = time.time()
    cfg = cfg_with(name, widths)
    om, nm = models(cfg, 8)
    nm = nm.set_mode(mode).to("cuda:0")
    batch = random_batch(cfg, B, seed=sum(widths) + 1, dtype=dtype)
    _, names = profiled(lambda: native_train_step(cfg, nm, batch))
    w, live = engine_facts(nm)
    check_kernels(names, expected_kernels(w, live, mode, x_dtype=dtype), (cfg.name, dtype))
    check_training_batch(cfg, nm, om, batch, mode, f"{cfg.name} {dtype}", {"kernels": sorted(names)}, t0)


MISALIGNED_CASES = [(MI, (12, 4, 388)), (K4C, (12, 4)), (K4C, (1988, 4))]     # K % 4 == 0: aligned, these take k_tc_encoder_stream


@pytest.mark.gpu
@pytest.mark.parametrize("mode", ["tc", "fp32"])
@pytest.mark.parametrize("offset", [4, 8])
@pytest.mark.parametrize("name,widths", MISALIGNED_CASES, ids=[case_id(c) for c in MISALIGNED_CASES])
def test_misaligned_feature_views_at_input_width(name, widths, offset, mode, restore_encoder_options):
    """A 4-byte offset leaves only scalar loads, an 8-byte one 2-wide loads; neither may take the tensor maps of the persistent
    encoder or of the TMA-fed weight gradient (option encoder_dw_tma 1 is set to show that it falls back too)."""
    t0 = time.time()
    cfg = cfg_with(name, widths)
    om, nm = models(cfg, 8)
    nm = nm.set_mode(mode).to("cuda:0")
    batch = misaligned(random_batch(cfg, B, seed=sum(widths) + 2), offset)
    v = (-1, 0, 1)
    set_variant(v)
    _, names = profiled(lambda: native_train_step(cfg, nm, batch))
    w, live = engine_facts(nm)
    exp = expected_kernels(w, live, mode, v, misalign=offset)
    if mode == "tc":
        assert exp["fwd"] == "k_tc_encoder_pair" and exp["dw"] == "k_tc_encoder_dw<false>"
        assert expected_kernels(w, live, mode, v)["fwd"] == "k_tc_encoder_stream"        # aligned, the same widths stream
    check_kernels(names, exp, (cfg.name, offset))
    check_training_batch(cfg, nm, om, batch, mode, f"{cfg.name} base + {offset} B", {"kernels": sorted(names)}, t0)


# ---- 5: a model batch at K = 12 / 4 -----------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_model_batch_at_narrow_widths_is_bit_identical_to_single_models():
    """Three Solo12 K4 COM models at h = 2 (K = 12 / 4): one model-batch step gives every model the bits of its own single-model
    step.  The single models take the persistent encoder, the model batch the two-tile one (api.cu launch_tc_encoder)."""
    from test_gpu_model_batch import batched, check, singles
    cfg = cfg_with(K4C, (12, 4))
    dev = torch.device("cuda:0")
    ms = [build_model(cfg, layers=8, seed=10 + m).to(dev).set_mode("tc") for m in range(3)]
    batches = [random_batch(cfg, B, seed=20 + m) for m in range(3)]
    engs = []
    for nm, b in zip(ms, batches):
        eng, _ = nm._engine_for(b.x_dict, b.edge_index_dict)
        nm._ensure_flat(dev)
        engs.append(eng)
    eng = engs[0]
    w, live = dict(zip(eng.spec["node_types"], eng.spec["in_width"])), live_slots(eng.plan, eng.spec)
    _, n_single = profiled(lambda: singles(cfg, ms, batches, eng))
    _, n_batch = profiled(lambda: batched(cfg, ms, batches, eng))
    check_kernels(n_single, expected_kernels(w, live, "tc"), "single models", input_grad=False)        # a model batch has no x.grad
    check_kernels(n_batch, expected_kernels(w, live, "tc", n_models=3), "model batch", input_grad=False)
    assert "k_tc_encoder_stream" in n_single and "k_tc_encoder_pair" in n_batch
    print(f"\nmodel batch [{cfg.name} M=3 B={B}]: single models {sorted(n_single & ENCODER_FWD)}, model batch {sorted(n_batch & ENCODER_FWD)}")
    check(cfg, ms, batches, eng, tag=cfg.name)


# ---- 6: depth ---------------------------------------------------------------------------------------------------------------
DEPTH_CASES = [(name, L, mode) for name in ("mini_cheetah-k4-contact", "mi-contact", K4C) for L in (1, 9, 15) for mode in ("tc", "fp32")]


def assert_alive(cfg, nm, batch, L):
    """A deep random init whose activations die checks nothing: non-zero outputs, a non-zero encoder weight gradient for every
    type with a live encoder slot, and both ReLU signs among the live rows of the last layer's native mask."""
    out, _, g, _ = native_train_step(cfg, nm, batch)
    assert out.abs().max().item() > 0, "all outputs are zero"
    _, live = engine_facts(nm)
    for t, n in live.items():
        if n:
            assert g[f"encoder.lins.{t}.weight"].abs().max().item() > 0, f"encoder weight gradient of {t} is zero"
    pat = native_relu_pattern(nm, batch.batch_size, "cuda:0")
    last = [bits[live_rows] for key, (bits, live_rows) in pat.items() if key[0] != "enc" and key[1] == L - 1]
    bits = torch.cat([b.reshape(-1) for b in last])
    pos = bits.float().mean().item()
    assert 0.0 < pos < 1.0, f"last layer's ReLU mask is all {'ones' if pos else 'zeros'}"
    return pos


@pytest.mark.gpu
@pytest.mark.parametrize("name,L,mode", DEPTH_CASES)
def test_depth_matches_oracle(name, L, mode):
    t0 = time.time()
    cfg = CONFIGS[name]
    om, nm = models(cfg, L)
    nm = nm.set_mode(mode).to("cuda:0")
    batch = random_batch(cfg, B, seed=L)
    pos = assert_alive(cfg, nm, batch, L)
    check_training_batch(cfg, nm, om, batch, mode, f"{name} L={L}", {"layers": L, "last-layer ReLU ones": round(pos, 3)}, t0)


@pytest.mark.gpu
def test_15_layers_on_the_cta_pair_stack_kernel():
    t0 = time.time()
    cfg = CONFIGS["mini_cheetah-k4-contact"]
    L, Bp = 15, STACK_PAIR_MIN_GRAPHS
    om, nm = models(cfg, L)
    nm = nm.set_mode("tc").to("cuda:0")
    f = plan_facts(nm, random_batch(cfg, 1, seed=0))
    batch = random_batch(cfg, Bp, seed=L)
    sel = selection(nm, Bp, "tc", f)
    assert sel["stack"] == "CTA-pair"
    pos = assert_alive(cfg, nm, batch, L)
    check_training_batch(cfg, nm, om, batch, "tc", f"{cfg.name} L={L}", dict(sel, layers=L, last_relu_ones=round(pos, 3)), t0)


# ---- host checks ------------------------------------------------------------------------------------------------------------
def test_plan_takes_15_layers_and_rejects_16():
    for name in ("mini_cheetah-k4-contact", "mi-contact", K4C):
        plan, spec = host_plan(CONFIGS[name], layers=15)
        assert len(plan.describe()["need"]) == 16
        spec["num_layers"] = 16
        with pytest.raises(RuntimeError, match=re.escape("num_layers out of range (1..15)")):
            N.NativePlan(spec)


def test_width_grid_covers_the_widths_and_the_encoder_paths():
    """The restated selection rule over the width grid: every required width and every window-builder width is in it, and it runs
    each encoder path the GPU cases claim to exercise."""
    widths = {k for _, ws in WIDTH_CASES for k in ws}
    assert REQUIRED_WIDTHS <= widths, sorted(REQUIRED_WIDTHS - widths)
    assert window_widths() <= widths, sorted(window_widths() - widths)
    assert any(1900 <= k <= 2100 and k % 64 for k in widths)
    paths = set()
    for name, ws in WIDTH_CASES:
        cfg = cfg_with(name, ws)
        plan, spec = host_plan(cfg)
        w = dict(zip(spec["node_types"], spec["in_width"]))
        live = live_slots(plan, spec)
        assert all(live.values()), (cfg.name, live)              # at 8 layers every type's encoder is live
        if 4 in ws and max(ws) >= 1900:
            assert plan.describe()["enc_kmax"] >= 1920
            paths.add("narrow type in a wide weight image")
        for v in VARIANTS:
            e = expected_kernels(w, live, "tc", v)
            if v == DEFAULT:
                if e["fwd"] == "k_tc_encoder_stream" and min(ws) < 64:
                    paths.add("persistent encoder at K < 64")
                if e["fwd"] == "k_tc_encoder_stream" and cfg.model == "COM_HGNN_K4" and w["joint"] == 4:
                    paths.add("persistent encoder at K = 4 with signs")
                if e["fwd"] == "k_tc_encoder_pair":
                    paths.add("pair encoder when a row is not 16-byte aligned")
                if any(w[t] < 32 for t in e["dx_tma"]):
                    paths.add("tensor-map x.grad store at K < 32")
            if e["dw"] == "k_tc_encoder_dw<true>" and any(k % 64 and k > 192 for k in ws):
                paths.add("TMA-fed weight gradient at a K tail")
    assert paths == {"narrow type in a wide weight image", "persistent encoder at K < 64", "persistent encoder at K = 4 with signs",
                     "pair encoder when a row is not 16-byte aligned", "tensor-map x.grad store at K < 32",
                     "TMA-fed weight gradient at a K tail"}, paths


def test_selection_rule_fallbacks():
    """The rule's fallbacks on their own: odd / non-multiple-of-4 rows, misaligned bases, fp16 / fp64 features and model batches
    never take a tensor map of the features; option encoder 1 / 2 names its kernel."""
    w, live = {"base": 4, "joint": 12}, {"base": 4, "joint": 12}
    assert expected_kernels(w, live, "tc")["fwd"] == "k_tc_encoder_stream"
    assert expected_kernels(w, live, "tc", (0, 0, 1))["dw"] == "k_tc_encoder_dw<true>"
    assert expected_kernels(w, live, "tc")["dw"] == "k_tc_encoder_dw<false>"                   # TMA-fed rows only on request
    for kw in ({"misalign": 4}, {"misalign": 8}, {"x_dtype": torch.float16}, {"x_dtype": torch.float64}, {"n_models": 3}):
        e = expected_kernels(w, live, "tc", (0, 0, 1), **kw)
        assert e["fwd"] == "k_tc_encoder_pair" and e["dw"] == "k_tc_encoder_dw<false>", kw
    assert expected_kernels({"base": 4, "joint": 6}, live, "tc")["fwd"] == "k_tc_encoder_pair"
    assert expected_kernels({"base": 2, "joint": 12}, live, "tc")["fwd"] == "k_tc_encoder_pair"
    assert expected_kernels({"base": 2, "joint": 12}, {"base": 0, "joint": 12}, "tc")["fwd"] == "k_tc_encoder_stream"   # dead types do not count
    assert expected_kernels(w, {"base": 20, "joint": 13}, "tc")["fwd"] == "k_tc_encoder_pair"                          # > 32 live slots
    assert expected_kernels(w, live, "tc", (1, 0, 0))["fwd"] == "k_tc_encoder"
    assert expected_kernels(w, live, "tc", (2, 0, 0))["fwd"] == "k_tc_encoder_pair"
    assert expected_kernels({"base": 2, "joint": 12}, live, "tc")["dx_tma"] == ["joint"]


def test_kernel_names_are_read_from_both_name_forms():
    assert kernel_name("void mshgnn::k_tc_encoder_dw<true>(CUtensorMap_st, mshgnn::EncXMaps)") == "k_tc_encoder_dw<true>"
    assert kernel_name("mshgnn::k_tc_encoder_stream(mshgnn::EnqMaps, mshgnn::Tile const*, int)") == "k_tc_encoder_stream"
    assert kernel_name("mshgnn::k_tc_encoder(mshgnn::EncMaps, mshgnn::Tile const*)") == "k_tc_encoder"
    assert kernel_name("_ZN6mshgnn15k_tc_encoder_dwILb0EEEv14CUtensorMap_st") == "k_tc_encoder_dw<false>"
    assert kernel_name("_ZN6mshgnn17k_tc_encoder_pairENS_7EncMapsE") == "k_tc_encoder_pair"
    assert kernel_name("void at::native::vectorized_elementwise_kernel<4>(int)") is None
