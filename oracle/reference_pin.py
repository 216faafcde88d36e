"""TEST INFRASTRUCTURE ONLY - runs the reference's UNMODIFIED model files on the CPU.

The reference's model classes (``src/ms_hgnn/lightning_py/hgnn*.py`` of the MorphSym-HGNN repository) import four names
from ``torch_geometric.nn`` and nothing else outside torch / yaml.  With ``oracle/pyg_shim`` first on ``sys.path`` they
import and run as they are: this module loads them from where they lie (nothing is copied), builds the class a
``synthetic.Config`` names with the reference's own yaml (``cfg/*.yaml``), and returns fp64 outputs, loss and every
parameter gradient.  The reference is found through the environment variable ``MSHGNN_REFERENCE`` (the directory of a
checkout of that repository).  ``tests/test_reference_pin.py`` compares the oracle with it live when it is set, and
always through the fixtures ``tools/make_golden.py`` stores under ``tests/golden/``.
"""
from __future__ import annotations

import contextlib
import importlib.util
import io
import os
import sys
from typing import Dict

import torch

REF_ROOT = os.environ.get("MSHGNN_REFERENCE", "")          # checkout of the reference repository; unset: live checks skip
REF_MODELS = os.path.join(REF_ROOT, "src", "ms_hgnn", "lightning_py")
SHIM = os.path.join(os.path.dirname(os.path.abspath(__file__)), "pyg_shim")

# class name -> reference file
REF_FILE = {
    "GRF_HGNN": "hgnn.py", "COM_HGNN": "hgnn.py", "GRF_HGNN_K4": "hgnn_k4.py", "GRF_HGNN_C2": "hgnn_c2.py",
    "COM_HGNN_K4": "hgnn_k4_com.py", "COM_HGNN_C2": "hgnn_c2_com.py", "COM_HGNN_S4": "hgnn_s4_com.py",
}


def available() -> bool:
    return bool(REF_ROOT) and os.path.isdir(REF_MODELS)


def load_reference_class(name: str):
    """Imports the reference file that defines ``name`` (unmodified, by path) against the torch_geometric shim."""
    path = os.path.join(REF_MODELS, REF_FILE[name])
    had = sys.modules.get("torch_geometric"), sys.modules.get("torch_geometric.nn")
    sys.path.insert(0, SHIM)
    try:
        for m in ("torch_geometric", "torch_geometric.nn"):
            sys.modules.pop(m, None)
        spec = importlib.util.spec_from_file_location("_reference_" + REF_FILE[name][:-3], path)
        mod = importlib.util.module_from_spec(spec)
        spec.loader.exec_module(mod)
        import torch_geometric
        assert torch_geometric.__version__.endswith("+shim"), "a real torch_geometric shadows the shim"
    finally:
        sys.path.remove(SHIM)
        for key, old in zip(("torch_geometric", "torch_geometric.nn"), had):
            if old is not None:
                sys.modules[key] = old
    return getattr(mod, name)


def build_reference_model(cfg, layers: int, seed: int, hidden: int = 128):
    """The reference class ``cfg.model`` with seeded fp64 weights whose values are exactly representable in fp32."""
    from ms_hgnn import morphology as M
    tpl = M.TEMPLATES[cfg.template]
    cls = load_reference_class(cfg.model)
    kw = dict(hidden_channels=hidden, num_layers=layers, data_metadata=tpl.metadata, regression=cfg.regression)
    if cfg.group is not None:
        kw.update(symmetry_mode="MorphSym", group_operator_path=os.path.join(REF_ROOT, "cfg", cfg.group + ".yaml"))
    if cfg.model in ("GRF_HGNN_C2", "GRF_HGNN"):
        kw["grf_dimension"] = cfg.grf_dimension
    prev = torch.get_default_dtype()
    torch.set_default_dtype(torch.float64)
    try:
        torch.manual_seed(3000 + seed)
        with contextlib.redirect_stdout(io.StringIO()):           # the reference constructors print their sign tables
            model = cls(**kw)
    finally:
        torch.set_default_dtype(prev)
    return model


def materialize(model, batch) -> None:
    """First forward allocates the lazy encoder (HeteroDictLinear(-1, ...)); then round every weight through fp32."""
    x = {k: v.double().clone() for k, v in batch.x_dict.items()}
    with torch.no_grad():
        model(x, batch.edge_index_dict)
        for p in model.parameters():
            p.copy_(p.float().double())


def reference_run(cfg, model, batch, loss_fn):
    """fp64 forward + loss + backward of the reference model; ``loss_fn(cfg, out, y, B)`` is the test's loss head."""
    x = {k: v.double().clone() for k, v in batch.x_dict.items()}      # the reference mutates its input dict
    model.zero_grad()
    out = model(x, batch.edge_index_dict)
    loss = loss_fn(cfg, out, batch.y.double(), batch.batch_size)
    loss.backward()
    grads: Dict[str, torch.Tensor] = {n: (p.grad.clone() if p.grad is not None else torch.zeros_like(p))
                                      for n, p in model.named_parameters()}
    return out.detach(), loss.detach(), grads


# ------------------------------------------------------------------------------------------------
# weights / probes both sides can regenerate from a seed (no reference needed on the GPU box)
# ------------------------------------------------------------------------------------------------
def seeded_state_dict(model_or_items, seed: int) -> Dict[str, torch.Tensor]:
    """U(+-1/sqrt(fan_in)) weights drawn tensor by tensor from one seeded generator and rounded through fp32.

    ``model_or_items``: a module (its ``state_dict()`` order is used) or a list of ``(key, shape)`` in the order to
    draw - the fixture stores the reference model's order, so the oracle loads the very same numbers without it."""
    if hasattr(model_or_items, "state_dict"):
        items = [(k, tuple(v.shape)) for k, v in model_or_items.state_dict().items()]
    else:
        items = [(k, tuple(s)) for k, s in model_or_items]
    gen = torch.Generator().manual_seed(7000 + seed)
    out = {}
    for k, shape in items:
        fan_in = shape[1] if len(shape) == 2 else shape[0]
        w = (torch.rand(shape, generator=gen, dtype=torch.float64) * 2.0 - 1.0) / (fan_in ** 0.5)
        out[k] = w.float().double()
    return out


def grad_digest(grads: Dict[str, torch.Tensor], seed: int = 0) -> Dict[str, tuple]:
    """Per tensor: (L2 norm, dot product with a seeded +-1 probe).  Two numbers pin a tensor far below 1e-12."""
    out = {}
    for i, k in enumerate(sorted(grads)):
        g = grads[k].double().reshape(-1)
        gen = torch.Generator().manual_seed(9000 + seed + i)
        probe = (torch.randint(0, 2, g.shape, generator=gen, dtype=torch.int64) * 2 - 1).double()
        out[k] = (g.norm().item(), torch.dot(g, probe).item())
    return out
