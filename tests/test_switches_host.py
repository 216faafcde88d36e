"""Kernel choices are mshgnn_set_option options only: the environment variables that once selected kernels, item orders,
row splits or instrumented builds change nothing (CPU only, no compute calls)."""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

# every variable the library once read to pick a kernel or a measurement variant, each set to a non-default value
RETIRED = {
    "MSHGNN_STACK": "0", "MSHGNN_STACK_2CTA": "2", "MSHGNN_ENCODER": "v1", "MSHGNN_ENC_TPI": "2", "MSHGNN_ENC_DW": "tma",
    "MSHGNN_ROWGEMM": "tile", "MSHGNN_ENC_PREFETCH": "1", "MSHGNN_ENC_PF": "4", "MSHGNN_ENC_DEBUG": "1",
    "MSHGNN_STACK_RC": "8", "MSHGNN_STACK_DELAY": "3", "MSHGNN_STACK_ORDER": "diag", "MSHGNN_STACK_LOOKAHEAD": "3",
    "MSHGNN_STACK_DEBUG": "1", "MSHGNN_STACK_TIMING": "1", "MSHGNN_STACK_PRIVATE_DH": "0", "MSHGNN_DW_ROWS": "512",
    "MSHGNN_DW_FIT": "0",
}

# what the library reports for the K4 Mini Cheetah contact model in a fresh process
PROBE = r"""
import json, sys
sys.path.insert(0, sys.argv[1])
from ms_hgnn import _native as N
from ms_hgnn import morphology as M
from ms_hgnn.engine import build_spec
tpl = M.K4_MINI_CHEETAH
spec = build_spec(tpl.node_types, tpl.nodes_per_graph, {"base": 900, "joint": 300, "foot": 900}, tpl.edge_types, tpl.edges,
                  ("gt", "gs", "center_bb"), 128, 8, True, "base", "foot", 2, {}, None)
plan = N.NativePlan(spec)
out = {"options": {k: N.get_option(k) for k in ("stack", "stack_pair", "encoder", "encoder_tpi", "encoder_dw_tma")},
       "workspace": {f"{B}/{train}/{mode}": plan.workspace_bytes(B, train, mode)
                     for B in (2048, 16384) for train in (True, False) for mode in (N.MODE_TC, N.MODE_FP32)},
       "dw_layout": {B: [list(e) for e in plan.dw_layout(B, N.MODE_TC)] for B in (2048, 16384)},
       "timing_entry": hasattr(N.lib(), "mshgnn_stack_timing_offset")}
print(json.dumps(out))
"""


def _probe(extra_env):
    env = {k: v for k, v in os.environ.items() if k not in RETIRED}
    env.update(extra_env)
    r = subprocess.run([sys.executable, "-c", PROBE, os.path.join(ROOT, "morphsym-hgnn_b200")], env=env,
                       capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr
    return json.loads(r.stdout.strip().splitlines()[-1])


def test_retired_environment_variables_change_nothing():
    clean, retired = _probe({}), _probe(RETIRED)
    assert clean == retired
    assert clean["options"] == {"stack": 1, "stack_pair": 1, "encoder": -1, "encoder_tpi": 0, "encoder_dw_tma": -1}
    assert not clean["timing_entry"]
