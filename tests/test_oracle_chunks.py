"""The chunked fp64 oracle (helpers.oracle_run / oracle_grads_with_forced with ``device`` and ``chunk``) against the host oracle.

The host oracle, in one piece, is the one pinned to the reference (test_reference_pin.py, test_oracle_anchor.py).  The large-batch
parity tests run it on the GPU in chunks of graphs; these tests tie that run to the pinned one: outputs, loss, every parameter
gradient and every input gradient, with and without a forced ReLU sign pattern, agree to fp64 rounding.
"""
import pytest
import torch

import mshgnn_oracle as O
from helpers import graph_chunks, oracle_grads_with_forced, oracle_model, oracle_run, rel_err
from ms_hgnn.synthetic import CONFIGS, make_batch
from test_gpu_parity import CASES

FP64_TOL = 1e-12


def flip_smallest(model, batch, k=5):
    """A forced pattern that matters: the k pre-activations of smallest |x| of every ReLU call take the opposite sign."""
    with torch.no_grad(), O.ReluTap(record=True) as tap:
        model({n: v.double() for n, v in batch.x_dict.items()}, batch.edge_index_dict)
    forced = {}
    for i, pre in enumerate(tap.pre):
        v = pre.reshape(-1)
        idx = v.abs().topk(min(k, v.numel()), largest=False).indices
        forced[i] = (idx, ~(v[idx] > 0))
    return forced


def assert_same(a, b, what):
    out_a, loss_a, g_a, dx_a = a
    out_b, loss_b, g_b, dx_b = b
    assert rel_err(out_a, out_b) <= FP64_TOL, what
    assert abs(loss_a.item() - loss_b.item()) <= FP64_TOL * abs(loss_b.item()), what
    assert set(g_a) == set(g_b)
    for n in g_b:
        if g_b[n].norm() == 0:
            assert g_a[n].abs().max().item() == 0.0, (what, n)
        assert rel_err(g_a[n], g_b[n]) <= FP64_TOL, (what, n, rel_err(g_a[n], g_b[n]))
    for k in dx_b:
        assert rel_err(dx_a[k], dx_b[k]) <= FP64_TOL, (what, k, rel_err(dx_a[k], dx_b[k]))


def test_graph_chunks_cover_the_batch():
    assert graph_chunks(10, None) == [(0, 10)]
    assert graph_chunks(10, 4) == [(0, 4), (4, 8), (8, 10)]
    assert graph_chunks(8, 8) == [(0, 8)]


@pytest.mark.parametrize("name", ["mini_cheetah-k4-contact", "a1-c2-grf", "solo12-k4-com", "mi-contact"])
def test_chunked_host_oracle_equals_the_whole_batch_run(name):
    """Host, fp64: chunks of 3 graphs (the last one short) give the whole-batch outputs, loss and gradients to rounding, and a forced
    pattern sliced chunk by chunk gives the gradients of forcing it on the whole batch."""
    cfg = CONFIGS[name]
    B = 10
    batch = make_batch(cfg, B, seed=4)
    om = oracle_model(cfg, layers=3, seed=1)
    whole = oracle_run(cfg, om, batch, x_grad=True)
    chunked = oracle_run(cfg, om, batch, chunk=3, x_grad=True)
    assert_same(chunked, whole, "plain")
    forced = flip_smallest(om, batch)
    g_w, dx_w = oracle_grads_with_forced(cfg, om, batch, forced, x_grad=True)
    g_c, dx_c = oracle_grads_with_forced(cfg, om, batch, forced, chunk=3, x_grad=True)
    assert_same((whole[0], whole[1], g_c, dx_c), (whole[0], whole[1], g_w, dx_w), "forced")
    # the forced pattern changes the gradients: a slicing that dropped or misplaced it would not pass the line above
    assert max(rel_err(g_w[n], whole[2][n]) for n in g_w if whole[2][n].norm() > 0) > 1e-9


@pytest.mark.gpu
@pytest.mark.parametrize("name", sorted({c[0] for c in CASES}))
def test_device_oracle_equals_the_host_oracle(name):
    """Every config of the parity suite, at B = 37 / 130 / 300 in chunks of 16 / 64 / 128 graphs on the GPU, against the host oracle
    in one piece: outputs, loss, every parameter gradient and x.grad, plain and under a forced ReLU pattern, to 1e-12."""
    cfg = CONFIGS[name]
    om = oracle_model(cfg, layers=8, seed=1)
    worst = 0.0
    for B, chunk in ((37, 16), (130, 64), (300, 128)):
        batch = make_batch(cfg, B, seed=B)
        host = oracle_run(cfg, om, batch, x_grad=True)
        dev = oracle_run(cfg, om, batch, device="cuda:0", chunk=chunk, x_grad=True)
        assert dev[0].is_cuda and all(g.is_cuda for g in dev[2].values())
        assert_same(dev, host, f"B={B} plain")
        forced = flip_smallest(om, batch)
        g_h, dx_h = oracle_grads_with_forced(cfg, om, batch, forced, x_grad=True)
        g_d, dx_d = oracle_grads_with_forced(cfg, om, batch, forced, device="cuda:0", chunk=chunk, x_grad=True)
        assert_same((dev[0], dev[1], g_d, dx_d), (host[0], host[1], g_h, dx_h), f"B={B} forced")
        worst = max([worst, rel_err(dev[0], host[0])] + [rel_err(g_d[n], g_h[n]) for n in g_h] + [rel_err(dx_d[k], dx_h[k]) for k in dx_h])
    print(f"device oracle [{name}]: worst relative difference from the host oracle {worst:.1e}")
