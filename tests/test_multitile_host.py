"""CPU checks of the references that tests/test_multitile_gpu.py relies on: the full-model oracle run in chunks of
graphs is the one-shot oracle, and the fp64 context makes each kernel contract used there compute in fp64."""
import types

import pytest
import torch

from immunostruct_b200.synthetic import split_graphs
from oracle import kernel_contracts as KC
from oracle import reference_ops as R

from conftest import rel_err
from helpers import fp64_default, oracle_training_step
from test_kernels_gpu import egnn_weights, random_multigraph_arrays, rnd
from test_models_gpu import _bench_shape_case


def test_chunked_oracle_equals_the_one_shot_oracle():
    """Batch 12 in chunks of 4 against batch 12 in one piece, in fp64: logits, loss and every gradient within 1e-12 (of
    the gradient's scale, floored at 1e-2 of the largest gradient as in assert_grads_close: the key bias's true
    gradient is exactly zero)."""
    b = 12
    arr, dense, model, eps = _bench_shape_case(b, seed=5, n_pad=10, device="cpu")
    state = model.state_dict()
    out1, loss1, g1 = oracle_training_step(state, arr, dense, eps, torch.float64)
    out4, loss4, g4 = oracle_training_step(state, arr, dense, eps, torch.float64, chunk=4)
    assert out1.dtype == loss1.dtype == torch.float64 and out1.shape == out4.shape == (b, 1)
    assert float(out1.std()) > 0.0
    assert rel_err(out4, out1) < 1e-12 and rel_err(loss4, loss1) < 1e-12
    assert g1.keys() == g4.keys()
    gmax = max(float(g.abs().max()) for g in g1.values() if g is not None)
    n_grads = 0
    for k, g in g1.items():
        assert (g is None) == (g4[k] is None), k
        if g is not None:
            err = float((g4[k] - g).abs().max())
            assert g.dtype == torch.float64 and err <= 1e-12 * max(float(g.abs().max()), 1e-2 * gmax), (k, err)
            n_grads += 1
    assert n_grads > 50


def _beyond_fp32(t):
    """True when some value of ``t`` is not an fp32 number: a contract that computed in fp32 and copied its result into
    an fp64 buffer would hold fp32 numbers only."""
    return t.dtype == torch.float64 and bool((t - t.float().double()).abs().max() > 0)


def _contract_outputs():
    """Each contract that tests/test_multitile_gpu.py runs in fp64, on small double inputs -> {name: [outputs]}."""
    gen = torch.Generator().manual_seed(3)
    arrays = random_multigraph_arrays(5, [17, 1, 64, 33], 5.0)
    g = R.dgl_batch(split_graphs(arrays))
    cg = types.SimpleNamespace(**R.csr_from_coo(g["src"], g["dst"], g["num_nodes"]))
    cg.node_off = torch.zeros(5, dtype=torch.int64)
    cg.node_off[1:] = torch.cumsum(g["batch_num_nodes"], 0)
    n, e, f = int(g["num_nodes"]), int(g["src"].numel()), 64
    d = lambda *s, scale=1.0: rnd(gen, *s, scale=scale).double()          # noqa: E731
    w = {k: v.double() for k, v in egnn_weights(gen, f).items()}
    h, hn, x, ea = d(n, f), d(n, 64), arrays["x"][:, 20:].double(), arrays["edge_attr"].double()
    out = {}
    e64 = lambda *s: torch.empty(*s, dtype=torch.float64)                  # noqa: E731
    o = [e64(n, 64), e64(n, 64), e64(1, 64 * (f + 64) + 4224)]
    KC.egnn_node_post_bwd(d(n, 64), h, hn, w["W5"], w["b5"], w["W6"], *o)
    out["egnn_node_post_bwd"] = o
    o = [e64(n, 64), e64(n, 3), e64(1, 128 * f + 64)]
    KC.egnn_node_pre_bwd(d(e, 64), d(n, 64), d(e, 3), d(n, 3), d(n, 3), d(n, 64), cg, h, w["W1"], *o)
    out["egnn_node_pre_bwd"] = o
    o = [e64(n, 64), e64(n, 128)]
    KC.egnn_node_post_pre_tc(h, hn, w["W5"], w["b5"], w["W6"], w["b6"], o[0], w["W1"], w["b1"], o[1], 3)
    out["egnn_node_post_pre_tc"] = o
    o = [e64(n, 128)]
    KC.egnn_node_pre_fwd(h, w["W1"], w["b1"], o[0])
    out["egnn_node_pre_fwd"] = o
    o = [e64(n, 64)]
    KC.egnn_node_post_fwd(h, hn, w["W5"], w["b5"], w["W6"], w["b6"], o[0])
    out["egnn_node_post_fwd"] = o
    names = ("W1", "W2", "b2", "W3", "b3", "w4")
    o = [e64(n, 64), e64(n, 3)]
    KC.egnn_edge_fwd(cg, d(n, 128), x, ea, f, *(w[k] for k in names), True, *o)
    out["egnn_edge_fwd"] = o
    o = [e64(e, 64), e64(n, 64), e64(e, 3), e64(n, 3), e64(1, 8512)]
    KC.egnn_edge_bwd(cg, d(n, 128), x, ea, f, *(w[k] for k in names), d(n, 64), d(n, 3), *o)
    out["egnn_edge_bwd"] = o[:4] + [o[4][:, :8192]]
    off, QKV, gp = cg.node_off, d(n, 192, scale=0.7), d(4, 64)
    o = [e64(n, 64), e64(n, 1), e64(4, 64)]
    KC.attn_pool_fwd(QKV, off, 1, 64, *o)
    out["attn_pool_fwd"] = o
    o = [e64(4, 64)]
    KC.attn_pool_infer(QKV, off, 8, 64, o[0])
    out["attn_pool_infer"] = o
    o = [e64(n, 192)]
    KC.attn_pool_bwd(QKV, None, None, off, 8, 64, gp, d(n, 64), o[0])
    out["attn_pool_bwd"] = o
    o = [e64(n, 192)]
    KC.attn_pool_bwd_tc(QKV, off, 64, gp, o[0])
    out["attn_pool_bwd_tc"] = o
    return out


def test_fp64_context_makes_the_contracts_compute_in_fp64():
    with fp64_default():
        outs = _contract_outputs()
    assert torch.get_default_dtype() == torch.float32
    for name, tensors in outs.items():
        for i, t in enumerate(tensors):
            assert bool(torch.isfinite(t).all()), (name, i)
            assert _beyond_fp32(t), f"{name} output {i} holds fp32 values only"


def test_fp64_context_restores_the_default_dtype_when_the_body_raises():
    assert torch.get_default_dtype() == torch.float32
    with pytest.raises(ZeroDivisionError):
        with fp64_default():
            assert torch.get_default_dtype() == torch.float64
            assert torch.zeros(1).dtype == torch.float64
            1 / 0
    assert torch.get_default_dtype() == torch.float32
