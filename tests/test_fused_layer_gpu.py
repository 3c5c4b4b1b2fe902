"""The fp16x2 inference forward runs each EGNN layer as ONE launch (edge kernel with the node MLP and the next projections as
its tail, csrc/egnn_tc2.cu).  It must equal the two-launch fp16x2 path (edge kernel, then node kernel) bit for bit, and the
fp32 SIMT path within 1e-5, over batch shapes whose per-CTA node ranges are not multiples of the 128-node tile, grids
smaller than the SM count, isolated (zero in-degree) nodes and nodes whose in-edges fill a whole tile."""
import pytest
import torch

from immunostruct_b200 import _C
from immunostruct_b200 import functional as IF
from immunostruct_b200.graph import GraphBatch
from immunostruct_b200.synthetic import synthetic_graph_arrays

pytestmark = pytest.mark.gpu
DEV = "cuda"
H = 64


def _linear(gen, n_out, n_in, bias=True):
    bound = n_in ** -0.5                                   # nn.Linear's default initialisation range
    w = (torch.rand(n_out, n_in, generator=gen, device=DEV) * 2 - 1) * bound
    b = (torch.rand(n_out, generator=gen, device=DEV) * 2 - 1) * bound if bias else None
    return w, b


def _stack_params(seed, n_layers=6, edge_scale=1.0):
    """``edge_scale`` shrinks the edge messages so that hn = the sum over a node's in-edges stays at the size it has with ten
    in-edges: with 128 in-edges and default-sized weights the activations leave fp16's range within six layers (NaN)."""
    gen = torch.Generator(device=DEV).manual_seed(seed)
    params = []
    for l in range(n_layers):
        f = 20 if l == 0 else H
        W1, b1 = _linear(gen, H, 2 * f + 2)
        W2, b2 = _linear(gen, H, H)
        W2, b2 = W2 * edge_scale, b2 * edge_scale
        W3, b3 = _linear(gen, H, H)
        w4, _ = _linear(gen, 1, H, bias=False)
        W5, b5 = _linear(gen, H, f + H)
        W6, b6 = _linear(gen, H, H)
        params.append([W1, b1, W2, b2, W3, b3, w4, W5, b5, W6, b6])
    return params, _linear(gen, 3 * H, H)


def _two_launch_fp16x2(g, x23, edge_attr, params, qkv):
    """The stack as it runs without the node tail: edge kernel, then node kernel, per layer."""
    h, x = x23[:, :20], x23[:, 20:]
    n = h.shape[0]
    PQ = torch.empty(n, 2 * H, device=DEV)
    QKV = None
    _C.egnn_node_pre_fwd(h, params[0][0], params[0][1], PQ)
    last = len(params) - 1
    for l, (W1, b1, W2, b2, W3, b3, w4, W5, b5, W6, b6) in enumerate(params):
        upd = l != last
        hn, h_out = torch.empty(n, H, device=DEV), torch.empty(n, H, device=DEV)
        x_out = torch.empty(n, 3, device=DEV) if upd else None
        _C.egnn_edge_fwd_tc(g, PQ, x, edge_attr, h.shape[1], W1, W2, b2, W3, b3, w4, upd, _C.PREC_FP16X2, hn, x_out,
                            fast_act=True)
        PQ_next = torch.empty(n, 2 * H, device=DEV) if upd else None
        if not upd and qkv is not None:
            QKV = torch.empty(n, 3 * H, device=DEV)
            _C.egnn_node_post_pre_tc(h, hn, W5, b5, W6, b6, h_out, qkv[0], qkv[1], QKV, _C.PREC_FP16X2, next_kind=2)
        else:
            nxt = params[l + 1] if upd else (None, None)
            _C.egnn_node_post_pre_tc(h, hn, W5, b5, W6, b6, h_out, nxt[0], nxt[1], PQ_next, _C.PREC_FP16X2)
        h, PQ = h_out, PQ_next
        if upd:
            x = x_out
    return h, QKV


def _rel(a, b):
    return float((a - b).abs().max() / b.abs().max().clamp_min(1e-30))


# (graphs, nodes per graph, in-degree, isolated padding nodes per graph)
SHAPES = [(512, 200, 10, 0), (1, 200, 10, 0), (3, 200, 10, 0), (37, 200, 10, 0), (6, 200, 10, 40), (4, 150, 128, 0)]


@pytest.mark.parametrize("shape", SHAPES, ids=lambda s: "b{}_n{}_k{}_pad{}".format(*s))
@pytest.mark.parametrize("with_qkv", [True, False], ids=["qkv", "no_qkv"])
def test_fused_stack_equals_two_launch_path_and_fp32(shape, with_qkv):
    n_graphs, n_nodes, k, n_pad = shape
    arr = synthetic_graph_arrays(n_graphs, n_nodes, k, seed=n_graphs + k, device=DEV, n_pad=n_pad)
    g = GraphBatch.from_arrays(*(arr[kk] for kk in ("x", "src", "dst", "edge_attr", "node_counts", "edge_counts")),
                               max_nodes=n_nodes)
    x23, edge_attr = arr["x"], arr["edge_attr"].contiguous()
    params, (Wqkv, bqkv) = _stack_params(seed=n_graphs, edge_scale=min(1.0, 10.0 / k))
    qkv = (Wqkv, bqkv) if with_qkv else None
    prev = IF.get_precision()
    try:
        IF.set_precision("fp16x2")
        with torch.no_grad():
            before = _C.LAUNCHES
            out = IF.egnn_stack_infer(g, x23, edge_attr, params, qkv)
            assert _C.LAUNCHES - before == 1 + len(params)          # node_pre of layer 0, then one launch per layer
            h, QKV = out if with_qkv else (out, None)
            h_ref, QKV_ref = _two_launch_fp16x2(g, x23, edge_attr, params, qkv)
            IF.set_precision("fp32")
            out32 = IF.egnn_stack_infer(g, x23, edge_attr, params, qkv)
            h32 = out32[0] if with_qkv else out32
        torch.cuda.synchronize()
    finally:
        IF.set_precision(prev)
    bits = lambda t: t.view(torch.int32)
    assert torch.equal(bits(h), bits(h_ref))
    assert bool(torch.isfinite(h).all())
    if with_qkv:
        assert torch.equal(bits(QKV), bits(QKV_ref))
        assert _rel(QKV, h32 @ Wqkv.t() + bqkv) < 1e-5
    assert _rel(h, h32) < 1e-5
