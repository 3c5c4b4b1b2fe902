"""``torch.library`` registration of the fused operators (SURVEY 8(b)): every op is a ``torch.library.custom_op`` in
the ``immunostruct_b200::`` namespace with a fake (meta) implementation and ``register_autograd``, so that autograd,
``no_grad``, ``torch.compile`` / fake-tensor tracing and DDP-style hooks see ordinary operators:

    torch.ops.immunostruct_b200.egnn_stack       6 x dgl.nn.EGNNConv             models/hybrid_models.py:89-90 / 323-324
    torch.ops.immunostruct_b200.attention_pool   per-graph attention + mean pool models/layers.py:13-22,67-78; :92-97
    torch.ops.immunostruct_b200.segment_pool     global_mean_pool / max_pool     hybrid_models.py:97; ablation_models.py:296-297
    torch.ops.immunostruct_b200.linear           vae_fc1 / vae_fc4               hybrid_models.py:297-308
    torch.ops.immunostruct_b200.fusion_attention combined_attention + mean       hybrid_models.py:344-347
    torch.ops.immunostruct_b200.fused_loss       Losses.*                        utils/loss.py:13-31

Each implementation enqueues the same C-ABI launchers as ``functional.py`` (no second code path for the arithmetic).
The model classes call the lean ``torch.autograd.Function`` wrappers of ``functional.py`` by default -- the dispatcher
adds 20-40 us of host time per call to a step that issues ~300 launches in ~11 ms -- and route through these
registered ops after ``immunostruct_b200.use_custom_ops(True)`` (tests/test_custom_ops.py runs both and compares).
"""
from __future__ import annotations

from types import SimpleNamespace
from typing import List, Optional

import torch
from torch import Tensor

from . import _C
from . import functional as IF

H = IF.H
_GRAPH_FIELDS = ("indptr", "csr_src", "csr_dst", "csr_eid", "outptr", "csc_pos", "status", "node_off", "stats")


def graph_tensors(graph) -> List[Tensor]:
    """The tensors of a collated GraphBatch that the EGNN / attention ops consume, in ``_GRAPH_FIELDS`` order."""
    return [getattr(graph, f) for f in _GRAPH_FIELDS]


def _graph_ns(tensors: List[Tensor], n_edges: int, n_graphs: int, max_nodes: int):
    ns = SimpleNamespace(**dict(zip(_GRAPH_FIELDS, tensors)))
    ns.n_edges, ns.n_graphs, ns.max_nodes = n_edges, n_graphs, max_nodes
    return ns


# ---- segment pooling ------------------------------------------------------------------------------
@torch.library.custom_op("immunostruct_b200::segment_pool", mutates_args=())
def segment_pool(x: Tensor, node_off: Tensor, mode: str) -> Tensor:
    x = x if x.stride(-1) == 1 else x.contiguous()
    out = x.new_empty(node_off.numel() - 1, x.shape[1])
    _C.segment_pool_fwd(x, node_off, mode, out)
    return out


@segment_pool.register_fake
def _(x, node_off, mode):
    return x.new_empty(node_off.numel() - 1, x.shape[1])


@torch.library.custom_op("immunostruct_b200::segment_pool_bwd", mutates_args=())
def segment_pool_bwd(x: Tensor, node_off: Tensor, mode: str, pooled: Tensor, g_out: Tensor) -> Tensor:
    x = x if x.stride(-1) == 1 else x.contiguous()
    gx = torch.empty_like(x, memory_format=torch.contiguous_format)
    _C.segment_pool_bwd(x, node_off, mode, pooled, g_out.contiguous(), gx)
    return gx


@segment_pool_bwd.register_fake
def _(x, node_off, mode, pooled, g_out):
    return torch.empty_like(x, memory_format=torch.contiguous_format)


def _segment_pool_setup(ctx, inputs, output):
    x, node_off, mode = inputs
    ctx.mode = mode
    ctx.save_for_backward(x, node_off, output)


def _segment_pool_backward(ctx, g):
    x, node_off, pooled = ctx.saved_tensors
    return segment_pool_bwd(x, node_off, ctx.mode, pooled, g), None, None


segment_pool.register_autograd(_segment_pool_backward, setup_context=_segment_pool_setup)


# ---- dense Linear on the TMA-fed tensor-core GEMM -----------------------------------------------------
@torch.library.custom_op("immunostruct_b200::linear", mutates_args=())
def linear(x: Tensor, weight: Tensor, bias: Optional[Tensor], relu: bool) -> Tensor:
    n = IF._n_planes()
    xp, _, _, flag = _C.split_planes(x if x.stride(-1) == 1 else x.contiguous(), n, flag=(n == 3))
    wp, _ = IF._planes_of_weight(weight, False)
    return _C.gemm_planes(xp, wp, None if bias is None else bias.contiguous(), relu, a_flag=flag)


@linear.register_fake
def _(x, weight, bias, relu):
    return x.new_empty(x.shape[0], weight.shape[0])


@torch.library.custom_op("immunostruct_b200::linear_bwd", mutates_args=())
def linear_bwd(gy: Tensor, x: Tensor, weight: Tensor, y: Optional[Tensor], need_dx: bool, need_dw: bool,
               need_db: bool) -> List[Tensor]:
    """-> [gx | empty, gW | empty, gb | empty]; ``y`` = the ReLU output when the layer had one (its mask)."""
    n = IF._n_planes()
    gy = gy if gy.stride(-1) == 1 else gy.contiguous()
    gp, gpt, part, _ = _C.split_planes(gy, n, rows=need_dx, transposed=need_dw, relu_src=y, colsum=need_db)
    gx, gw, gb = gy.new_empty(0), gy.new_empty(0), gy.new_empty(0)
    if need_dx:
        gx = _C.gemm_planes(gp, IF._planes_of_weight(weight, True)[1])
    if need_dw:
        _, xpt, _, xflag = _C.split_planes(x if x.stride(-1) == 1 else x.contiguous(), n, rows=False, transposed=True,
                                           flag=(n == 3))
        gw = _C.gemm_planes(gpt, xpt, b_flag=xflag)
    if need_db:
        gb = gy.new_empty(gy.shape[1])
        _C.reduce_partials(part, gb)
    return [gx, gw, gb]


@linear_bwd.register_fake
def _(gy, x, weight, y, need_dx, need_dw, need_db):
    e = gy.new_empty(0)
    return [torch.empty_like(x) if need_dx else e, torch.empty_like(weight) if need_dw else e,
            gy.new_empty(gy.shape[1]) if need_db else e]


def _linear_setup(ctx, inputs, output):
    x, weight, bias, relu = inputs
    ctx.has_bias = bias is not None
    ctx.save_for_backward(x, weight, output if relu else None)


def _linear_backward(ctx, gy):
    x, weight, y = ctx.saved_tensors
    need = ctx.needs_input_grad
    gx, gw, gb = linear_bwd(gy, x, weight, y, need[0], need[1], ctx.has_bias and need[2])
    return (gx if need[0] else None, gw if need[1] else None, gb if ctx.has_bias and need[2] else None, None)


linear.register_autograd(_linear_backward, setup_context=_linear_setup)


# ---- fusion attention (closed form) -----------------------------------------------------------------
@torch.library.custom_op("immunostruct_b200::fusion_attention", mutates_args=())
def fusion_attention(c: Tensor, coef: Tensor, n_head: int) -> Tensor:
    c, coef = c.contiguous(), coef.contiguous()
    out = torch.empty_like(c)
    _C.fusion_attn_fwd(c, n_head, coef, out)
    return out


@fusion_attention.register_fake
def _(c, coef, n_head):
    return torch.empty_like(c, memory_format=torch.contiguous_format)


@torch.library.custom_op("immunostruct_b200::fusion_attention_bwd", mutates_args=())
def fusion_attention_bwd(c: Tensor, coef: Tensor, n_head: int, gout: Tensor) -> List[Tensor]:
    c, coef, gout = c.contiguous(), coef.contiguous(), gout.contiguous()
    gc, part = torch.empty_like(c), c.new_empty(c.shape[0], 4 * n_head)
    _C.fusion_attn_bwd(c, n_head, coef, gout, gc, part)
    return [gc, torch.cat([part.sum(0), gout.sum().reshape(1)])]


@fusion_attention_bwd.register_fake
def _(c, coef, n_head, gout):
    return [torch.empty_like(c, memory_format=torch.contiguous_format), torch.empty_like(coef)]


def _fusion_setup(ctx, inputs, output):
    c, coef, n_head = inputs
    ctx.n_head = n_head
    ctx.save_for_backward(c, coef)


def _fusion_backward(ctx, gout):
    c, coef = ctx.saved_tensors
    gc, gcoef = fusion_attention_bwd(c, coef, ctx.n_head, gout)
    return gc, gcoef, None


fusion_attention.register_autograd(_fusion_backward, setup_context=_fusion_setup)


# ---- per-graph attention + mean pool (pooled rows only) -------------------------------------------------
@torch.library.custom_op("immunostruct_b200::attention_pool", mutates_args=())
def attention_pool(qkv: Tensor, node_off: Tensor, n_head: int, max_nodes: int) -> Tensor:
    qkv = qkv.contiguous()
    pooled = qkv.new_empty(node_off.numel() - 1, H)
    prec = IF._PRECISIONS[IF.get_precision()]
    if n_head == 1 and prec is not None and max_nodes <= 256:
        _C.attn_pool_infer_tc(qkv, node_off, max_nodes, pooled, _C.PREC_BF16 if prec == _C.PREC_BF16 else _C.PREC_BF16X3)
    else:
        _C.attn_pool_infer(qkv, node_off, n_head, max_nodes, pooled)
    return pooled


@attention_pool.register_fake
def _(qkv, node_off, n_head, max_nodes):
    return qkv.new_empty(node_off.numel() - 1, H)


@torch.library.custom_op("immunostruct_b200::attention_pool_bwd", mutates_args=())
def attention_pool_bwd(qkv: Tensor, node_off: Tensor, n_head: int, max_nodes: int, g_pooled: Tensor) -> Tensor:
    qkv, g_pooled = qkv.contiguous(), g_pooled.contiguous()
    gqkv = torch.empty_like(qkv)
    if n_head == 1 and IF._PRECISIONS[IF.get_precision()] is not None and max_nodes <= 256:
        _C.attn_pool_bwd_tc(qkv, node_off, max_nodes, g_pooled, gqkv)
    else:                                                   # row statistics recomputed (O = NULL), LSE is scratch
        lse = qkv.new_empty(qkv.shape[0], n_head)
        _C.attn_pool_bwd(qkv, None, lse, node_off, n_head, max_nodes, g_pooled, None, gqkv)
    return gqkv


@attention_pool_bwd.register_fake
def _(qkv, node_off, n_head, max_nodes, g_pooled):
    return torch.empty_like(qkv, memory_format=torch.contiguous_format)


def _attn_setup(ctx, inputs, output):
    qkv, node_off, n_head, max_nodes = inputs
    ctx.cfg = (n_head, max_nodes)
    ctx.save_for_backward(qkv, node_off)


def _attn_backward(ctx, g):
    qkv, node_off = ctx.saved_tensors
    return attention_pool_bwd(qkv, node_off, ctx.cfg[0], ctx.cfg[1], g), None, None, None


attention_pool.register_autograd(_attn_backward, setup_context=_attn_setup)


# ---- fused loss ----------------------------------------------------------------------------------------
@torch.library.custom_op("immunostruct_b200::fused_loss", mutates_args=())
def fused_loss(recon: Optional[Tensor], seq: Optional[Tensor], mu: Optional[Tensor], logvar: Optional[Tensor], logits: Tensor,
               y: Tensor, mode: int, pos_weight: float, w_pred: float, w_mse: float, w_kld: float) -> Tensor:
    """-> [total, prediction term, recon MSE, KLD]"""
    lg, yy = logits.reshape(-1).contiguous(), y.reshape(-1).contiguous().float()
    if recon is not None:
        recon, seq = recon.contiguous(), seq.reshape(recon.shape[0], -1).contiguous()
        mu, logvar = mu.contiguous(), logvar.contiguous()
    out = lg.new_empty(4)
    _C.loss_fwd(recon, seq, mu, logvar, lg, yy, mode, pos_weight, w_pred, w_mse, w_kld, lg.new_empty(_C.loss_num_partials()), out)
    return out


@fused_loss.register_fake
def _(recon, seq, mu, logvar, logits, y, mode, pos_weight, w_pred, w_mse, w_kld):
    return logits.new_empty(4)


@torch.library.custom_op("immunostruct_b200::fused_loss_bwd", mutates_args=())
def fused_loss_bwd(recon: Optional[Tensor], seq: Optional[Tensor], mu: Optional[Tensor], logvar: Optional[Tensor],
                   logits: Tensor, y: Tensor, mode: int, pos_weight: float, w_pred: float, w_mse: float, w_kld: float,
                   gout: Tensor) -> List[Tensor]:
    lg, yy = logits.reshape(-1).contiguous(), y.reshape(-1).contiguous().float()
    g_logits = torch.empty_like(lg)
    if recon is not None:
        recon, seq = recon.contiguous(), seq.reshape(recon.shape[0], -1).contiguous()
        mu, logvar = mu.contiguous(), logvar.contiguous()
        g_recon, g_mu, g_lv = torch.empty_like(recon), torch.empty_like(mu), torch.empty_like(logvar)
    else:
        g_recon = g_mu = g_lv = None
    _C.loss_bwd(recon, seq, mu, logvar, lg, yy, mode, pos_weight, w_pred, w_mse, w_kld, gout.reshape(1).contiguous().float(),
                g_recon, g_mu, g_lv, g_logits)
    e = lambda: lg.new_empty(0)
    return [g_recon if g_recon is not None else e(), g_mu if g_mu is not None else e(), g_lv if g_lv is not None else e(),
            g_logits.view(logits.shape)]


@fused_loss_bwd.register_fake
def _(recon, seq, mu, logvar, logits, y, mode, pos_weight, w_pred, w_mse, w_kld, gout):
    e = logits.new_empty(0)
    return [torch.empty_like(recon) if recon is not None else e, torch.empty_like(mu) if mu is not None else e,
            torch.empty_like(logvar) if logvar is not None else e, torch.empty_like(logits)]


def _loss_setup(ctx, inputs, output):
    recon, seq, mu, logvar, logits, y, *cfg = inputs
    ctx.cfg = cfg
    ctx.has_seq = recon is not None
    ctx.save_for_backward(recon, seq, mu, logvar, logits, y)


def _loss_backward(ctx, g):
    recon, seq, mu, logvar, logits, y = ctx.saved_tensors
    g_recon, g_mu, g_lv, g_logits = fused_loss_bwd(recon, seq, mu, logvar, logits, y, *ctx.cfg, g[0])
    none = (None,) * 5
    if ctx.has_seq:
        return (g_recon, None, g_mu, g_lv, g_logits, None) + none
    return (None, None, None, None, g_logits, None) + none


fused_loss.register_autograd(_loss_backward, setup_context=_loss_setup)


# ---- EGNN stack ----------------------------------------------------------------------------------------
@torch.library.custom_op("immunostruct_b200::egnn_stack", mutates_args=())
def egnn_stack(x23: Tensor, edge_attr: Tensor, params: List[Tensor], graph: List[Tensor], n_layers: int, n_edges: int,
               n_graphs: int, max_nodes: int, qkv: List[Tensor]) -> List[Tensor]:
    """-> [h_final, QKV, then per layer (h_in, x_in, PQ, hn)]: the intermediates are outputs so that autograd can keep them.
    ``qkv`` = [W [192,64], b [192]] or []: the attention projections fused into the last node kernel; QKV is an empty
    tensor when they were not computed (no ``qkv``, or the fp32 mode's SIMT node kernels)."""
    g = _graph_ns(graph, n_edges, n_graphs, max_nodes)
    pl = [[t.contiguous() for t in params[11 * l:11 * l + 11]] for l in range(n_layers)]
    keep: list = []
    res = IF._egnn_stack_forward(g, x23, edge_attr.contiguous(), pl, False, keep,
                                 tuple(t.contiguous() for t in qkv) if qkv else None)
    h, QKV = res if qkv else (res, None)
    out = [h, x23.new_empty(0) if QKV is None else QKV]
    for hl, xl, pq, hn in keep:
        out += [hl.contiguous(), xl.contiguous(), pq, hn]       # (layer 0's h / x are strided views of x23)
    return out


@egnn_stack.register_fake
def _(x23, edge_attr, params, graph, n_layers, n_edges, n_graphs, max_nodes, qkv):
    n = x23.shape[0]
    fused = bool(qkv) and IF.get_precision() != "fp32"
    out = [x23.new_empty(n, H), x23.new_empty(n, 3 * H) if fused else x23.new_empty(0)]
    for l in range(n_layers):
        out += [x23.new_empty(n, 20 if l == 0 else H), x23.new_empty(n, 3), x23.new_empty(n, 2 * H), x23.new_empty(n, H)]
    return out


@torch.library.custom_op("immunostruct_b200::egnn_stack_bwd", mutates_args=())
def egnn_stack_bwd(gh: Tensor, edge_attr: Tensor, saved: List[Tensor], params: List[Tensor], graph: List[Tensor],
                   n_layers: int, n_edges: int, n_graphs: int, max_nodes: int, need_x23: bool,
                   need_edge_attr: bool) -> List[Tensor]:
    """-> 11 * n_layers parameter gradients (an empty tensor where the reference reports None: the last layer's coord_mlp),
    then the gradients of x23 [N, 23] and of edge_attr (empty tensors where not requested)"""
    g = _graph_ns(graph, n_edges, n_graphs, max_nodes)
    edge_attr = edge_attr.contiguous()
    grads: list = [None] * (11 * n_layers)
    gx = None
    g_attr = torch.empty_like(edge_attr) if need_edge_attr else None
    for l in range(n_layers - 1, -1, -1):
        hl, xl, pq, hn = saved[4 * l:4 * l + 4]
        pl = [t.contiguous() for t in params[11 * l:11 * l + 11]]
        need = l > 0 or need_x23
        gh, gx_in, gl = IF._egnn_layer_backward(g, hl, xl, edge_attr, pq, hn, pl, gh, gx, need, need, g_attr,
                                                l != n_layers - 1)
        grads[11 * l:11 * l + 11] = gl
        gx = gx_in
    # (the per-layer gradients are views of three reduction buffers, and registered operators may not return aliases --
    #  not even the same empty tensor twice)
    out = [edge_attr.new_empty(0) if t is None else t.clone() for t in grads]
    return out + [torch.cat([gh, gx], 1) if need_x23 else edge_attr.new_empty(0),
                  g_attr if need_edge_attr else edge_attr.new_empty(0)]


@egnn_stack_bwd.register_fake
def _(gh, edge_attr, saved, params, graph, n_layers, n_edges, n_graphs, max_nodes, need_x23, need_edge_attr):
    out = [torch.empty_like(p) for p in params]
    for i in (4, 5, 6):                                  # the last layer's coord_mlp: no gradient
        out[11 * (n_layers - 1) + i] = gh.new_empty(0)
    return out + [gh.new_empty(gh.shape[0], 23) if need_x23 else gh.new_empty(0),
                  torch.empty_like(edge_attr, memory_format=torch.contiguous_format) if need_edge_attr else gh.new_empty(0)]


def _egnn_setup(ctx, inputs, output):
    x23, edge_attr, params, graph, n_layers, n_edges, n_graphs, max_nodes, qkv = inputs
    ctx.cfg = (n_layers, n_edges, n_graphs, max_nodes)
    ctx.n_params, ctx.n_graph, ctx.n_qkv = len(params), len(graph), len(qkv)
    ctx.has_qkv = bool(qkv) and output[1].numel() > 0
    ctx.set_materialize_grads(False)
    ctx.save_for_backward(edge_attr, *output[2:], *params, *graph, *((output[0], qkv[0]) if ctx.has_qkv else ()))


def _egnn_backward(ctx, grads):
    n_layers = ctx.cfg[0]
    t = ctx.saved_tensors
    edge_attr, saved = t[0], list(t[1:1 + 4 * n_layers])
    params = list(t[1 + 4 * n_layers:1 + 4 * n_layers + ctx.n_params])
    graph = list(t[1 + 4 * n_layers + ctx.n_params:1 + 4 * n_layers + ctx.n_params + ctx.n_graph])
    gh, gqkv = grads[0], grads[1]
    g_qkv_in = [None] * ctx.n_qkv
    if ctx.has_qkv and gqkv is not None:                 # same arithmetic as functional._EGNNStack.backward
        ghq, gw, gb = IF._qkv_backward(ctx.cfg[2], ctx.cfg[3], t[-2], t[-1], gqkv)
        gh = ghq if gh is None else gh + ghq
        g_qkv_in = [gw, gb]
    if gh is None:
        return None, None, [None] * ctx.n_params, [None] * ctx.n_graph, None, None, None, None, g_qkv_in
    need_x23, need_attr = ctx.needs_input_grad[0], ctx.needs_input_grad[1]
    gp = egnn_stack_bwd(gh.contiguous(), edge_attr, saved, params, graph, *ctx.cfg, need_x23, need_attr)
    gp, gx23, g_attr = gp[:ctx.n_params], gp[-2], gp[-1]
    return (gx23 if need_x23 else None, g_attr if need_attr else None,
            [None if g.numel() == 0 and p.numel() != 0 else g for g, p in zip(gp, params)], [None] * ctx.n_graph,
            None, None, None, None, g_qkv_in)


egnn_stack.register_autograd(_egnn_backward, setup_context=_egnn_setup)


# ---- routing switch ----------------------------------------------------------------------------------------
_enabled = False


def use_custom_ops(flag: bool = True) -> None:
    """Route the model classes' fused calls through the registered ``torch.ops.immunostruct_b200.*`` operators."""
    global _enabled
    _enabled = bool(flag)


def enabled() -> bool:
    return _enabled
