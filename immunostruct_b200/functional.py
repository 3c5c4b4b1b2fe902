"""Differentiable host wrappers around the C-ABI kernels (``torch.autograd.Function`` per fused op).

Nothing here computes on the host: each ``forward`` / ``backward`` allocates outputs with torch and
enqueues kernels through ``immunostruct_b200._C``.  Gradients are deterministic (fixed-order
reductions; per-CTA partials summed in CTA order by ``is_reduce_partials``).
"""
from __future__ import annotations

import os

import torch

from . import _C

H = 64   # hidden width of the EGNN MLPs and of the node embedding (hybrid_models.py:247)


# Arithmetic of the EGNN GEMMs.  Forward modes below; the edge BACKWARD runs on the tensor cores with the
# fp32-accurate bf16x3 split in every mode except "fp32" (which keeps the fp32 SIMT backward):
#   "fp32"   : fp32 SIMT FMA kernels (csrc/egnn.cu)
#   "bf16x3" : tcgen05 tensor cores, operands split into three bf16 terms, six partial products --
#              fp32-accurate (csrc/egnn_tc2.cu); what training runs in every tensor-core mode but "bf16"
#   "tf32x3" : tcgen05 tensor cores with the 3xTF32 split -- fp32-accurate, one 512-thread CTA per SM
#   "bf16"   : tcgen05 tensor cores, bf16 operands, fp32 accumulate, fast SiLU (1e-2 tolerance mode)
#   "fp16x2" : THE DEFAULT.  The EGNN stack and the attention scores of the NO-GRAD forward on fp16 hi / lo operand pairs
#              (fp32-accurate to 2^-22, two thirds of the operand bytes and half the MMAs of "bf16x3"; activations beyond
#              +-65504 overflow to inf / NaN) -- everything else (training forward and backward, the dense layers) runs as
#              in "bf16x3"
_PRECISIONS = {"fp32": None, "bf16x3": _C.PREC_BF16X3, "tf32x3": _C.PREC_TF32X3, "bf16": _C.PREC_BF16, "fp16x2": _C.PREC_FP16X2}
_precision = "fp16x2"


def set_precision(name: str) -> None:
    global _precision
    if name not in _PRECISIONS:
        raise ValueError(f"precision must be one of {sorted(_PRECISIONS)}")
    _precision = name


def get_precision() -> str:
    return _precision


# Tile streams of the tensor-core edge backward: 2 = csrc/egnn_bwd_ws.cu (two 112-edge tiles in flight per SM; batches
# with a node of more than 112 in-edges fall through to the lock-step kernel on the device), 1 = the lock-step
# kernel of csrc/egnn_bwd_tc.cu only (A/B timing).
_edge_bwd_streams = int(os.environ.get("IS_EDGE_BWD_STREAMS", "2"))


def set_edge_bwd_streams(n: int) -> None:
    global _edge_bwd_streams
    if n not in (1, 2):
        raise ValueError("edge backward tile streams: 1 or 2")
    _edge_bwd_streams = n


# Generation counter of every parameter-derived cache (fused projection weights, fusion coefficients, pre-split weight
# planes).  The caches are keyed on (storage pointer, in-place version counter) of their source parameters, which
# misses writes through ``p.data`` (EMA, clipping, legacy init code: they do not bump the version counter); model
# ``train()`` / ``load_state_dict()`` / ``to()`` bump this generation, and ``invalidate_caches()`` does so explicitly.
_cache_generation = 0


def invalidate_caches() -> None:
    """Drop every cached parameter-derived tensor (call after writing parameters through ``.data``)."""
    global _cache_generation
    _cache_generation += 1
    _weight_planes.clear()


def cache_generation() -> int:
    return _cache_generation


def _ops():
    """The torch.library registration (ops.py), when routing through it has been switched on; else None."""
    from . import ops
    return ops if ops.enabled() else None


def _new(like, *shape):
    return torch.empty(*shape, dtype=torch.float32, device=like.device)


# ==================================================================================================
# EGNN layer
# ==================================================================================================
class _EGNNLayer(torch.autograd.Function):
    """dgl.nn.EGNNConv.forward (reference call site models/hybrid_models.py:89-90 / :323-324).

    forward(graph, update_coords, h, x, edge_attr, W1, b1, W2, b2, W3, b3, w4, W5, b5, W6, b6)
      -> (h_out [N,64], x_out [N,3] or None when ``update_coords`` is False)
    The per-edge activations are NOT saved; the backward recomputes them tile by tile.
    """

    @staticmethod
    def forward(ctx, graph, update_coords, h, x, edge_attr, W1, b1, W2, b2, W3, b3, w4, W5, b5, W6, b6):
        n, f = h.shape
        if W2.shape != (H, H) or W6.shape != (H, H) or W1.shape != (H, 2 * f + 2) or W5.shape != (H, f + H):
            raise NotImplementedError("EGNN kernels are specialised for hidden = out = 64 and edge_feat_size = 1")
        params = [t.contiguous() for t in (W1, b1, W2, b2, W3, b3, w4, W5, b5, W6, b6)]
        W1, b1, W2, b2, W3, b3, w4, W5, b5, W6, b6 = params
        edge_attr = edge_attr.contiguous()
        PQ, hn, h_out = _new(h, n, 2 * H), _new(h, n, H), _new(h, n, H)
        x_out = _new(h, n, 3) if update_coords else None
        _C.egnn_node_pre_fwd(h, W1, b1, PQ)
        prec = _PRECISIONS[_precision]
        if prec == _C.PREC_FP16X2:
            prec = _C.PREC_BF16X3              # (an autograd forward: see _PRECISIONS)
        if prec is None:
            _C.egnn_edge_fwd(graph, PQ, x, edge_attr, f, W1, W2, b2, W3, b3, w4, update_coords, hn, x_out)
        else:
            _C.egnn_edge_fwd_tc(graph, PQ, x, edge_attr, f, W1, W2, b2, W3, b3, w4, update_coords, prec, hn, x_out)
        _C.egnn_node_post_fwd(h, hn, W5, b5, W6, b6, h_out)
        ctx.graph = graph
        ctx.update_coords = update_coords
        ctx.save_for_backward(h, x, edge_attr, PQ, hn, *params)
        ctx.set_materialize_grads(False)
        return h_out, x_out

    @staticmethod
    def backward(ctx, gh_out, gx_out):
        h, x, edge_attr, PQ, hn, *params = ctx.saved_tensors
        has_coord = ctx.update_coords and gx_out is not None
        g_attr = _new(edge_attr, *edge_attr.shape) if ctx.needs_input_grad[4] else None
        gh, gx, grads = _egnn_layer_backward(ctx.graph, h, x, edge_attr, PQ, hn, params, gh_out,
                                             gx_out if has_coord else None, ctx.needs_input_grad[2],
                                             ctx.needs_input_grad[3], g_attr)
        return (None, None, gh, gx, g_attr, *grads)


def _egnn_layer_backward(g, h, x, edge_attr, PQ, hn, params, gh_out, gx_out, need_gh, need_gx, g_attr=None,
                         attr_accumulate=False):
    """Backward of one EGNN layer from its saved inputs: node_post_bwd -> edge_bwd -> node_pre_bwd ->
    deterministic reduction of the per-CTA partials.  ``gx_out`` None = the layer's coordinate output
    received no gradient (coord_mlp then gets NO gradient: None, as in the reference).  ``gh`` is [N, F] (F = 20 for
    the input layer).  ``g_attr`` (or None): buffer of the edge-feature gradient [E] or [E, 1], written (or, with
    ``attr_accumulate``, added to) from the layer's edge pre-activation gradient.
    Returns (gh or None, gx or None, 11 parameter gradients)."""
    W1, b1, W2, b2, W3, b3, w4, W5, b5, W6, b6 = params
    n, f = h.shape
    e = g.n_edges
    k = f + H
    if gh_out is None:
        gh_out = torch.zeros(n, H, dtype=torch.float32, device=h.device)
    gh_out = gh_out.contiguous()
    has_coord = gx_out is not None
    if has_coord:
        gx_out = gx_out.contiguous()
    grid_n, grid_e = _C.egnn_node_grid(n), _C.egnn_edge_bwd_grid(n)
    # node_post backward
    ghn = _new(h, n, H)
    gh_direct = _new(h, n, f) if need_gh else None
    p_post = _new(h, grid_n, H * k + H + H * H + H)
    tc = _PRECISIONS[_precision] is not None          # tensor-core (bf16x3) backward kernels in every mode but "fp32"
    (_C.egnn_node_post_bwd_tc if tc else _C.egnn_node_post_bwd)(gh_out, h, hn, W5, b5, W6, gh_direct, ghn, p_post)
    # edge backward
    gz1, gQ, gD, gxd = _new(h, e, H), _new(h, n, H), _new(h, e, 3), _new(h, n, 3)
    p_edge = _new(h, grid_e, 2 * H * H + 5 * H)
    bwd = _C.egnn_edge_bwd if _PRECISIONS[_precision] is None else (_C.egnn_edge_bwd_ws if _edge_bwd_streams == 2 else _C.egnn_edge_bwd_tc)
    bwd(g, PQ, x, edge_attr, f, W1, W2, b2, W3, b3, w4, ghn, gx_out, gz1, gQ, gD, gxd, p_edge)
    # node_pre backward (source-side reduction through the CSC transpose)
    gh = _new(h, n, f) if need_gh else None
    gx = _new(h, n, 3) if need_gx else None
    p_pre = _new(h, grid_n, 2 * H * f + H)
    (_C.egnn_node_pre_bwd_tc if tc else _C.egnn_node_pre_bwd)(gz1, gQ, gD, gxd, gx_out, gh_direct, g, h, W1, gh, gx, p_pre)
    if g_attr is not None:
        _C.egnn_edge_attr_grad(gz1, g, W1, f, g_attr, attr_accumulate)
    # deterministic reduction of the per-CTA weight-gradient partials
    r_post, r_edge, r_pre = _new(h, p_post.shape[1]), _new(h, p_edge.shape[1]), _new(h, p_pre.shape[1])
    _C.reduce_partials3((p_post, p_edge, p_pre), (r_post, r_edge, r_pre))

    gW5 = r_post[:H * k].view(H, k)
    gb5 = r_post[H * k:H * k + H]
    gW6 = r_post[H * k + H:H * k + H + H * H].view(H, H)
    gb6 = r_post[H * k + H + H * H:]
    gW2 = r_edge[:H * H].view(H, H)
    gb2 = r_edge[2 * H * H:2 * H * H + H]
    gwr = r_edge[2 * H * H + 3 * H:2 * H * H + 4 * H]
    gwa = r_edge[2 * H * H + 4 * H:2 * H * H + 5 * H]
    if has_coord:
        gW3 = r_edge[H * H:2 * H * H].view(H, H)
        gb3 = r_edge[2 * H * H + H:2 * H * H + 2 * H]
        gw4 = r_edge[2 * H * H + 2 * H:2 * H * H + 3 * H].view(1, H)
    else:
        gW3 = gb3 = gw4 = None            # coord_mlp never influenced the loss: report NO gradient
    gWs = r_pre[:H * f].view(H, f)
    gWd = r_pre[H * f:2 * H * f].view(H, f)
    gb1 = r_pre[2 * H * f:]
    gW1 = torch.cat([gWs, gWd, gwr.unsqueeze(1), gwa.unsqueeze(1)], dim=1)
    return gh, gx, (gW1, gb1, gW2, gb2, gW3, gb3, gw4, gW5, gb5, gW6, gb6)


def _egnn_stack_forward(graph, x23, edge_attr, params, fast_act, keep, qkv=None):
    """Shared forward of the EGNN stack.  ``keep``: list that receives (h, x, PQ, hn) per layer for the
    backward pass (None = inference, nothing kept).  ``qkv`` = (W [192,64], b [192]): the attention projections
    that follow the stack, fused into the last node kernel when it runs on the tensor cores; the function then
    returns (h, QKV [N,192] or None)."""
    h, x = x23[:, :20], x23[:, 20:]
    n = h.shape[0]
    prec = _PRECISIONS[_precision]
    if prec == _C.PREC_FP16X2 and keep is not None:
        prec = _C.PREC_BF16X3                  # training: the backward kernels recompute the forward in the bf16x3 split
    node_prec = {None: None, _C.PREC_BF16: _C.PREC_BF16, _C.PREC_TF32X3: _C.PREC_BF16X3, _C.PREC_BF16X3: _C.PREC_BF16X3,
                 _C.PREC_FP16X2: _C.PREC_FP16X2}[prec]
    # (training forward: the fused tensor-core node kernel with the accurate SiLU and all eight bf16x3 partial
    #  products, fast_act = False -- with six products a handful of parameter gradients landed at 1.0-1.3e-5 of
    #  their scale on the B200, just outside the 1e-5 gradient tolerance)
    PQ = _new(h, n, 2 * H)
    QKV = None
    _C.egnn_node_pre_fwd(h, params[0][0], params[0][1], PQ)
    last = len(params) - 1
    for l, (W1, b1, W2, b2, W3, b3, w4, W5, b5, W6, b6) in enumerate(params):
        f = h.shape[1]
        upd = l != last
        hn, h_out = _new(h, n, H), _new(h, n, H)
        x_out = _new(h, n, 3) if upd else None
        if prec is None:
            _C.egnn_edge_fwd(graph, PQ, x, edge_attr, f, W1, W2, b2, W3, b3, w4, upd, hn, x_out)
        else:
            _C.egnn_edge_fwd_tc(graph, PQ, x, edge_attr, f, W1, W2, b2, W3, b3, w4, upd, prec, hn, x_out,
                                fast_act=fast_act)
        nxt = params[l + 1] if upd else None
        PQ_next = _new(h, n, 2 * H) if upd else None
        if node_prec is None:
            _C.egnn_node_post_fwd(h, hn, W5, b5, W6, b6, h_out)
            if upd:
                _C.egnn_node_pre_fwd(h_out, nxt[0], nxt[1], PQ_next)
        elif not upd and qkv is not None:
            QKV = _new(h, n, 3 * H)
            _C.egnn_node_post_pre_tc(h, hn, W5, b5, W6, b6, h_out, qkv[0], qkv[1], QKV, node_prec,
                                     fast_act=fast_act, next_kind=2)
        else:
            _C.egnn_node_post_pre_tc(h, hn, W5, b5, W6, b6, h_out, nxt[0] if upd else None,
                                     nxt[1] if upd else None, PQ_next, node_prec, fast_act=fast_act)
        if keep is not None:
            keep.append((h, x, PQ, hn))
        h, PQ = h_out, PQ_next
        if upd:
            x = x_out
    return h if qkv is None else (h, QKV)


def _qkv_backward(n_graphs, max_nodes, h_fin, w, gqkv, need_w=True, need_b=True):
    """Backward of ``QKV = h' W^T + b`` over all node rows of the batch -> (gh', gW, gb).  Equal node counts per graph (the
    reference's own assumption, hybrid_models.py:86-92): the weight / bias gradients are per-graph partial products (one
    batched GEMM, [B, out, K]) summed over the graphs in a fixed order -- a tenth of the time of autograd's single long-K
    GEMM (K = 102 400 at batch 512) and column reduction."""
    gqkv = gqkv.contiguous()
    ghq = gqkv @ w
    if n_graphs * max_nodes == h_fin.shape[0]:
        g3, h3 = gqkv.reshape(n_graphs, -1, gqkv.shape[1]), h_fin.reshape(n_graphs, -1, h_fin.shape[1])
        gw = torch.bmm(g3.transpose(1, 2), h3).sum(0) if need_w else None
        gb = g3.sum(1).sum(0) if need_b else None
    else:
        gw = gqkv.t() @ h_fin if need_w else None
        gb = gqkv.sum(0) if need_b else None
    return ghq, gw, gb


class _EGNNStack(torch.autograd.Function):
    """The whole ``for layer in self.GCN_layers`` loop (models/hybrid_models.py:89-90) as ONE autograd node:
    forward through the fused kernels (node side fused across layer boundaries on the tensor cores), backward
    layer by layer in reverse.  The last layer's coordinate branch is skipped, so its coord_mlp parameters get
    ``None`` gradients exactly as in the reference.  Input gradients, as DGL's autograd gives them: ``x23`` [N, 23]
    (residue features and coordinates) when it requires grad, ``edge_attr`` (summed over the layers) when it does;
    neither costs anything when not requested.

    forward(graph, n_layers, x23, edge_attr, qkv_w, qkv_b, *flat_params) -> (h_final [N,64], QKV [N,192] or None)

    ``qkv_w`` [192,64] / ``qkv_b`` [192] (or None): the attention projections that follow the stack
    (models/layers.py:13-16 / :67-69).  They ride in the last node kernel exactly as in inference (h' is still on chip:
    +27 us instead of a 0.17 ms cuBLAS SIMT GEMM + bias kernel over 102 400 rows); their backward -- h' gets
    ``gQKV W``, the weight / bias gradients are per-graph partial products summed in a fixed order -- runs here, before the
    layer loop.  QKV is None when the node side runs on the SIMT kernels (fp32 mode): the caller projects itself.
    """

    @staticmethod
    def forward(ctx, graph, n_layers, x23, edge_attr, qkv_w, qkv_b, *flat):
        params = [[t.contiguous() for t in flat[11 * l:11 * l + 11]] for l in range(n_layers)]
        edge_attr = edge_attr.contiguous()
        keep = []
        qkv = None if qkv_w is None else (qkv_w.contiguous(), qkv_b.contiguous())
        out = _egnn_stack_forward(graph, x23, edge_attr, params, False, keep, qkv)
        h, QKV = out if qkv is not None else (out, None)
        ctx.graph, ctx.n_layers, ctx.has_qkv = graph, n_layers, QKV is not None
        ctx.set_materialize_grads(False)
        saved = [edge_attr]
        for (hl, xl, PQl, hnl), pl in zip(keep, params):
            saved += [hl, xl, PQl, hnl, *pl]
        if QKV is not None:
            saved += [h, qkv[0]]
        ctx.save_for_backward(*saved)
        return h, QKV

    @staticmethod
    def backward(ctx, gh, gqkv):
        saved = ctx.saved_tensors
        edge_attr = saved[0]
        nl = ctx.n_layers
        grads = [None] * (11 * nl)
        gw = gb = None
        if ctx.has_qkv and gqkv is not None:
            ghq, gw, gb = _qkv_backward(ctx.graph.n_graphs, int(ctx.graph.max_nodes), saved[-2], saved[-1], gqkv,
                                        ctx.needs_input_grad[4], ctx.needs_input_grad[5])
            gh = ghq if gh is None else gh + ghq
        if gh is None:
            return (None,) * (6 + 11 * nl)
        gh = gh.contiguous()
        gx = None
        need_x23 = ctx.needs_input_grad[2]
        g_attr = _new(edge_attr, *edge_attr.shape) if ctx.needs_input_grad[3] else None
        for l in range(nl - 1, -1, -1):
            hl, xl, PQl, hnl, *pl = saved[1 + 15 * l:1 + 15 * (l + 1)]
            need = l > 0 or need_x23
            gh, gx_in, gl = _egnn_layer_backward(ctx.graph, hl, xl, edge_attr, PQl, hnl, pl, gh, gx, need, need, g_attr,
                                                 l != nl - 1)
            grads[11 * l:11 * l + 11] = gl
            gx = gx_in
        gx23 = torch.cat([gh, gx], 1) if need_x23 else None
        return (None, None, gx23, g_attr, gw, gb, *grads)


def egnn_stack(graph, x23, edge_attr, layer_params, qkv=None):
    """EGNN stack with autograd (training).  ``layer_params``: list of EGNNConv.kernel_params() tuples.  Returns the final
    h [N,64]; with ``qkv`` = (W [192,64], b [192]) (differentiable) returns (h, QKV [N,192]) with the projections fused
    into the last node kernel -- QKV is None where that kernel does not run (fp32 mode, registered-operator route)."""
    flat = [t for lp in layer_params for t in lp]
    ops = _ops()
    if ops is not None:
        out = ops.egnn_stack(x23, edge_attr, flat, ops.graph_tensors(graph), len(layer_params), graph.n_edges, graph.n_graphs,
                             int(graph.max_nodes), [] if qkv is None else list(qkv))
        return out[0] if qkv is None else (out[0], out[1] if out[1].numel() else None)
    if qkv is None:
        return _EGNNStack.apply(graph, len(layer_params), x23, edge_attr, None, None, *flat)[0]
    return _EGNNStack.apply(graph, len(layer_params), x23, edge_attr, qkv[0], qkv[1], *flat)


def egnn_stack_infer(graph, x23, edge_attr, layer_params, qkv=None):
    """No-grad EGNN stack (models/hybrid_models.py:82,89-90): node_pre(0) -> [edge(l) -> node_post(l) +
    node_pre(l+1)]; the last layer's coordinate branch is skipped (its output is never consumed).  In the
    tensor-core precisions the node side runs fused across the layer boundary (csrc/egnn_node_tc.cu).
    ``layer_params``: list of the 11-tuples of EGNNConv.kernel_params().  Returns the final h [N,64]; with
    ``qkv`` = (W [192,64], b [192]) returns (h, QKV [N,192]) -- QKV is None when the node side runs on the SIMT
    kernels (fp32 mode) and the caller applies the projection itself."""
    params = [[t.detach().contiguous() for t in lp] for lp in layer_params]
    if qkv is not None:
        qkv = tuple(t.detach().contiguous() for t in qkv)
    return _egnn_stack_forward(graph, x23, edge_attr.contiguous(), params, True, None, qkv)


def egnn_layer(graph, h, x, edge_attr, params, update_coords=True):
    """params = (W1, b1, W2, b2, W3, b3, w4, W5, b5, W6, b6); returns (h_out, x_out|None)."""
    return _EGNNLayer.apply(graph, update_coords, h, x, edge_attr, *params)


# ==================================================================================================
# per-graph attention + mean pool
# ==================================================================================================
class _AttnPool(torch.autograd.Function):
    """softmax(QK^T/sqrt(d)) V per graph and head, plus the per-graph mean of the rows.

    forward(graph, n_head, want_attn, want_nodes, QKV [N,192]) -> (O [N,64] or None, pooled [B,64], attn or None)
    ``attn`` is the dense weights tensor [B, H, n, n] (equal node counts) when requested.  When only the pooled rows
    are wanted (every model's training path) and the arithmetic mode is a tensor-core one, the forward is the
    pooled-rows-only tcgen05 kernel (csrc/attn_pool_tc.cu) and nothing but QKV is saved: the backward
    (csrc/attn_pool_bwd_tc.cu) recomputes the scores and their row statistics on the tensor cores.
    """

    @staticmethod
    def forward(ctx, graph, n_head, want_attn, want_nodes, QKV):
        QKV = QKV.contiguous()
        n = QKV.shape[0]
        b = graph.n_graphs
        ctx.graph, ctx.n_head = graph, n_head
        ctx.set_materialize_grads(False)
        prec = _PRECISIONS[_precision]
        if not want_attn and not want_nodes and n_head == 1 and prec is not None and graph.max_nodes <= 256:
            pooled = _new(QKV, b, H)
            # (fp16x2: the no-grad forward only -- the backward kernel recomputes the scores in the bf16x3 split)
            fwd_only = prec == _C.PREC_FP16X2 and not ctx.needs_input_grad[4]
            _C.attn_pool_infer_tc(QKV, graph.node_off, graph.max_nodes, pooled,
                                  _C.PREC_BF16 if prec == _C.PREC_BF16 else _C.PREC_FP16X2 if fwd_only else _C.PREC_BF16X3)
            ctx.pooled_only = True
            ctx.save_for_backward(QKV)
            return None, pooled, None
        O, LSE, pooled = _new(QKV, n, H), _new(QKV, n, n_head), _new(QKV, b, H)
        attn = attn_off = None
        if want_attn:
            m = graph.max_nodes
            if m * b != n:
                raise NotImplementedError("return_attention needs equal node counts per graph (as the reference does)")
            attn = _new(QKV, b, n_head, m, m)
            attn_off = torch.arange(b, device=QKV.device, dtype=torch.int64) * (n_head * m * m)
        _C.attn_pool_fwd(QKV, graph.node_off, n_head, graph.max_nodes, O, LSE, pooled, attn, attn_off)
        ctx.pooled_only = False
        ctx.save_for_backward(QKV, O, LSE)
        if want_attn:
            ctx.mark_non_differentiable(attn)
        return O, pooled, attn

    @staticmethod
    def backward(ctx, gO, g_pooled, _g_attn):
        if ctx.pooled_only:
            (QKV,) = ctx.saved_tensors
            gQKV = _new(QKV, *QKV.shape)
            if g_pooled is None:
                gQKV.zero_()
                return None, None, None, None, gQKV
            # row statistics, both score products and the two gradient products on the tensor cores (bf16x3)
            _C.attn_pool_bwd_tc(QKV, ctx.graph.node_off, ctx.graph.max_nodes, g_pooled.contiguous(), gQKV)
            return None, None, None, None, gQKV
        QKV, O, LSE = ctx.saved_tensors
        gQKV = _new(QKV, *QKV.shape)
        if gO is None and g_pooled is None:
            gQKV.zero_()
            return None, None, None, None, gQKV
        gO = gO.contiguous() if gO is not None else None
        g_pooled = g_pooled.contiguous() if g_pooled is not None else None
        _C.attn_pool_bwd(QKV, O, LSE, ctx.graph.node_off, ctx.n_head, ctx.graph.max_nodes, g_pooled, gO, gQKV)
        return None, None, None, None, gQKV


def attention_pool(graph, QKV, n_head=1, want_attn=False, want_nodes=False):
    """-> (O [N,64] or None, pooled [B,64], attention weights or None).  Without autograd and when only
    the pooled rows are wanted, the inference kernel (column sums of P, no P V product) is used."""
    if not want_attn and not want_nodes and not (torch.is_grad_enabled() and QKV.requires_grad):
        QKV = QKV.contiguous()
        pooled = _new(QKV, graph.n_graphs, H)
        prec = _PRECISIONS[_precision]
        if n_head == 1 and prec is not None and graph.max_nodes <= 256:
            # single head: Q K^T on the tensor cores, softmax statistics straight from TMEM (csrc/attn_pool_tc.cu)
            _C.attn_pool_infer_tc(QKV, graph.node_off, graph.max_nodes, pooled,
                                  prec if prec in (_C.PREC_BF16, _C.PREC_FP16X2) else _C.PREC_BF16X3)
        else:
            _C.attn_pool_infer(QKV, graph.node_off, n_head, graph.max_nodes, pooled)
        return None, pooled, None
    ops = _ops()
    if ops is not None and not want_attn and not want_nodes:
        return None, ops.attention_pool(QKV, graph.node_off, n_head, int(graph.max_nodes)), None
    return _AttnPool.apply(graph, n_head, want_attn, want_nodes, QKV)


# ==================================================================================================
# fusion attention (closed form)
# ==================================================================================================
class _FusionAttn(torch.autograd.Function):
    """out[b,i] = btilde + sum_h (alpha_h E^h_i + beta_h); see csrc/fusion.cu.  coef = [A|C|alpha|beta|btilde]."""

    @staticmethod
    def forward(ctx, c, coef, n_head):
        c, coef = c.contiguous(), coef.contiguous()
        out = _new(c, *c.shape)
        _C.fusion_attn_fwd(c, n_head, coef, out)
        ctx.n_head = n_head
        ctx.save_for_backward(c, coef)
        return out

    @staticmethod
    def backward(ctx, gout):
        c, coef = ctx.saved_tensors
        hh = ctx.n_head
        gout = gout.contiguous()
        gc, part = _new(c, *c.shape), _new(c, c.shape[0], 4 * hh)
        _C.fusion_attn_bwd(c, hh, coef, gout, gc, part)
        gcoef = torch.cat([part.sum(0), gout.sum().reshape(1)])
        return gc, gcoef, None


def fusion_attention(c, coef, n_head):
    ops = _ops()
    if ops is not None:
        return ops.fusion_attention(c, coef, n_head)
    return _FusionAttn.apply(c, coef, n_head)


# ==================================================================================================
# fused loss
# ==================================================================================================
class _FusedLoss(torch.autograd.Function):
    """w_pred * pred(out, y) + w_mse * MSE(recon, seq) + w_kld * KLD(mu, logvar)  (utils/loss.py:13-31)."""

    @staticmethod
    def forward(ctx, recon, seq, mu, logvar, logits, y, mode, pos_weight, w_pred, w_mse, w_kld):
        ctx.logits_shape = logits.shape
        logits = logits.reshape(-1).contiguous()
        y = y.reshape(-1).contiguous().float()
        if logits.numel() != y.numel():
            raise ValueError("prediction and target must have the same number of elements")
        if w_mse != 0.0 or w_kld != 0.0:
            recon, seq = recon.contiguous(), seq.reshape(recon.shape[0], -1).contiguous()
            if recon.shape != seq.shape:
                raise ValueError(f"recon {tuple(recon.shape)} vs sequence {tuple(seq.shape)}")
            mu, logvar = mu.contiguous(), logvar.contiguous()
        else:
            recon = seq = mu = logvar = None
        out = _new(logits, 4)
        partial = _new(logits, _C.loss_num_partials())
        _C.loss_fwd(recon, seq, mu, logvar, logits, y, mode, pos_weight, w_pred, w_mse, w_kld, partial, out)
        ctx.cfg = (mode, pos_weight, w_pred, w_mse, w_kld)
        ctx.has_seq = recon is not None
        saved = (logits, y) + ((recon, seq, mu, logvar) if recon is not None else ())
        ctx.save_for_backward(*saved)
        ctx.mark_non_differentiable(out)
        return out[0].clone(), out

    @staticmethod
    def backward(ctx, gout, _gcomp):
        mode, pos_weight, w_pred, w_mse, w_kld = ctx.cfg
        if ctx.has_seq:
            logits, y, recon, seq, mu, logvar = ctx.saved_tensors
            g_recon, g_mu, g_lv = _new(recon, *recon.shape), _new(mu, *mu.shape), _new(mu, *mu.shape)
        else:
            logits, y = ctx.saved_tensors
            recon = seq = mu = logvar = g_recon = g_mu = g_lv = None
        g_logits = _new(logits, logits.numel())
        gout = gout.reshape(1).contiguous().float()
        _C.loss_bwd(recon, seq, mu, logvar, logits, y, mode, pos_weight, w_pred, w_mse, w_kld, gout,
                    g_recon, g_mu, g_lv, g_logits)
        return g_recon, None, g_mu, g_lv, g_logits.view(ctx.logits_shape), None, None, None, None, None, None


def fused_loss(recon, seq, mu, logvar, logits, y, mode, pos_weight, w_pred, w_mse, w_kld, return_components=False):
    ops = _ops()
    if ops is not None:
        if w_mse == 0.0 and w_kld == 0.0:
            recon = seq = mu = logvar = None
        comps = ops.fused_loss(recon, seq, mu, logvar, logits, y, int(mode), float(pos_weight), float(w_pred), float(w_mse),
                               float(w_kld))
        return (comps[0], comps.detach()) if return_components else comps[0]
    total, comps = _FusedLoss.apply(recon, seq, mu, logvar, logits, y, int(mode), float(pos_weight),
                                    float(w_pred), float(w_mse), float(w_kld))
    return (total, comps) if return_components else total


# ==================================================================================================
# segment pooling (global_mean_pool / global_max_pool)
# ==================================================================================================
class _SegmentPool(torch.autograd.Function):
    """torch_geometric.nn.global_{mean,max}_pool over the batch's node segments (models/hybrid_models.py:97,331;
    models/ablation_models.py:296-297) -- csrc/segment_pool.cu."""

    @staticmethod
    def forward(ctx, X, node_off, mode):
        X = X if X.stride(-1) == 1 else X.contiguous()
        out = _new(X, node_off.numel() - 1, X.shape[1])
        _C.segment_pool_fwd(X, node_off, mode, out)
        ctx.mode = mode
        ctx.save_for_backward(X, node_off, out)
        return out

    @staticmethod
    def backward(ctx, g_out):
        X, node_off, out = ctx.saved_tensors
        gX = _new(X, *X.shape)
        _C.segment_pool_bwd(X, node_off, ctx.mode, out, g_out.contiguous(), gX)
        return gX, None, None


def segment_pool(graph_or_offsets, X, mode="mean"):
    """Per-graph mean / max / sum of the rows of X [N, C] -> [B, C]; segments = the batch's node offsets."""
    node_off = getattr(graph_or_offsets, "node_off", graph_or_offsets)
    if mode not in _C.POOL_MODES:
        raise ValueError(f"mode must be one of {sorted(_C.POOL_MODES)}")
    ops = _ops()
    if ops is not None:
        return ops.segment_pool(X, node_off, mode)
    return _SegmentPool.apply(X, node_off, mode)


# ==================================================================================================
# paired contrastive loss
# ==================================================================================================
class _Contrastive(torch.autograd.Function):
    """PairedContrastiveLoss.forward (utils/contrastive.py:37-83) -- csrc/contrastive.cu.

    forward(Ec, Ew, target, W1, gamma, beta, W2, run_mean, run_var, n_tracked, bn_eps, momentum, lambda_off) -> loss"""

    @staticmethod
    def forward(ctx, Ec, Ew, target, W1, gamma, beta, W2, run_mean, run_var, n_tracked, bn_eps, momentum, lambda_off):
        Ec, Ew, W1, gamma, beta, W2 = (t.contiguous() for t in (Ec, Ew, W1, gamma, beta, W2))
        target = target.reshape(-1).float().contiguous()
        b, z = Ec.shape[0], W1.shape[0]
        scratch = _new(Ec, _C.contrastive_scratch_floats(b, z))
        out = _new(Ec, 4)
        _C.contrastive_fwd(Ec, Ew, target, W1, gamma, beta, W2, bn_eps, momentum, run_mean, run_var, n_tracked,
                           lambda_off, scratch, out)
        ctx.save_for_backward(Ec, Ew, W1, gamma, beta, W2, scratch)
        return out[0].clone()

    @staticmethod
    def backward(ctx, gout):
        Ec, Ew, W1, gamma, beta, W2, scratch = ctx.saved_tensors
        b, z = Ec.shape[0], W1.shape[0]
        need = ctx.needs_input_grad
        gEc, gEw = _new(Ec, *Ec.shape), _new(Ew, *Ew.shape)
        gW1 = _new(W1, *W1.shape) if need[3] else None
        gg = _new(gamma, z) if need[4] else None
        gb = _new(beta, z) if need[5] else None
        gW2 = _new(W2, *W2.shape) if need[6] else None
        work = _new(Ec, 4 * b * z)
        _C.contrastive_bwd(Ec, Ew, W1, gamma, beta, W2, scratch, gout.reshape(1).contiguous().float(), work,
                           gEc, gEw, gW1, gg, gb, gW2)
        return gEc, gEw, None, gW1, gg, gb, gW2, None, None, None, None, None, None


def paired_contrastive(Ec, Ew, target, W1, gamma, beta, W2, run_mean, run_var, n_tracked, bn_eps, momentum, lambda_off):
    return _Contrastive.apply(Ec, Ew, target, W1, gamma, beta, W2, run_mean, run_var, n_tracked, float(bn_eps),
                              float(momentum), float(lambda_off))


# ==================================================================================================
# dense Linear on the TMA-fed tensor-core GEMM (forward, dgrad, wgrad)
# ==================================================================================================
_linear_impl = "tma"       # "tma": csrc/gemm_tma.cu (default); "fused": csrc/linear_tc.cu in the no-grad path (A/B timing)
_weight_planes = {}       # id(weight) -> (key, planes [n, out, in_p], planes_t [n, in, out_p])


def _n_planes():
    prec = _PRECISIONS[_precision]
    return 1 if prec == _C.PREC_BF16 else 3


def _planes_of_weight(weight, need_t):
    """Pre-split bf16 planes of a weight matrix, row-major ([out, in]: forward) and transposed ([in, out]: dgrad),
    cached per parameter version -- in inference the weights are constants, in training they change once per step."""
    n = _n_planes()
    key = None
    if isinstance(weight, torch.nn.Parameter):          # temporaries (e.g. a concatenated [Wq; Wk; Wv]) are not cached
        try:
            key = (weight.data_ptr(), weight._version, n, _cache_generation)
        except RuntimeError:
            key = None
    hit = _weight_planes.get(id(weight))
    if key is not None and hit is not None and hit[0] == key and (hit[2] is not None or not need_t):
        return hit[1], hit[2]
    with torch.no_grad():
        planes, planes_t, _, _ = _C.split_planes(weight.detach(), n, rows=True, transposed=need_t)
    if key is not None:
        _weight_planes[id(weight)] = (key, planes, planes_t)
    return planes, planes_t


class _LinearTC(torch.autograd.Function):
    """``relu?(x @ W^T + b)`` with all three GEMMs of the layer (forward, input gradient, weight gradient) on the
    TMA-fed tcgen05 kernel (csrc/gemm_tma.cu), fp32-accurate through the bf16x3 split.  Reference: the nn.Linear
    layers of the sequence VAE and their autograd (models/hybrid_models.py:63-74 / 297-308)."""

    @staticmethod
    def forward(ctx, x, weight, bias, relu):
        n = _n_planes()
        need_dx, need_dw = ctx.needs_input_grad[0], ctx.needs_input_grad[1]
        xp, xpt, _, xflag = _C.split_planes(x, n, rows=True, transposed=need_dw, flag=(n == 3))
        wp, wpt = _planes_of_weight(weight, need_dx)
        y = _C.gemm_planes(xp, wp, None if bias is None else bias.detach().contiguous(), relu, a_flag=xflag)
        ctx.relu, ctx.n, ctx.has_bias = relu, n, bias is not None
        ctx.save_for_backward(xpt, xflag, wpt, y if relu else None)
        return y

    @staticmethod
    def backward(ctx, gy):
        xpt, xflag, wpt, y = ctx.saved_tensors
        need_dx, need_dw, need_db = ctx.needs_input_grad[0], ctx.needs_input_grad[1], ctx.has_bias and ctx.needs_input_grad[2]
        gy = gy if gy.stride(-1) == 1 else gy.contiguous()
        gp, gpt, part, _ = _C.split_planes(gy, ctx.n, rows=need_dx, transposed=need_dw, relu_src=y if ctx.relu else None,
                                           colsum=need_db)
        gx = _C.gemm_planes(gp, wpt) if need_dx else None                     # gX = gY W
        gw = _C.gemm_planes(gpt, xpt, b_flag=xflag) if need_dw else None       # gW = gY^T X
        gb = None
        if need_db:
            gb = _new(gy, gy.shape[1])
            _C.reduce_partials(part, gb)
        return gx, gw, gb, None


def linear_tc(x, weight, bias=None, relu=False):
    """Differentiable ``relu?(F.linear(x, weight, bias))`` on the tensor cores; x [M, K] fp32 with unit inner stride."""
    ops = _ops()
    if ops is not None:
        return ops.linear(x, weight, bias, relu)
    return _LinearTC.apply(x, weight, bias, relu)
