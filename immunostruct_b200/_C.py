"""ctypes binding of ``libimmunostruct_b200.so`` (the C ABI declared in include/immunostruct_b200.h).

Every function here takes torch CUDA tensors, checks device / dtype / layout, and enqueues the
kernel on torch's current stream.  There is NO CPU fallback: a missing library or a CPU tensor
raises.  The caller owns (pre-allocates) every output and scratch buffer.
"""
from __future__ import annotations

import ctypes
import os

import torch

from .build import LIB_PATH

_lib = None

_i64, _i32, _f32, _vp = ctypes.c_int64, ctypes.c_int, ctypes.c_float, ctypes.c_void_p


class ExtensionMissing(RuntimeError):
    pass


def lib():
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise ExtensionMissing(
                f"{LIB_PATH} not built. Run `python -c 'import __graft_entry__ as g; g.build()'` "
                "(nvcc, sm_100a). immunostruct_b200 has no CPU or eager fallback.")
        # IS_B200_DEBUG_LIB: a debug build of the same sources (e.g. -DIS_TRACE, scripts/trace_edge_fwd.sh); never set in tests / bench
        _lib = ctypes.CDLL(os.environ.get("IS_B200_DEBUG_LIB", LIB_PATH))
    return _lib


def lib_is_patched() -> bool:
    """True when a test has replaced the kernel entry points by the CPU contracts (tests/test_host_glue.py)."""
    return getattr(split_planes, "__module__", __name__) != __name__


def exported_symbols():
    """Names declared in include/immunostruct_b200.h (used by the CPU symbol-presence test)."""
    return ["is_num_sms", "is_egnn_node_grid", "is_egnn_edge_bwd_grid", "is_attn_max_nodes",
            "is_loss_num_partials", "is_collate_csr", "is_egnn_node_pre_fwd", "is_egnn_edge_fwd",
            "is_egnn_node_post_fwd", "is_egnn_node_post_bwd", "is_egnn_edge_bwd", "is_egnn_node_pre_bwd",
            "is_reduce_partials", "is_attn_pool_fwd", "is_attn_pool_bwd", "is_fusion_attn_fwd",
            "is_fusion_attn_bwd", "is_loss_fwd", "is_loss_bwd", "is_umma_selftest", "is_umma_timing", "is_egnn_edge_fwd_tc", "is_attn_pool_infer", "is_egnn_node_post_pre_tc", "is_egnn_edge_bwd_tc", "is_egnn_edge_bwd_ws", "is_egnn_set_bwd_ws_warps", "is_linear_tc", "is_linear_tc_split_k", "is_attn_pool_infer_tc", "is_vae_mid_infer", "is_head_infer", "is_unpack_nodes", "is_unpack_edges", "is_onehot_tokens", "is_egnn_node_post_bwd_tc", "is_egnn_node_pre_bwd_tc", "is_attn_pool_bwd_tc",
            "is_segment_pool_fwd", "is_segment_pool_bwd", "is_contrastive_scratch_floats", "is_contrastive_fwd",
            "is_contrastive_bwd", "is_fused_adam", "is_rotate_coords", "is_mask_single_residue", "is_mask_rows", "is_gemm_tma_split_k",
            "is_split_planes", "is_gemm_planes_tma", "is_egnn_set_ws_buffers", "is_egnn_set_ws_variant", "is_reduce_partials3", "is_fused_adam_capturable",
            "is_egnn_edge_attr_grad", "is_head_mc_infer", "is_mutscan_expand", "is_variant_expand", "is_design_expand",
            "is_design_select", "is_egnn_layer_fwd_fp16x2", "is_occlusion_expand", "is_coord_noise_expand",
            "is_shapley_plan", "is_shapley_expand", "is_shapley_reduce", "is_head_features_infer", "is_knn",
            "is_shapley_edge_plan", "is_shapley_edge_expand"]


def _check(rc: int, name: str):
    if rc != 0:
        kind = {-1: "bad argument", -2: "unsupported size"}.get(rc, f"cudaError {rc}")
        raise RuntimeError(f"{name} failed: {kind}")


_dev_seen = None        # device index of the tensors of the call being assembled (checked in _call)


def _t(t, dtype, name, contiguous=True):
    """Device pointer of a checked tensor argument (None passes through as NULL).  Kept lean: a training step makes
    ~300 calls with ~20 arguments each, so every attribute access here is paid thousands of times per step."""
    global _dev_seen
    if t is None:
        return None
    d = t.get_device()                              # -1 for a CPU tensor
    if d < 0:
        raise RuntimeError(f"{name}: expected a CUDA tensor (immunostruct_b200 has no CPU path), got {t.device}")
    if t.dtype is not dtype:
        raise TypeError(f"{name}: expected {dtype}, got {t.dtype}")
    if contiguous and not t.is_contiguous():
        raise ValueError(f"{name}: expected a contiguous tensor")
    if _dev_seen is None:
        _dev_seen = d
    elif _dev_seen != d:
        seen, _dev_seen = _dev_seen, None
        raise RuntimeError(f"{name}: tensors of one kernel call live on different devices (cuda:{seen} and cuda:{d})")
    return _vp(t.data_ptr())


def _rows(t, name):
    """[n, k] fp32 view whose rows are contiguous (inner stride 1); returns (ptr, leading dim)."""
    global _dev_seen
    d = t.get_device()
    if d < 0 or t.dtype is not torch.float32 or t.dim() != 2 or (t.shape[1] > 1 and t.stride(1) != 1):
        raise ValueError(f"{name}: expected a CUDA fp32 [n,k] tensor with unit inner stride")
    if _dev_seen is None:
        _dev_seen = d
    elif _dev_seen != d:
        seen, _dev_seen = _dev_seen, None
        raise RuntimeError(f"{name}: tensors of one kernel call live on different devices (cuda:{seen} and cuda:{d})")
    return _vp(t.data_ptr()), _i64(t.stride(0))


_raw_stream = getattr(torch._C, "_cuda_getCurrentRawStream", None)
_raw_device = getattr(torch._C, "_cuda_getDevice", None)


def _stream():
    """torch's current stream on the current device as a raw cudaStream_t (the direct C accessors when this torch build
    has them: ``torch.cuda.current_stream()`` builds a Stream object per call, ~15 us x 200 launches per step)."""
    if _raw_stream is not None and _raw_device is not None:
        return _vp(_raw_stream(_raw_device()))
    return _vp(torch.cuda.current_stream().cuda_stream)


def _current_device():
    return _raw_device() if _raw_device is not None else torch.cuda.current_device()


_FN = {}              # launcher name -> ctypes function (restype set once)
LAUNCHES = 0          # number of immunostruct_b200 kernels enqueued so far (bench.py reports the delta)
_KERNELS_PER_CALL = {"is_collate_csr": 1, "is_egnn_edge_bwd_ws": 2, "is_loss_fwd": 2, "is_loss_bwd": 2, "is_contrastive_fwd": 9,
                     "is_contrastive_bwd": 9, "is_head_mc_infer": 2}


def _call(name, *args):
    """Enqueue one C-ABI launcher.  The tensors seen while the arguments were assembled must share one device; if that
    device is not the current one (model on cuda:1 without set_device) the call runs under a device guard, because the
    launchers use the current device and the stream handed over must belong to it."""
    global LAUNCHES, _dev_seen
    dev, _dev_seen = _dev_seen, None
    fn = _FN.get(name)
    if fn is None:
        fn = _FN[name] = getattr(lib(), name)
        fn.restype = ctypes.c_int
    if dev is not None and dev != _current_device():
        with torch.cuda.device(dev):
            args = args[:-1] + (_stream(),)          # the stream argument is always last: re-take it on that device
            _check(fn(*args), name)
    else:
        _check(fn(*args), name)
    LAUNCHES += _KERNELS_PER_CALL.get(name, 1)


def set_bwd_ws_warps(n: int) -> None:
    """Warps per tile stream (8 default, 12, 16) of the two-stream edge backward kernel."""
    rc = lib().is_egnn_set_bwd_ws_warps(ctypes.c_int(n))
    if rc != 0:
        raise ValueError("edge backward warps per stream: 8, 12 or 16")


def set_ws_variant(bits: int) -> None:
    """Variant bits of the warp-specialised edge forward kernel: bit 0 = A operand of MMA 2 from tensor memory (default 1)."""
    fn = lib().is_egnn_set_ws_variant
    fn.restype = ctypes.c_int
    _check(fn(_i32(bits)), "is_egnn_set_ws_variant")


def set_ws_buffers(n: int) -> None:
    """Operand-buffer depth of the warp-specialised edge forward kernel (only 2 is supported; 3 was measured, see DESIGN.md)."""
    fn = lib().is_egnn_set_ws_buffers
    fn.restype = ctypes.c_int
    _check(fn(_i32(n)), "is_egnn_set_ws_buffers")


# ---- sizing queries ----------------------------------------------------------------------------
def num_sms() -> int:
    return int(lib().is_num_sms())


def egnn_node_grid(n_nodes: int) -> int:
    fn = lib().is_egnn_node_grid
    fn.argtypes = [_i64]
    return int(fn(n_nodes))


def egnn_edge_bwd_grid(n_nodes: int) -> int:
    fn = lib().is_egnn_edge_bwd_grid
    fn.argtypes = [_i64]
    return int(fn(n_nodes))


def attn_max_nodes() -> int:
    return int(lib().is_attn_max_nodes())


def loss_num_partials() -> int:
    return int(lib().is_loss_num_partials())


# ---- collation ---------------------------------------------------------------------------------
def collate_csr(src_local, dst_local, node_counts, edge_counts, n_nodes, n_edges, out):
    i64, i32 = torch.int64, torch.int32
    _call("is_collate_csr", _t(src_local, i64, "src"), _t(dst_local, i64, "dst"),
          _t(node_counts, i64, "node_counts"), _t(edge_counts, i64, "edge_counts"),
          _i32(node_counts.numel()), _i64(n_nodes), _i64(n_edges),
          _t(out["node_off"], i64, "node_off"), _t(out["edge_off"], i64, "edge_off"),
          _t(out["edge_index"], i64, "edge_index"), _t(out["batch"], i64, "batch"),
          _t(out["indptr"], i32, "indptr"), _t(out["csr_src"], i32, "csr_src"),
          _t(out["csr_dst"], i32, "csr_dst"), _t(out["csr_eid"], i32, "csr_eid"),
          _t(out["outptr"], i32, "outptr"), _t(out["csc_pos"], i32, "csc_pos"),
          _t(out["scratch"], i32, "scratch"), _t(out["stats"], i32, "stats"), _stream())


# ---- EGNN --------------------------------------------------------------------------------------
def _csr(g):
    i32 = torch.int32
    return (_t(g.indptr, i32, "indptr"), _t(g.csr_src, i32, "csr_src"), _t(g.csr_dst, i32, "csr_dst"),
            _t(g.csr_eid, i32, "csr_eid"))


def egnn_node_pre_fwd(h, W1, b1, PQ):
    f32 = torch.float32
    hp, ldh = _rows(h, "h")
    _call("is_egnn_node_pre_fwd", hp, ldh, _i32(h.shape[1]), _t(W1, f32, "W1"), _t(b1, f32, "b1"),
          _t(PQ, f32, "PQ"), _i64(h.shape[0]), _stream())


def egnn_edge_fwd(g, PQ, x, edge_attr, F, W1, W2, b2, W3, b3, w4, update_coords, hn, x_out):
    f32 = torch.float32
    xp, ldx = _rows(x, "x")
    _call("is_egnn_edge_fwd", *_csr(g), _t(PQ, f32, "PQ"), xp, ldx, _t(edge_attr, f32, "edge_attr"),
          _t(W1, f32, "W1"), _i32(F), _t(W2, f32, "W2"), _t(b2, f32, "b2"), _t(W3, f32, "W3"),
          _t(b3, f32, "b3"), _t(w4, f32, "w4"), _i32(1 if update_coords else 0), _t(hn, f32, "hn"),
          _t(x_out, f32, "x_out"), _i64(PQ.shape[0]), _t(g.status, torch.int32, "status"), _stream())


PREC_BF16, PREC_TF32X3, PREC_BF16X3, PREC_FP16X2 = 0, 2, 3, 4


def egnn_node_post_pre_tc(h, hn, W5, b5, W6, b6, h_out, W1n, b1n, PQn, precision, fast_act=True, next_kind=1):
    """node_post(l) + node_pre(l+1) on the tensor cores (csrc/egnn_node_tc.cu); W1n/b1n/PQn None = nothing follows;
    next_kind 2: W1n = [Wq;Wk;Wv] [192,64], b1n [192], PQn = QKV [N,192] (attention projections after the last layer)."""
    f32 = torch.float32
    hp, ldh = _rows(h, "h")
    _call("is_egnn_node_post_pre_tc", hp, ldh, _i32(h.shape[1]), _t(hn, f32, "hn"), _t(W5, f32, "W5"),
          _t(b5, f32, "b5"), _t(W6, f32, "W6"), _t(b6, f32, "b6"), _t(h_out, f32, "h_out"), _t(W1n, f32, "W1n"),
          _t(b1n, f32, "b1n"), _t(PQn, f32, "PQn"), _i64(h.shape[0]), _i32(precision), _i32(1 if fast_act else 0),
          _i32(next_kind), _stream())


def egnn_edge_fwd_tc(g, PQ, x, edge_attr, F, W1, W2, b2, W3, b3, w4, update_coords, precision, hn, x_out,
                     fast_act=False):
    """tcgen05 / TMEM variant of egnn_edge_fwd (csrc/egnn_tc.cu); precision PREC_BF16 or PREC_TF32X3."""
    f32 = torch.float32
    xp, ldx = _rows(x, "x")
    _call("is_egnn_edge_fwd_tc", *_csr(g), _t(PQ, f32, "PQ"), xp, ldx, _t(edge_attr, f32, "edge_attr"),
          _t(W1, f32, "W1"), _i32(F), _t(W2, f32, "W2"), _t(b2, f32, "b2"), _t(W3, f32, "W3"),
          _t(b3, f32, "b3"), _t(w4, f32, "w4"), _i32(1 if update_coords else 0), _i32(precision),
          _i32(1 if fast_act else 0), _t(hn, f32, "hn"), _t(x_out, f32, "x_out"), _i64(PQ.shape[0]), _t(g.status, torch.int32, "status"),
          _stream())


def egnn_layer_fwd_fp16x2(g, PQ, x, edge_attr, W1, W2, b2, W3, b3, w4, update_coords, hn, x_out,
                          h, W5, b5, W6, b6, h_out, W1n, b1n, PQn, next_kind=1):
    """One whole EGNN layer of the fp16x2 inference forward in one launch (csrc/egnn_tc2.cu): egnn_edge_fwd_tc followed by
    egnn_node_post_pre_tc, both in PREC_FP16X2, bit for bit.  ``h`` is the layer's input [N, F]; W1n / b1n / PQn and
    next_kind as in egnn_node_post_pre_tc (next_kind 2, the QKV projections, only without ``update_coords``)."""
    f32 = torch.float32
    xp, ldx = _rows(x, "x")
    hp, ldh = _rows(h, "h")
    _call("is_egnn_layer_fwd_fp16x2", *_csr(g), _t(PQ, f32, "PQ"), xp, ldx, _t(edge_attr, f32, "edge_attr"),
          _t(W1, f32, "W1"), _i32(h.shape[1]), _t(W2, f32, "W2"), _t(b2, f32, "b2"), _t(W3, f32, "W3"),
          _t(b3, f32, "b3"), _t(w4, f32, "w4"), _i32(1 if update_coords else 0), _t(hn, f32, "hn"), _t(x_out, f32, "x_out"),
          hp, ldh, _t(W5, f32, "W5"), _t(b5, f32, "b5"), _t(W6, f32, "W6"), _t(b6, f32, "b6"), _t(h_out, f32, "h_out"),
          _t(W1n, f32, "W1n"), _t(b1n, f32, "b1n"), _t(PQn, f32, "PQn"), _i32(next_kind), _i64(PQ.shape[0]),
          _t(g.status, torch.int32, "status"), _stream())


def egnn_node_post_fwd(h, hn, W5, b5, W6, b6, h_out):
    f32 = torch.float32
    hp, ldh = _rows(h, "h")
    _call("is_egnn_node_post_fwd", hp, ldh, _i32(h.shape[1]), _t(hn, f32, "hn"), _t(W5, f32, "W5"),
          _t(b5, f32, "b5"), _t(W6, f32, "W6"), _t(b6, f32, "b6"), _t(h_out, f32, "h_out"),
          _i64(h.shape[0]), _stream())


def egnn_node_post_bwd(gh_out, h, hn, W5, b5, W6, gh_direct, ghn, partials):
    f32 = torch.float32
    hp, ldh = _rows(h, "h")
    _call("is_egnn_node_post_bwd", _t(gh_out, f32, "gh_out"), hp, ldh, _i32(h.shape[1]), _t(hn, f32, "hn"),
          _t(W5, f32, "W5"), _t(b5, f32, "b5"), _t(W6, f32, "W6"), _t(gh_direct, f32, "gh_direct"),
          _t(ghn, f32, "ghn"), _t(partials, f32, "partials"), _i64(h.shape[0]), _stream())


def egnn_node_post_bwd_tc(gh_out, h, hn, W5, b5, W6, gh_direct, ghn, partials):
    """tcgen05 (bf16x3) variant of egnn_node_post_bwd (csrc/egnn_node_bwd_tc.cu): same outputs and partial layout."""
    f32 = torch.float32
    hp, ldh = _rows(h, "h")
    _call("is_egnn_node_post_bwd_tc", _t(gh_out, f32, "gh_out"), hp, ldh, _i32(h.shape[1]), _t(hn, f32, "hn"),
          _t(W5, f32, "W5"), _t(b5, f32, "b5"), _t(W6, f32, "W6"), _t(gh_direct, f32, "gh_direct"),
          _t(ghn, f32, "ghn"), _t(partials, f32, "partials"), _i64(h.shape[0]), _stream())


def egnn_edge_bwd(g, PQ, x, edge_attr, F, W1, W2, b2, W3, b3, w4, ghn, gx_out, gz1, gQ, gD, gxd, partials):
    f32 = torch.float32
    xp, ldx = _rows(x, "x")
    _call("is_egnn_edge_bwd", *_csr(g), _t(PQ, f32, "PQ"), xp, ldx, _t(edge_attr, f32, "edge_attr"),
          _t(W1, f32, "W1"), _i32(F), _t(W2, f32, "W2"), _t(b2, f32, "b2"), _t(W3, f32, "W3"),
          _t(b3, f32, "b3"), _t(w4, f32, "w4"), _t(ghn, f32, "ghn"), _t(gx_out, f32, "gx_out"),
          _t(gz1, f32, "gz1"), _t(gQ, f32, "gQ"), _t(gD, f32, "gD"), _t(gxd, f32, "gxd"),
          _t(partials, f32, "partials"), _i64(PQ.shape[0]), _t(g.status, torch.int32, "status"), _stream())


def egnn_edge_bwd_tc(g, PQ, x, edge_attr, F, W1, W2, b2, W3, b3, w4, ghn, gx_out, gz1, gQ, gD, gxd, partials):
    """tcgen05 / TMEM variant of egnn_edge_bwd (csrc/egnn_bwd_tc.cu): same outputs, same partial layout."""
    f32 = torch.float32
    xp, ldx = _rows(x, "x")
    _call("is_egnn_edge_bwd_tc", *_csr(g), _t(PQ, f32, "PQ"), xp, ldx, _t(edge_attr, f32, "edge_attr"),
          _t(W1, f32, "W1"), _i32(F), _t(W2, f32, "W2"), _t(b2, f32, "b2"), _t(W3, f32, "W3"),
          _t(b3, f32, "b3"), _t(w4, f32, "w4"), _t(ghn, f32, "ghn"), _t(gx_out, f32, "gx_out"),
          _t(gz1, f32, "gz1"), _t(gQ, f32, "gQ"), _t(gD, f32, "gD"), _t(gxd, f32, "gxd"),
          _t(partials, f32, "partials"), _i64(PQ.shape[0]), _t(g.status, torch.int32, "status"), _stream())


def egnn_edge_bwd_ws(g, PQ, x, edge_attr, F, W1, W2, b2, W3, b3, w4, ghn, gx_out, gz1, gQ, gD, gxd, partials):
    """Two-tile-stream tcgen05 edge backward (csrc/egnn_bwd_ws.cu): same outputs, same partial layout.  The batch's
    maximum in-degree stays on the device (``g.stats[0]``): batches with a node of more than 112 in-edges are taken by
    the lock-step kernel that the same call enqueues behind it."""
    f32 = torch.float32
    xp, ldx = _rows(x, "x")
    _call("is_egnn_edge_bwd_ws", *_csr(g), _t(PQ, f32, "PQ"), xp, ldx, _t(edge_attr, f32, "edge_attr"),
          _t(W1, f32, "W1"), _i32(F), _t(W2, f32, "W2"), _t(b2, f32, "b2"), _t(W3, f32, "W3"),
          _t(b3, f32, "b3"), _t(w4, f32, "w4"), _t(ghn, f32, "ghn"), _t(gx_out, f32, "gx_out"),
          _t(gz1, f32, "gz1"), _t(gQ, f32, "gQ"), _t(gD, f32, "gD"), _t(gxd, f32, "gxd"),
          _t(partials, f32, "partials"), _t(getattr(g, "stats", None), torch.int32, "stats"), _i64(PQ.shape[0]),
          _t(g.status, torch.int32, "status"), _stream())


def egnn_node_pre_bwd(gz1, gQ, gD, gxd, gx_out, gh_direct, g, h, W1, gh, gx, partials):
    f32, i32 = torch.float32, torch.int32
    hp, ldh = _rows(h, "h")
    _call("is_egnn_node_pre_bwd", _t(gz1, f32, "gz1"), _t(gQ, f32, "gQ"), _t(gD, f32, "gD"), _t(gxd, f32, "gxd"),
          _t(gx_out, f32, "gx_out"), _t(gh_direct, f32, "gh_direct"), _t(g.outptr, i32, "outptr"),
          _t(g.csc_pos, i32, "csc_pos"), hp, ldh, _i32(h.shape[1]), _t(W1, f32, "W1"), _t(gh, f32, "gh"),
          _t(gx, f32, "gx"), _t(partials, f32, "partials"), _i64(h.shape[0]), _stream())


def egnn_node_pre_bwd_tc(gz1, gQ, gD, gxd, gx_out, gh_direct, g, h, W1, gh, gx, partials):
    """tcgen05 (bf16x3) variant of egnn_node_pre_bwd (csrc/egnn_node_bwd_tc.cu): same outputs and partial layout."""
    f32, i32 = torch.float32, torch.int32
    hp, ldh = _rows(h, "h")
    _call("is_egnn_node_pre_bwd_tc", _t(gz1, f32, "gz1"), _t(gQ, f32, "gQ"), _t(gD, f32, "gD"), _t(gxd, f32, "gxd"),
          _t(gx_out, f32, "gx_out"), _t(gh_direct, f32, "gh_direct"), _t(g.outptr, i32, "outptr"),
          _t(g.csc_pos, i32, "csc_pos"), hp, ldh, _i32(h.shape[1]), _t(W1, f32, "W1"), _t(gh, f32, "gh"),
          _t(gx, f32, "gx"), _t(partials, f32, "partials"), _i64(h.shape[0]), _stream())


def egnn_edge_attr_grad(gz1, g, W1, F, g_attr, accumulate):
    """g_attr [E] (original edge order) (+)= gz1 [E, 64] (CSR order) . W1[:, 2F+1]: one layer's gradient of the scalar edge
    features (csrc/egnn_edge_attr.cu)."""
    f32 = torch.float32
    _call("is_egnn_edge_attr_grad", _t(gz1, f32, "gz1"), _t(g.csr_eid, torch.int32, "csr_eid"), _t(W1, f32, "W1"), _i32(F),
          _t(g_attr, f32, "g_attr"), _i64(gz1.shape[0]), _i32(1 if accumulate else 0), _stream())


def reduce_partials(partials, out):
    f32 = torch.float32
    _call("is_reduce_partials", _t(partials, f32, "partials"), _i32(partials.shape[0]), _i64(partials.shape[1]),
          _t(out, f32, "out"), _stream())


def reduce_partials3(parts, outs):
    """Three (partials [n, stride], out [stride]) pairs reduced in CTA order by one launch."""
    f32 = torch.float32
    args = []
    for p, o in zip(parts, outs):
        args += [_t(p, f32, "partials"), _i32(p.shape[0]), _i64(p.shape[1]), _t(o, f32, "out")]
    _call("is_reduce_partials3", *args, _stream())


# ---- attention + pooling -----------------------------------------------------------------------
def attn_pool_fwd(QKV, node_off, n_head, max_nodes, O, LSE, pooled, attn=None, attn_off=None):
    f32, i64 = torch.float32, torch.int64
    _call("is_attn_pool_fwd", _t(QKV, f32, "QKV"), _t(node_off, i64, "node_off"), _i32(node_off.numel() - 1),
          _i32(n_head), _i32(max_nodes), _t(O, f32, "O"), _t(LSE, f32, "LSE"), _t(pooled, f32, "pooled"),
          _t(attn, f32, "attn"), _t(attn_off, i64, "attn_off"), _stream())


def attn_pool_infer(QKV, node_off, n_head, max_nodes, pooled):
    f32, i64 = torch.float32, torch.int64
    _call("is_attn_pool_infer", _t(QKV, f32, "QKV"), _t(node_off, i64, "node_off"), _i32(node_off.numel() - 1),
          _i32(n_head), _i32(max_nodes), _t(pooled, f32, "pooled"), _stream())


def attn_pool_infer_tc(QKV, node_off, max_nodes, pooled, precision=PREC_BF16X3):
    """single-head per-graph attention + mean pool on the tensor cores (csrc/attn_pool_tc.cu); pooled rows only"""
    f32, i64 = torch.float32, torch.int64
    _call("is_attn_pool_infer_tc", _t(QKV, f32, "QKV"), _t(node_off, i64, "node_off"), _i32(node_off.numel() - 1),
          _i32(max_nodes), _i32(precision), _t(pooled, f32, "pooled"), _stream())


def attn_pool_bwd_tc(QKV, node_off, max_nodes, g_pooled, gQKV):
    """backward of attn_pool_infer_tc (single head, pooled rows only) on the tensor cores (csrc/attn_pool_bwd_tc.cu)"""
    f32, i64 = torch.float32, torch.int64
    _call("is_attn_pool_bwd_tc", _t(QKV, f32, "QKV"), _t(node_off, i64, "node_off"), _i32(node_off.numel() - 1),
          _i32(max_nodes), _t(g_pooled, f32, "g_pooled"), _t(gQKV, f32, "gQKV"), _stream())


def attn_pool_bwd(QKV, O, LSE, node_off, n_head, max_nodes, g_pooled, gO_full, gQKV):
    f32, i64 = torch.float32, torch.int64
    _call("is_attn_pool_bwd", _t(QKV, f32, "QKV"), _t(O, f32, "O"), _t(LSE, f32, "LSE"),
          _t(node_off, i64, "node_off"), _i32(node_off.numel() - 1), _i32(n_head), _i32(max_nodes),
          _t(g_pooled, f32, "g_pooled"), _t(gO_full, f32, "gO_full"), _t(gQKV, f32, "gQKV"), _stream())


# ---- fusion attention --------------------------------------------------------------------------
def fusion_attn_fwd(c, n_head, coef, out):
    f32 = torch.float32
    _call("is_fusion_attn_fwd", _t(c, f32, "c"), _i32(c.shape[0]), _i32(c.shape[1]), _i32(n_head),
          _t(coef, f32, "coef"), _t(out, f32, "out"), _stream())


def fusion_attn_bwd(c, n_head, coef, gout, gc, gcoef_part):
    f32 = torch.float32
    _call("is_fusion_attn_bwd", _t(c, f32, "c"), _i32(c.shape[0]), _i32(c.shape[1]), _i32(n_head),
          _t(coef, f32, "coef"), _t(gout, f32, "gout"), _t(gc, f32, "gc"), _t(gcoef_part, f32, "gcoef_part"),
          _stream())


# ---- losses ------------------------------------------------------------------------------------
def loss_fwd(recon, seq, mu, logvar, logits, y, mode, pos_weight, w_pred, w_mse, w_kld, partial, out):
    f32 = torch.float32
    _call("is_loss_fwd", _t(recon, f32, "recon"), _t(seq, f32, "seq"),
          _i64(recon.numel() if recon is not None else 0), _t(mu, f32, "mu"), _t(logvar, f32, "logvar"),
          _i64(mu.numel() if mu is not None else 0), _t(logits, f32, "logits"), _t(y, f32, "y"),
          _i64(logits.numel()), _i32(mode), _f32(pos_weight), _f32(w_pred), _f32(w_mse), _f32(w_kld),
          _t(partial, f32, "partial"), _t(out, f32, "out"), _stream())


def loss_bwd(recon, seq, mu, logvar, logits, y, mode, pos_weight, w_pred, w_mse, w_kld, gout,
             g_recon, g_mu, g_logvar, g_logits):
    f32 = torch.float32
    _call("is_loss_bwd", _t(recon, f32, "recon"), _t(seq, f32, "seq"),
          _i64(recon.numel() if recon is not None else 0), _t(mu, f32, "mu"), _t(logvar, f32, "logvar"),
          _i64(mu.numel() if mu is not None else 0), _t(logits, f32, "logits"), _t(y, f32, "y"),
          _i64(logits.numel()), _i32(mode), _f32(pos_weight), _f32(w_pred), _f32(w_mse), _f32(w_kld),
          _t(gout, f32, "gout"), _t(g_recon, f32, "g_recon"), _t(g_mu, f32, "g_mu"),
          _t(g_logvar, f32, "g_logvar"), _t(g_logits, f32, "g_logits"), _stream())


# ---- tcgen05 self-test ---------------------------------------------------------------------------
def linear_tc(x, weight, bias=None, relu=False, precision=PREC_BF16X3, out=None):
    """``act(x @ weight.T + bias)`` on the tensor cores (csrc/linear_tc.cu): x [M,K] (any row stride), weight [N,K],
    bias [N] or None -> [M,N] fp32.  precision PREC_BF16X3 (fp32-accurate) or PREC_BF16."""
    global LAUNCHES
    f32 = torch.float32
    xp, lda = _rows(x, "x")
    wp, ldw = _rows(weight, "weight")
    m, k = x.shape
    n = weight.shape[0]
    if weight.shape[1] != k:
        raise ValueError(f"linear_tc: x {tuple(x.shape)} vs weight {tuple(weight.shape)}")
    if out is None:
        out = torch.empty(m, n, dtype=f32, device=x.device)
    split = int(lib().is_linear_tc_split_k(_i64(m), _i64(n), _i64(k)))
    ws = torch.empty(split * m * n, dtype=f32, device=x.device) if split > 1 else None
    cp, ldc = _rows(out, "out")
    _call("is_linear_tc", xp, lda, wp, ldw, _t(bias, f32, "bias"), cp, ldc, _i64(m), _i64(n), _i64(k),
          _i32(1 if relu else 0), _i32(precision), _i32(split), _t(ws, f32, "workspace"), _stream())
    if split > 1:
        LAUNCHES += 1
    return out


def vae_mid_infer(h1, prop, eps, Wp0, bp0, Wp3, bp3, W21, b21, W22, b22, W3, b3):
    """Eval-mode middle of the sequence branch in one kernel (csrc/head.cu) -> (mu, logvar, z_vae, h3)."""
    f32 = torch.float32
    b, hd = h1.shape
    ld, pd = W21.shape[0], Wp3.shape[0]
    if Wp0.shape != (32, 2) or Wp3.shape[1] != 32 or W3.shape != (hd, ld + pd) or eps.shape != (b, ld):
        raise ValueError("vae_mid_infer: unexpected layer shapes")
    mu, logvar = torch.empty(b, ld, dtype=f32, device=h1.device), torch.empty(b, ld, dtype=f32, device=h1.device)
    zv, h3 = torch.empty(b, ld + pd, dtype=f32, device=h1.device), torch.empty(b, hd, dtype=f32, device=h1.device)
    args = [_t(t, f32, n) for t, n in ((h1, "h1"), (prop, "prop"), (eps, "eps"), (Wp0, "Wp0"), (bp0, "bp0"), (Wp3, "Wp3"),
                                       (bp3, "bp3"), (W21, "W21"), (b21, "b21"), (W22, "W22"), (b22, "b22"), (W3, "W3"),
                                       (b3, "b3"), (mu, "mu"), (logvar, "logvar"), (zv, "z_vae"), (h3, "h3"))]
    _call("is_vae_mid_infer", *args, _i32(b), _i32(hd), _i32(ld), _i32(pd), _stream())
    return mu, logvar, zv, h3


def head_infer(pooled, Wc, bc, z_vae, coef, n_head, W1, b1, W2, b2):
    """Eval-mode fusion head in one kernel (csrc/head.cu) -> (x_gat [B,64], out [B,n_out] or [B,32] when W2 is None)."""
    f32 = torch.float32
    b, lz = z_vae.shape
    if pooled.shape != (b, 64) or W1.shape != (32, 64 + lz):
        raise ValueError("head_infer: unexpected shapes")
    n_out = 0 if W2 is None else W2.shape[0]
    x_gat = torch.empty(b, 64, dtype=f32, device=pooled.device)
    out = torch.empty(b, n_out if W2 is not None else 32, dtype=f32, device=pooled.device)
    _call("is_head_infer", _t(pooled, f32, "pooled"), _t(Wc, f32, "Wc"), _t(bc, f32, "bc"), _t(z_vae, f32, "z_vae"), _i32(lz),
          _t(coef, f32, "coef"), _i32(n_head), _t(W1, f32, "W1"), _t(b1, f32, "b1"), _t(W2, f32, "W2"), _t(b2, f32, "b2"),
          _i32(n_out), _t(x_gat, f32, "x_gat"), _t(out, f32, "out"), _i32(b), _stream())
    return x_gat, out


def head_mc_infer(items, Wc, bc, coef, n_head, W1, b1, W2, b2):
    """The eval-mode head over K reparameterisation draws (csrc/head.cu).  ``items``: one (pooled [B,64], mu [B,LD],
    logvar [B,LD], z_vae [B,LD+PD], eps [K,B,LD]) tuple, or two for a cancer / wild-type pair (tokens item-major).
    -> (logits [B,K], prob_mean [B], prob_std [B])."""
    f32 = torch.float32
    if len(items) not in (1, 2) or any(len(it) != 5 for it in items):
        raise ValueError("head_mc_infer: one or two (pooled, mu, logvar, z_vae, eps) items")
    b, ld = items[0][1].shape
    k, lz = items[0][4].shape[0], items[0][3].shape[1]
    for pooled, mu, logvar, zv, eps in items:
        if (pooled.shape != (b, 64) or mu.shape != (b, ld) or logvar.shape != (b, ld) or zv.shape != (b, lz)
                or eps.shape != (k, b, ld)):
            raise ValueError("head_mc_infer: unexpected item shapes")
    L = len(items) * (64 + lz)
    if W1.shape != (32, L) or b1.shape != (32,) or W2.shape != (1, 32) or b2.shape != (1,) or lz < ld or L > 256:
        raise ValueError("head_mc_infer: unexpected classifier shapes")
    if (Wc is None) != (bc is None) or (Wc is not None and (Wc.shape != (64, 64) or bc.shape != (64,))):
        raise ValueError("head_mc_infer: Wc / bc must both be None or [64,64] / [64]")
    if coef is not None and (not 1 <= n_head <= 8 or coef.shape != (4 * n_head + 1,)):
        raise ValueError("head_mc_infer: coef must hold 4 n_head + 1 values, 1 <= n_head <= 8")
    dev = items[0][0].device
    logits = torch.empty(b, k, dtype=f32, device=dev)
    mean, std = torch.empty(b, dtype=f32, device=dev), torch.empty(b, dtype=f32, device=dev)
    names = ("pooled", "mu", "logvar", "z_vae", "eps")
    ptrs = [_t(t, f32, f"{n}{i}") for i, it in enumerate((items[0], items[1] if len(items) == 2 else (None,) * 5))
            for t, n in zip(it, names)]
    _call("is_head_mc_infer", *ptrs, _i32(len(items)), _i32(ld), _i32(lz - ld), _t(Wc, f32, "Wc"), _t(bc, f32, "bc"),
          _t(coef, f32, "coef"), _i32(n_head), _t(W1, f32, "W1"), _t(b1, f32, "b1"), _t(W2, f32, "W2"), _t(b2, f32, "b2"),
          _t(logits, f32, "logits"), _t(mean, f32, "prob_mean"), _t(std, f32, "prob_std"), _i32(b), _i32(k), _stream())
    return logits, mean, std


def head_features_infer(items, Wc, bc, coef, n_head, W1, b1):
    """The classifier's hidden layer of the eval-mode head at z = mu (csrc/head.cu).  ``items``: one (pooled [B,64],
    mu [B,LD], z_vae [B,LD+PD]) tuple, or two for a cancer / wild-type pair (tokens item-major); the weights as in
    ``head_mc_infer``.  -> hid [B,32]."""
    f32 = torch.float32
    if len(items) not in (1, 2) or any(len(it) != 3 for it in items):
        raise ValueError("head_features_infer: one or two (pooled, mu, z_vae) items")
    b, ld = items[0][1].shape
    lz = items[0][2].shape[1]
    for pooled, mu, zv in items:
        if pooled.shape != (b, 64) or mu.shape != (b, ld) or zv.shape != (b, lz):
            raise ValueError("head_features_infer: unexpected item shapes")
    L = len(items) * (64 + lz)
    if b < 1 or W1.shape != (32, L) or b1.shape != (32,) or lz < ld or L > 256:
        raise ValueError("head_features_infer: unexpected classifier shapes")
    if (Wc is None) != (bc is None) or (Wc is not None and (Wc.shape != (64, 64) or bc.shape != (64,))):
        raise ValueError("head_features_infer: Wc / bc must both be None or [64,64] / [64]")
    if coef is not None and (not 1 <= n_head <= 8 or coef.shape != (4 * n_head + 1,)):
        raise ValueError("head_features_infer: coef must hold 4 n_head + 1 values, 1 <= n_head <= 8")
    hid = torch.empty(b, 32, dtype=f32, device=items[0][0].device)
    names = ("pooled", "mu", "z_vae")
    ptrs = [_t(t, f32, f"{n}{i}") for i, it in enumerate((items[0], items[1] if len(items) == 2 else (None,) * 3))
            for t, n in zip(it, names)]
    _call("is_head_features_infer", *ptrs, _i32(len(items)), _i32(ld), _i32(lz - ld), _t(Wc, f32, "Wc"),
          _t(bc, f32, "bc"), _t(coef, f32, "coef"), _i32(n_head), _t(W1, f32, "W1"), _t(b1, f32, "b1"),
          _t(hid, f32, "hid"), _i32(b), _stream())
    return hid


KNN_MAX_K, KNN_MAX_DIM, KNN_QUERY_TILE = 64, 256, 64


def knn_max_slices(n_bank: int) -> int:
    """Largest bank slice count of ``knn`` for a bank of ``n_bank`` rows (every slice holds a 128-row tile)."""
    return min(65535, (n_bank + 127) // 128)


def knn(query, bank, k, exclude=None, *, slices=1):
    """Exact k nearest bank rows of every query row in squared Euclidean distance (csrc/knn.cu; the contract is in its
    header).  query [Q, D], bank [R, D] fp32 CUDA contiguous, 1 <= k <= 64, 1 <= D <= 256, 1 <= R < 2^31; exclude int64
    [Q] in [-1, R) or None.  ``slices`` = S bank slices searched by separate CTAs, 1 .. ``knn_max_slices(R)``; S > 1
    adds a [Q, S, k] workspace and the merge kernel.  The range of ``exclude`` is checked with one host read.
    -> (index [Q, k] int64, distance [Q, k] fp32), ascending by (distance, index); unfilled slots -1 / +inf."""
    global LAUNCHES
    for t, name in ((query, "query"), (bank, "bank")):
        if not isinstance(t, torch.Tensor) or t.dim() != 2:
            raise ValueError(f"knn: {name} must be a 2-D tensor [n, D]")
        if t.dtype is not torch.float32:
            raise ValueError(f"knn: {name} must be float32, got {t.dtype}")
        if not t.is_contiguous():
            raise ValueError(f"knn: {name} must be contiguous")
    (q, d), (r, d2) = query.shape, bank.shape
    if d != d2:
        raise ValueError(f"knn: query and bank must have the same feature count, got {d} and {d2}")
    if not 1 <= d <= KNN_MAX_DIM:
        raise ValueError(f"knn: 1 <= D <= {KNN_MAX_DIM} features expected, got {d}")
    if q < 1 or not 1 <= r < 2 ** 31:
        raise ValueError(f"knn: at least one query and 1 <= R < 2^31 bank rows expected, got Q = {q}, R = {r}")
    if isinstance(k, bool) or not isinstance(k, int) or not 1 <= k <= KNN_MAX_K:
        raise ValueError(f"knn: k must be an int in [1, {KNN_MAX_K}], got {k!r}")
    if isinstance(slices, bool) or not isinstance(slices, int) or not 1 <= slices <= knn_max_slices(r):
        raise ValueError(f"knn: slices must be an int in [1, {knn_max_slices(r)}] for {r} bank rows, got {slices!r}")
    if exclude is not None:
        if not isinstance(exclude, torch.Tensor) or exclude.dtype is not torch.int64 or exclude.shape != (q,):
            raise ValueError(f"knn: exclude must be an int64 tensor of shape [{q}]")
        lo, hi = torch.stack([exclude.min(), exclude.max()]).tolist()
        if lo < -1 or hi >= r:
            raise ValueError(f"knn: exclude entries must lie in [-1, {r}), got [{lo}, {hi}]")
        exclude = exclude.contiguous()
    for t, name in ((query, "query"), (bank, "bank"), (exclude, "exclude")):
        if t is not None and not t.is_cuda:
            raise RuntimeError(f"knn: {name} must be a CUDA tensor (immunostruct_b200 has no CPU path), got {t.device}")
        if t is not None and t.device != query.device:
            raise RuntimeError(f"knn: {name} must live on {query.device}, got {t.device}")
    dev = query.device
    index = torch.empty(q, k, dtype=torch.int64, device=dev)
    distance = torch.empty(q, k, dtype=torch.float32, device=dev)
    ws = torch.empty(q * slices * k, dtype=torch.int64, device=dev) if slices > 1 else None
    _call("is_knn", _t(query, torch.float32, "query"), _t(bank, torch.float32, "bank"),
          _t(exclude, torch.int64, "exclude"), _i64(q), _i64(r), _i32(d), _i32(k), _i32(slices),
          _t(ws, torch.int64, "workspace"), _t(index, torch.int64, "index"), _t(distance, torch.float32, "distance"),
          _stream())
    if slices > 1:
        LAUNCHES += 1
    return index, distance


def mutscan_expand(x23, node_off, node_index, seq, seq_index, seq_columns, sites, x23_out, seq_out, flag):
    """One pass of an in-silico saturation scan (csrc/mutscan.cu): x23_out [r*N, 23] and seq_out [r*B, L, V] become r copies
    of the base batch, copy k with the substitution sites[k] = (site p, residue column c) at node row node_off[b] +
    node_index[b, p] and sequence row seq_index[b, p] of every sample b (-1 = absent site).  ``flag`` (int32 [1], zeroed by
    the caller) is raised if a site row is not exactly one-hot or does not follow ``seq_columns``."""
    f32, i64, i32 = torch.float32, torch.int64, torch.int32
    if node_index.dim() != 2 or seq.dim() != 3 or x23.dim() != 2 or sites.dim() != 2:
        raise ValueError("mutscan_expand: node_index [B,P], seq [B,L,V], x23 [N,23] and sites [r,2] expected")
    b, p = node_index.shape
    n, (_, L, V), r = x23.shape[0], seq.shape, sites.shape[0]
    if (x23.shape[1] != 23 or node_off.shape != (b + 1,) or seq_index.shape != (b, p) or seq.shape[0] != b
            or seq_columns.shape != (20,) or sites.shape[1] != 2 or r < 1 or p < 1):
        raise ValueError("mutscan_expand: unexpected input shapes")
    if x23_out.shape != (r * n, 23) or seq_out.shape != (r * b, L, V) or flag.shape != (1,):
        raise ValueError("mutscan_expand: unexpected output shapes")
    if r * b > 0x3fffffff or L * V > 0x7fffffff:
        raise ValueError("mutscan_expand: r * B or L * V too large")
    _call("is_mutscan_expand", _t(x23, f32, "x23"), _t(node_off, i64, "node_off"), _t(node_index, i64, "node_index"),
          _t(seq, f32, "seq"), _t(seq_index, i64, "seq_index"), _t(seq_columns, i64, "seq_columns"), _t(sites, i32, "sites"),
          _i32(r), _i32(b), _i32(p), _i64(n), _i32(L), _i32(V), _t(x23_out, f32, "x23_out"), _t(seq_out, f32, "seq_out"),
          _t(flag, i32, "flag"), _stream())


def variant_expand(x23, node_off, edge_off, src_local, dst_local, edge_attr, seq, sample, offsets, node_index, seq_index,
                   residue, seq_columns, node_out, edge_out, x23_out, src_out, dst_out, edge_attr_out, seq_out, flag):
    """One pass of a variant library (csrc/mutscan.cu): variant v is a copy of base graph sample[v] (x23 rows from
    node_out[v], graph-local edges from edge_out[v], sequence seq_out[v]) with the substitutions offsets[v] ..
    offsets[v+1]-1 of (node_index, seq_index, residue) applied: residue columns one_hot_20(residue) at graph-local node row
    node_index (-1 = not in the graph), one_hot_V(seq_columns[residue]) at sequence row seq_index.  ``flag`` (int32 [1],
    zeroed by the caller) is raised if a replaced row is not exactly one-hot, contradicts ``seq_columns`` or an index is
    out of range."""
    f32, i64, i32 = torch.float32, torch.int64, torch.int32
    if x23.dim() != 2 or seq.dim() != 3 or sample.dim() != 1 or offsets.dim() != 1 or node_index.dim() != 1:
        raise ValueError("variant_expand: x23 [N,23], seq [B,L,V], sample [r], offsets [r+1] and node_index [S] expected")
    b, L, V = seq.shape
    r, s, e = sample.shape[0], node_index.shape[0], src_local.shape[0]
    if (x23.shape[1] != 23 or node_off.shape != (b + 1,) or edge_off.shape != (b + 1,) or dst_local.shape != (e,)
            or edge_attr.numel() != e or seq_index.shape != (s,) or residue.shape != (s,) or seq_columns.shape != (20,)
            or offsets.shape != (r + 1,) or r < 1):
        raise ValueError("variant_expand: unexpected input shapes")
    n_out, e_out = x23_out.shape[0], src_out.shape[0]
    if (x23_out.dim() != 2 or x23_out.shape[1] != 23 or node_out.shape != (r + 1,) or edge_out.shape != (r + 1,)
            or dst_out.shape != (e_out,) or edge_attr_out.numel() != e_out or seq_out.shape != (r, L, V) or flag.shape != (1,)):
        raise ValueError("variant_expand: unexpected output shapes")
    if 3 * r > 0x7ffffffe:
        raise ValueError("variant_expand: too many variants in one pass")
    _call("is_variant_expand", _t(x23, f32, "x23"), _t(node_off, i64, "node_off"), _t(edge_off, i64, "edge_off"),
          _t(src_local, i64, "src_local"), _t(dst_local, i64, "dst_local"), _t(edge_attr, f32, "edge_attr"), _t(seq, f32, "seq"),
          _t(sample, i64, "sample"), _t(offsets, i64, "offsets"), _t(node_index, i64, "node_index"),
          _t(seq_index, i64, "seq_index"), _t(residue, i64, "residue"), _t(seq_columns, i64, "seq_columns"),
          _t(node_out, i64, "node_out"), _t(edge_out, i64, "edge_out"), _i32(r), _i32(b), _i64(s), _i32(L), _i32(V),
          _i64(n_out), _i64(e_out), _t(x23_out, f32, "x23_out"), _t(src_out, i64, "src_out"), _t(dst_out, i64, "dst_out"),
          _t(edge_attr_out, f32, "edge_attr_out"), _t(seq_out, f32, "seq_out"), _t(flag, i32, "flag"), _stream())


def design_expand(x23, node_off, node_index, seq, seq_index, seq_columns, beam, native, allowed, n_states, max_mutations,
                  slot0, x23_out, seq_out, flag):
    """One pass of a beam-search round (csrc/mutscan.cu): x23_out [r*N, 23] and seq_out [r*B, L, V] become r copies of the
    base batch, copy k holding slot slot0 + k = (w P + p) 20 + c: state w of ``beam`` = (states [B,W,P], keys [B,W],
    n_mut [B,W], valid [B,W] bool, ...) written at every present site, with residue column c at site p when the slot is
    valid (``native`` [B,P], ``allowed`` [B,P,20] bool, the first ``n_states`` beam entries, ``max_mutations``).  ``flag``
    (int32 [1], zeroed by the caller) is raised if the base rows of a slot's site are not exactly one-hot or do not
    follow ``seq_columns``."""
    f32, i64, i32, u8 = torch.float32, torch.int64, torch.int32, torch.bool
    states, keys, n_mut, valid = beam[:4]
    if node_index.dim() != 2 or seq.dim() != 3 or x23.dim() != 2 or states.dim() != 3:
        raise ValueError("design_expand: node_index [B,P], seq [B,L,V], x23 [N,23] and states [B,W,P] expected")
    b, p = node_index.shape
    n, (_, L, V), w = x23.shape[0], seq.shape, states.shape[1]
    if (x23.shape[1] != 23 or node_off.shape != (b + 1,) or seq_index.shape != (b, p) or seq.shape[0] != b
            or seq_columns.shape != (20,) or states.shape != (b, w, p) or keys.shape != (b, w) or n_mut.shape != (b, w)
            or valid.shape != (b, w) or native.shape != (b, p) or allowed.shape != (b, p, 20)):
        raise ValueError("design_expand: unexpected input shapes")
    r = seq_out.shape[0] // b
    if r < 1 or x23_out.shape != (r * n, 23) or seq_out.shape != (r * b, L, V) or flag.shape != (1,):
        raise ValueError("design_expand: unexpected output shapes")
    if not (1 <= p <= 14 and 1 <= n_states <= w <= 32 and 0 <= slot0 and slot0 + r <= n_states * p * 20):
        raise ValueError("design_expand: P <= 14, n_states <= W <= 32 and slots inside the round expected")
    if r * b > 0x3fffffff or L * V > 0x7fffffff:
        raise ValueError("design_expand: r * B or L * V too large")
    _call("is_design_expand", _t(x23, f32, "x23"), _t(node_off, i64, "node_off"), _t(node_index, i64, "node_index"),
          _t(seq, f32, "seq"), _t(seq_index, i64, "seq_index"), _t(seq_columns, i64, "seq_columns"),
          _t(states, i64, "states"), _t(n_mut, i64, "n_mut"), _t(valid, u8, "valid"),
          _t(native, i64, "native"), _t(allowed, u8, "allowed"), _i32(slot0), _i32(r), _i32(b), _i32(p), _i32(w),
          _i32(n_states), _i32(max_mutations), _i64(n), _i32(L), _i32(V), _t(x23_out, f32, "x23_out"),
          _t(seq_out, f32, "seq_out"), _t(flag, i32, "flag"), _stream())


def design_select(beam, round_logits, round_mean, round_std, native, allowed, node_index, n_states, max_mutations, kappa,
                  maximize, beam_out, best):
    """Selection of a beam-search round (csrc/mutscan.cu), one CTA per sample: the next beam ``beam_out`` = (states
    [B,W,P], keys [B,W], n_mut [B,W], valid [B,W] bool, logits [B,W,K], prob_mean, prob_std, objective [B,W]) is the top W
    of the first ``n_states`` entries of ``beam`` (same tuple; its objective is not read) and the round's valid slots
    (round_logits [n_states*P*20, B, K], round_mean / round_std [n_states*P*20, B]) by objective fmaf(kappa, std, mean),
    descending when ``maximize``, ties to the smaller key, NaN never taken.  ``best`` [B] (any stride) gets the best
    objective."""
    f32, i64, u8 = torch.float32, torch.int64, torch.bool
    if len(beam) != 8 or len(beam_out) != 8:
        raise ValueError("design_select: beams are (states, keys, n_mut, valid, logits, prob_mean, prob_std, objective)")
    states = beam[0]
    if states.dim() != 3 or node_index.dim() != 2:
        raise ValueError("design_select: states [B,W,P] and node_index [B,P] expected")
    b, w, p = states.shape
    k = beam[4].shape[-1]
    shapes = ((b, w, p), (b, w), (b, w), (b, w), (b, w, k), (b, w), (b, w), (b, w))
    n_slots = n_states * p * 20
    if (any(tuple(t.shape) != s for t, s in zip(beam, shapes)) or any(tuple(t.shape) != s for t, s in zip(beam_out, shapes))
            or round_logits.shape != (n_slots, b, k) or round_mean.shape != (n_slots, b)
            or round_std.shape != (n_slots, b) or native.shape != (b, p) or allowed.shape != (b, p, 20)
            or node_index.shape != (b, p) or best.shape != (b,)):
        raise ValueError("design_select: unexpected shapes")
    if not (1 <= p <= 14 and 1 <= n_states <= w <= 32):
        raise ValueError("design_select: P <= 14 and n_states <= W <= 32 expected")
    if any(x.data_ptr() == y.data_ptr() for x, y in zip(beam, beam_out)):
        raise ValueError("design_select: beam_out must not alias beam")
    names = ("states", "keys", "n_mut", "valid", "logits", "prob_mean", "prob_std", "objective")
    types = (i64, i64, i64, u8, f32, f32, f32, f32)
    _call("is_design_select", *(_t(t, d, n) for t, d, n in zip(beam[:7], types, names)),
          _t(round_logits, f32, "round_logits"), _t(round_mean, f32, "round_mean"), _t(round_std, f32, "round_std"),
          _t(native, i64, "native"), _t(allowed, u8, "allowed"), _t(node_index, i64, "node_index"), _i32(b), _i32(p),
          _i32(w), _i32(n_states), _i32(k), _i32(max_mutations), _f32(kappa), _i32(1 if maximize else 0),
          *(_t(t, d, n + "_out") for t, d, n in zip(beam_out, types, names)), _t(best, f32, "best", contiguous=False),
          _i64(best.stride(0)), _stream())


def occlusion_expand(x23, node_off, edge_off, src_local, dst_local, edge_attr, sample, node_a, node_b, node_out, edge_out,
                     x23_out, src_out, dst_out, edge_attr_out, flag):
    """One pass of structural occlusion variants (csrc/occlusion.cu): variant v is base graph sample[v] with row node_a[v]
    and its edges removed (node_b[v] == -1: the row's 23 floats become 0.0) or with every edge of the contact
    {node_a[v], node_b[v]} removed; x23 rows from node_out[v], the kept edges in base order (graph-local endpoints,
    attributes) from edge_out[v].  ``flag`` (int32 [1], zeroed by the caller) is raised, and the variant not written, for
    an index out of range, node_b == node_a, or output offsets that disagree with the node count or the kept edge count."""
    f32, i64, i32 = torch.float32, torch.int64, torch.int32
    if x23.dim() != 2 or sample.dim() != 1:
        raise ValueError("occlusion_expand: x23 [N,23] and sample [r] expected")
    b, r, e = node_off.shape[0] - 1, sample.shape[0], src_local.shape[0]
    if (x23.shape[1] != 23 or b < 1 or edge_off.shape != (b + 1,) or dst_local.shape != (e,) or edge_attr.numel() != e
            or node_a.shape != (r,) or node_b.shape != (r,) or r < 1):
        raise ValueError("occlusion_expand: unexpected input shapes")
    n_out, e_out = x23_out.shape[0], src_out.shape[0]
    if (x23_out.dim() != 2 or x23_out.shape[1] != 23 or node_out.shape != (r + 1,) or edge_out.shape != (r + 1,)
            or dst_out.shape != (e_out,) or edge_attr_out.numel() != e_out or flag.shape != (1,)):
        raise ValueError("occlusion_expand: unexpected output shapes")
    if 2 * r > 0x7ffffffe:
        raise ValueError("occlusion_expand: too many variants in one pass")
    _call("is_occlusion_expand", _t(x23, f32, "x23"), _t(node_off, i64, "node_off"), _t(edge_off, i64, "edge_off"),
          _t(src_local, i64, "src_local"), _t(dst_local, i64, "dst_local"), _t(edge_attr, f32, "edge_attr"),
          _t(sample, i64, "sample"), _t(node_a, i64, "node_a"), _t(node_b, i64, "node_b"), _t(node_out, i64, "node_out"),
          _t(edge_out, i64, "edge_out"), _i32(r), _i32(b), _i64(n_out), _i64(e_out), _t(x23_out, f32, "x23_out"),
          _t(src_out, i64, "src_out"), _t(dst_out, i64, "dst_out"), _t(edge_attr_out, f32, "edge_attr_out"),
          _t(flag, i32, "flag"), _stream())


def coord_noise_expand(x23, node_off, sigma, seed, item, draw0, x23_out):
    """One pass of seeded coordinate perturbations (csrc/coordnoise.cu): x23_out [r*N, 23] becomes r copies of the base
    batch in the layout of ``GraphBatch.replicate(r)``, copy k being structure draw m = draw0 + k: columns 20..22 of
    graph-local row a of graph b get ``fmaf(sigma[i], z, x)``, z the Philox4x32-10 / Box-Muller normals of the key
    (seed, item, m, b, a); columns 0..19 and rows with sigma 0 are copied.  Every argument is checked here: the kernel
    has no flag."""
    f32, i64 = torch.float32, torch.int64
    if x23.dim() != 2 or x23.shape[1] != 23 or node_off.dim() != 1 or node_off.shape[0] < 2:
        raise ValueError("coord_noise_expand: x23 [N,23] and node_off [B+1] expected")
    n, b = x23.shape[0], node_off.shape[0] - 1
    if sigma.shape != (n,):
        raise ValueError("coord_noise_expand: sigma [N] expected")
    if x23_out.dim() != 2 or x23_out.shape[1] != 23 or x23_out.shape[0] < n or (n and x23_out.shape[0] % n):
        raise ValueError("coord_noise_expand: x23_out [r*N, 23] expected")
    r = x23_out.shape[0] // n if n else 1
    if not (isinstance(seed, int) and 0 <= seed < 2 ** 64 and isinstance(item, int) and 0 <= item < 2 ** 32
            and isinstance(draw0, int) and 0 <= draw0 and draw0 + r <= 2 ** 32):
        raise ValueError("coord_noise_expand: seed in [0, 2^64), item in [0, 2^32) and draw0 + r <= 2^32 expected")
    if r * b > 0x7fffffff:
        raise ValueError("coord_noise_expand: r * B too large")
    if x23_out.data_ptr() == x23.data_ptr():
        raise ValueError("coord_noise_expand: x23_out must not alias x23")
    _call("is_coord_noise_expand", _t(x23, f32, "x23"), _t(node_off, i64, "node_off"), _t(sigma, f32, "sigma"), _i32(r),
          _i32(b), _i64(n), ctypes.c_uint64(seed), ctypes.c_uint32(item), ctypes.c_uint32(draw0),
          _t(x23_out, f32, "x23_out"), _stream())


def shapley_plan(node_off, edge_off, src_local, dst_local, players, player_off, var_off, seed, ranks, kept, flag):
    """Permutation plan of the Shapley chains (csrc/shapley.cu): ``ranks`` int32 [B, T, Pmax] gets the rank rows of the
    antithetic pairs of every sample (row 2u: Philox4x32-10 keys of counter (p, b, u, 2), key ``seed``; row 2u+1 its
    reverse; -1 past P_b), ``kept`` int64 [V] the kept-edge count of every chain variant.  ``players`` int32 [N] (graph-
    local ids, -1: never removed), ``player_off`` / ``var_off`` int64 [B+1] the running player and variant counts.
    ``flag`` (int32 [1], zeroed by the caller) is raised for counts that disagree."""
    i64, i32 = torch.int64, torch.int32
    if ranks.dim() != 3 or node_off.dim() != 1:
        raise ValueError("shapley_plan: ranks [B, T, Pmax] and node_off [B+1] expected")
    b, t, pmax = ranks.shape
    e = src_local.shape[0]
    if (node_off.shape != (b + 1,) or edge_off.shape != (b + 1,) or dst_local.shape != (e,) or players.dim() != 1
            or player_off.shape != (b + 1,) or var_off.shape != (b + 1,) or kept.dim() != 1 or flag.shape != (1,)):
        raise ValueError("shapley_plan: unexpected shapes")
    if not (b >= 1 and 2 <= t <= 2 ** 16 and t % 2 == 0 and 1 <= pmax <= 256):
        raise ValueError("shapley_plan: T even in [2, 2^16] and 1 <= Pmax <= 256 expected")
    if not (isinstance(seed, int) and 0 <= seed < 2 ** 64):
        raise ValueError("shapley_plan: seed in [0, 2^64) expected")
    _call("is_shapley_plan", _t(node_off, i64, "node_off"), _t(edge_off, i64, "edge_off"),
          _t(src_local, i64, "src_local"), _t(dst_local, i64, "dst_local"), _t(players, i32, "players"),
          _t(player_off, i64, "player_off"), _t(var_off, i64, "var_off"), _i32(b), _i32(t), _i32(pmax),
          ctypes.c_uint64(seed), _t(ranks, i32, "ranks"), _t(kept, i64, "kept"), _t(flag, i32, "flag"), _stream())


def shapley_expand(x23, node_off, edge_off, src_local, dst_local, edge_attr, players, ranks, sample, rank_row, threshold,
                   node_out, edge_out, x23_out, src_out, dst_out, edge_attr_out, flag):
    """One pass of coalition variants (csrc/shapley.cu): variant v is base graph sample[v] with every row i removed for
    which players[i] >= 0 and ranks[rank_row[v], players[i]] < threshold[v] (its 23 floats become 0.0, every edge touching
    it is dropped); x23 rows from node_out[v], the kept edges in base order from edge_out[v].  ``ranks`` int32 [R, Pmax]
    (or [B, T, Pmax], read as [B T, Pmax]).  ``flag`` (int32 [1], zeroed by the caller) is raised, and the variant not
    written, for an index out of range or offsets that disagree with the node count or the kept edge count."""
    f32, i64, i32 = torch.float32, torch.int64, torch.int32
    if x23.dim() != 2 or sample.dim() != 1 or ranks.dim() < 2:
        raise ValueError("shapley_expand: x23 [N,23], sample [r] and ranks [R, Pmax] expected")
    b, r, e, n = node_off.shape[0] - 1, sample.shape[0], src_local.shape[0], x23.shape[0]
    pmax = ranks.shape[-1]
    if (x23.shape[1] != 23 or b < 1 or edge_off.shape != (b + 1,) or dst_local.shape != (e,) or edge_attr.numel() != e
            or players.shape != (n,) or rank_row.shape != (r,) or threshold.shape != (r,) or r < 1 or pmax < 1):
        raise ValueError("shapley_expand: unexpected input shapes")
    n_out, e_out = x23_out.shape[0], src_out.shape[0]
    if (x23_out.dim() != 2 or x23_out.shape[1] != 23 or node_out.shape != (r + 1,) or edge_out.shape != (r + 1,)
            or dst_out.shape != (e_out,) or edge_attr_out.numel() != e_out or flag.shape != (1,)):
        raise ValueError("shapley_expand: unexpected output shapes")
    if 2 * r > 0x7ffffffe:
        raise ValueError("shapley_expand: too many variants in one pass")
    _call("is_shapley_expand", _t(x23, f32, "x23"), _t(node_off, i64, "node_off"), _t(edge_off, i64, "edge_off"),
          _t(src_local, i64, "src_local"), _t(dst_local, i64, "dst_local"), _t(edge_attr, f32, "edge_attr"),
          _t(players, i32, "players"), _t(ranks, i32, "ranks"), _t(sample, i64, "sample"), _t(rank_row, i64, "rank_row"),
          _t(threshold, i64, "threshold"), _t(node_out, i64, "node_out"), _t(edge_out, i64, "edge_out"), _i32(r),
          _i32(b), _i64(ranks.numel() // pmax), _i32(pmax), _i64(n_out), _i64(e_out), _t(x23_out, f32, "x23_out"),
          _t(src_out, i64, "src_out"), _t(dst_out, i64, "dst_out"), _t(edge_attr_out, f32, "edge_attr_out"),
          _t(flag, i32, "flag"), _stream())


def shapley_edge_plan(edge_off, edge_players, player_off, var_off, seed, ranks, kept, flag):
    """Permutation plan of the contact Shapley chains (csrc/shapley.cu): as ``shapley_plan`` with the players held by
    edges, ``edge_players`` int32 [E] (graph-local ids, -1: never removed), and the keys on counter (p, b, u, 3).  An edge
    of player q is kept in coalition j of permutation t iff j <= rank_t(q)."""
    i64, i32 = torch.int64, torch.int32
    if ranks.dim() != 3 or edge_off.dim() != 1:
        raise ValueError("shapley_edge_plan: ranks [B, T, Pmax] and edge_off [B+1] expected")
    b, t, pmax = ranks.shape
    if (edge_off.shape != (b + 1,) or edge_players.dim() != 1 or player_off.shape != (b + 1,)
            or var_off.shape != (b + 1,) or kept.dim() != 1 or flag.shape != (1,)):
        raise ValueError("shapley_edge_plan: unexpected shapes")
    if not (b >= 1 and 2 <= t <= 2 ** 16 and t % 2 == 0 and 1 <= pmax <= 256):
        raise ValueError("shapley_edge_plan: T even in [2, 2^16] and 1 <= Pmax <= 256 expected")
    if not (isinstance(seed, int) and 0 <= seed < 2 ** 64):
        raise ValueError("shapley_edge_plan: seed in [0, 2^64) expected")
    _call("is_shapley_edge_plan", _t(edge_off, i64, "edge_off"), _t(edge_players, i32, "edge_players"),
          _t(player_off, i64, "player_off"), _t(var_off, i64, "var_off"), _i32(b), _i32(t), _i32(pmax),
          ctypes.c_uint64(seed), _t(ranks, i32, "ranks"), _t(kept, i64, "kept"), _t(flag, i32, "flag"), _stream())


def shapley_edge_expand(x23, node_off, edge_off, src_local, dst_local, edge_attr, edge_players, ranks, sample, rank_row,
                        threshold, node_out, edge_out, x23_out, src_out, dst_out, edge_attr_out, flag):
    """One pass of contact coalition variants (csrc/shapley.cu): variant v is base graph sample[v] with its rows copied
    and every edge e with edge_players[e] >= 0 and ranks[rank_row[v], edge_players[e]] < threshold[v] dropped, the kept
    edges in base order from edge_out[v].  ``ranks`` int32 [R, Pmax] (or [B, T, Pmax]).  ``flag`` (int32 [1], zeroed by
    the caller) is raised, and the variant not written, for an index out of range, an edge player id >= Pmax, or
    offsets that disagree with the node count or the kept edge count."""
    f32, i64, i32 = torch.float32, torch.int64, torch.int32
    if x23.dim() != 2 or sample.dim() != 1 or ranks.dim() < 2:
        raise ValueError("shapley_edge_expand: x23 [N,23], sample [r] and ranks [R, Pmax] expected")
    b, r, e = node_off.shape[0] - 1, sample.shape[0], src_local.shape[0]
    pmax = ranks.shape[-1]
    if (x23.shape[1] != 23 or b < 1 or edge_off.shape != (b + 1,) or dst_local.shape != (e,) or edge_attr.numel() != e
            or edge_players.shape != (e,) or rank_row.shape != (r,) or threshold.shape != (r,) or r < 1
            or not 1 <= pmax <= 256):
        raise ValueError("shapley_edge_expand: unexpected input shapes")
    n_out, e_out = x23_out.shape[0], src_out.shape[0]
    if (x23_out.dim() != 2 or x23_out.shape[1] != 23 or node_out.shape != (r + 1,) or edge_out.shape != (r + 1,)
            or dst_out.shape != (e_out,) or edge_attr_out.numel() != e_out or flag.shape != (1,)):
        raise ValueError("shapley_edge_expand: unexpected output shapes")
    if 2 * r > 0x7ffffffe:
        raise ValueError("shapley_edge_expand: too many variants in one pass")
    _call("is_shapley_edge_expand", _t(x23, f32, "x23"), _t(node_off, i64, "node_off"), _t(edge_off, i64, "edge_off"),
          _t(src_local, i64, "src_local"), _t(dst_local, i64, "dst_local"), _t(edge_attr, f32, "edge_attr"),
          _t(edge_players, i32, "edge_players"), _t(ranks, i32, "ranks"), _t(sample, i64, "sample"),
          _t(rank_row, i64, "rank_row"), _t(threshold, i64, "threshold"), _t(node_out, i64, "node_out"),
          _t(edge_out, i64, "edge_out"), _i32(r), _i32(b), _i64(ranks.numel() // pmax), _i32(pmax), _i64(n_out),
          _i64(e_out), _t(x23_out, f32, "x23_out"), _t(src_out, i64, "src_out"), _t(dst_out, i64, "dst_out"),
          _t(edge_attr_out, f32, "edge_attr_out"), _t(flag, i32, "flag"), _stream())


def shapley_reduce(logits, base_logits, ranks, player_off, var_off, phi, se, gap, flag):
    """Shapley values of the chains (csrc/shapley.cu), one CTA per sample: from the variants' logits [V, K], the base
    logits [B, K] and the plan's ranks [B, T, Pmax], phi / se fp32 [2, Q] (row 0: of v_logit, row 1: of v_prob) at
    player_off[b] + p, and gap fp32 [2, B] = (v(base) - v(empty)) - Σ_p phi; fp64 throughout, fixed order.  ``flag``
    (int32 [1]) is raised for variant tables or ranks that disagree."""
    f32, i64, i32 = torch.float32, torch.int64, torch.int32
    if ranks.dim() != 3 or base_logits.dim() != 2 or logits.dim() != 2:
        raise ValueError("shapley_reduce: logits [V,K], base_logits [B,K] and ranks [B,T,Pmax] expected")
    b, t, pmax = ranks.shape
    k, v, q = base_logits.shape[1], logits.shape[0], phi.shape[-1]
    if (base_logits.shape[0] != b or logits.shape[1] != k or player_off.shape != (b + 1,) or var_off.shape != (b + 1,)
            or phi.shape != (2, q) or se.shape != (2, q) or gap.shape != (2, b) or flag.shape != (1,)):
        raise ValueError("shapley_reduce: unexpected shapes")
    if not (b >= 1 and 2 <= t <= 2 ** 16 and t % 2 == 0 and 1 <= pmax <= 256 and k >= 1):
        raise ValueError("shapley_reduce: T even in [2, 2^16], 1 <= Pmax <= 256 and K >= 1 expected")
    row1 = lambda x, n: _vp(x.data_ptr() + 4 * n)                      # row 1 of a contiguous fp32 [2, n]
    _call("is_shapley_reduce", _t(logits, f32, "logits"), _t(base_logits, f32, "base_logits"), _t(ranks, i32, "ranks"),
          _t(player_off, i64, "player_off"), _t(var_off, i64, "var_off"), _i32(b), _i32(t), _i32(pmax), _i32(k), _i64(v),
          _t(phi, f32, "phi"), row1(phi, q), _t(se, f32, "se"), row1(se, q), _t(gap, f32, "gap"), row1(gap, b),
          _t(flag, i32, "flag"), _stream())


def unpack_nodes(aa, xyz, x):
    _call("is_unpack_nodes", _t(aa, torch.uint8, "aa"), _t(xyz, torch.float32, "xyz"), _t(x, torch.float32, "x"),
          _i64(aa.numel()), _stream())


def unpack_edges(src, dst, edge_attr, src64, dst64, attr_out):
    _call("is_unpack_edges", _t(src, torch.int32, "src"), _t(dst, torch.int32, "dst"), _t(edge_attr, torch.float32, "edge_attr"),
          _t(src64, torch.int64, "src64"), _t(dst64, torch.int64, "dst64"), _t(attr_out, torch.float32, "attr_out"),
          _i64(src.numel()), _stream())


def onehot_tokens(tokens, out, vocab):
    _call("is_onehot_tokens", _t(tokens, torch.uint8, "tokens"), _t(out, torch.float32, "out"), _i64(tokens.numel()),
          _i32(vocab), _stream())


def umma_selftest(A, B, D, mode):
    """D[128,64] = A[128,64] @ B[64,64]^T on the tensor cores; mode 0 bf16, 1 tf32, 2 3xTF32."""
    f32 = torch.float32
    _call("is_umma_selftest", _t(A, f32, "A"), _t(B, f32, "B"), _t(D, f32, "D"), _i32(mode), _stream())


def umma_timing(out):
    """Cycles per tcgen05.mma of 16 operand-layout / accumulator-rotation configurations into out[16] (csrc/umma_selftest.cu)."""
    _call("is_umma_timing", _t(out, torch.float32, "out"), _stream())


# ---- segment pooling -----------------------------------------------------------------------------
POOL_MODES = {"mean": 0, "max": 1, "sum": 2}


def segment_pool_fwd(X, node_off, mode, out):
    xp, ldx = _rows(X, "X")
    _call("is_segment_pool_fwd", xp, ldx, _i32(X.shape[1]), _t(node_off, torch.int64, "node_off"),
          _i32(node_off.numel() - 1), _i32(POOL_MODES[mode]), _t(out, torch.float32, "out"), _stream())


def segment_pool_bwd(X, node_off, mode, pooled, g_out, gX):
    xp, ldx = _rows(X, "X")
    gp, ldg = _rows(gX, "gX")
    _call("is_segment_pool_bwd", xp, ldx, _i32(X.shape[1]), _t(node_off, torch.int64, "node_off"),
          _i32(node_off.numel() - 1), _i32(POOL_MODES[mode]), _t(pooled, torch.float32, "pooled"),
          _t(g_out, torch.float32, "g_out"), gp, ldg, _stream())


# ---- paired contrastive loss ---------------------------------------------------------------------
def contrastive_scratch_floats(b: int, z: int) -> int:
    fn = lib().is_contrastive_scratch_floats
    fn.restype = ctypes.c_int64
    return int(fn(_i32(b), _i32(z)))


def contrastive_fwd(Ec, Ew, target, W1, gamma, beta, W2, bn_eps, momentum, run_mean, run_var, n_tracked, lambda_off,
                    scratch, out):
    f32 = torch.float32
    b, d = Ec.shape
    z = W1.shape[0]
    _call("is_contrastive_fwd", _t(Ec, f32, "Ec"), _t(Ew, f32, "Ew"), _t(target, f32, "target"), _i32(b), _i32(d), _i32(z),
          _t(W1, f32, "W1"), _t(gamma, f32, "gamma"), _t(beta, f32, "beta"), _t(W2, f32, "W2"), _f32(bn_eps),
          _f32(momentum), _t(run_mean, f32, "run_mean"), _t(run_var, f32, "run_var"),
          _t(n_tracked, torch.int64, "num_batches_tracked"), _f32(lambda_off), _t(scratch, f32, "scratch"),
          _t(out, f32, "out"), _stream())


def contrastive_bwd(Ec, Ew, W1, gamma, beta, W2, scratch, gout, work, gEc, gEw, gW1, g_gamma, g_beta, gW2):
    f32 = torch.float32
    b, d = Ec.shape
    z = W1.shape[0]
    _call("is_contrastive_bwd", _t(Ec, f32, "Ec"), _t(Ew, f32, "Ew"), _i32(b), _i32(d), _i32(z), _t(W1, f32, "W1"),
          _t(gamma, f32, "gamma"), _t(beta, f32, "beta"), _t(W2, f32, "W2"), _t(scratch, f32, "scratch"),
          _t(gout, f32, "gout"), _t(work, f32, "work"), _t(gEc, f32, "gEc"), _t(gEw, f32, "gEw"), _t(gW1, f32, "gW1"),
          _t(g_gamma, f32, "g_gamma"), _t(g_beta, f32, "g_beta"), _t(gW2, f32, "gW2"), _stream())


# ---- fused Adam ----------------------------------------------------------------------------------
def fused_adam(p, g, m, v, lr, beta1, beta2, eps, weight_decay, decoupled, step_size, inv_bc2_sqrt, grad_scale=1.0):
    f32 = torch.float32
    _call("is_fused_adam", _t(p, f32, "p"), _t(g, f32, "g"), _t(m, f32, "m"), _t(v, f32, "v"), _i64(p.numel()), _f32(lr),
          _f32(beta1), _f32(beta2), _f32(eps), _f32(weight_decay), _i32(1 if decoupled else 0), _f32(step_size),
          _f32(inv_bc2_sqrt), _f32(grad_scale), _stream())


def fused_adam_capturable(p, g, m, v, lr, beta1, beta2, eps, weight_decay, decoupled, step, tick, grad_scale=1.0):
    f32 = torch.float32
    _call("is_fused_adam_capturable", _t(p, f32, "p"), _t(g, f32, "g"), _t(m, f32, "m"), _t(v, f32, "v"), _i64(p.numel()),
          _f32(lr), _f32(beta1), _f32(beta2), _f32(eps), _f32(weight_decay), _i32(1 if decoupled else 0),
          _t(step, f32, "step"), _i32(1 if tick else 0), _f32(grad_scale), _stream())


# ---- augmentations -------------------------------------------------------------------------------
def rotate_coords(x, c0, node_off, M, Qout=None):
    xp, ldx = _rows(x, "x")
    _call("is_rotate_coords", xp, ldx, _i32(c0), _t(node_off, torch.int64, "node_off"), _i32(node_off.numel() - 1),
          _t(M, torch.float32, "M"), _t(Qout, torch.float32, "Qout"), _stream())


def mask_single_residue(x, n_feat, node_off, u, want_aa, aa_out, node_out=None):
    xp, ldx = _rows(x, "x")
    i64 = torch.int64
    _call("is_mask_single_residue", xp, ldx, _i32(n_feat), _t(node_off, i64, "node_off"), _i32(node_off.numel() - 1),
          _t(u, torch.float32, "u"), _t(want_aa, i64, "want_aa"), _t(aa_out, i64, "aa_out"), _t(node_out, i64, "node_out"),
          _stream())


def mask_rows(data, n_cols, seg_off, limit, keys, count, fill_col, max_rows):
    dp, ld = _rows(data, "data")
    i64 = torch.int64
    _call("is_mask_rows", dp, ld, _i32(n_cols), _t(seg_off, i64, "seg_off"), _t(limit, i64, "limit"),
          _i32(seg_off.numel() - 1), _t(keys, torch.float32, "keys"), _i32(count), _i32(fill_col), _i32(max_rows), _stream())


# ---- TMA-fed tcgen05 GEMM on pre-split bf16 planes (csrc/gemm_tma.cu) ----------------------------------
def split_planes(x, n_planes=3, rows=True, transposed=False, relu_src=None, colsum=False, flag=False):
    """fp32 x [R, C] -> (planes [n, R, Cp] | None, planes_t [n, C, Rp] | None, colsum partials [gr, C] | None,
    residual flag int32 [1] | None); Cp / Rp = C / R rounded up to 8 (zero padded)."""
    xp, ld = _rows(x, "x")
    r, c = x.shape
    cp, rp = (c + 7) // 8 * 8, (r + 7) // 8 * 8
    bf, dev = torch.bfloat16, x.device
    planes = torch.empty(n_planes, r, cp, dtype=bf, device=dev) if rows else None
    planes_t = torch.empty(n_planes, c, rp, dtype=bf, device=dev) if transposed else None
    gr = ((rp if transposed else r) + 31) // 32
    part = torch.empty(gr, c, dtype=torch.float32, device=dev) if colsum else None
    fl = torch.zeros(1, dtype=torch.int32, device=dev) if flag else None
    rsp, ldr = (None, _i64(0)) if relu_src is None else _rows(relu_src, "relu_src")
    _call("is_split_planes", xp, ld, _i64(r), _i64(c), rsp, ldr, _i32(n_planes), _t(planes, bf, "planes"),
          _t(planes_t, bf, "planes_t"), _t(part, torch.float32, "colsum"), _t(fl, torch.int32, "flag"), _stream())
    return planes, planes_t, part, fl


def gemm_planes(a_planes, b_planes, bias=None, relu=False, out=None, a_flag=None, b_flag=None):
    """out [M, N] = act(A B^T + bias): A planes [n, M, Kp], B planes [n, N, Kp] (bf16, from split_planes)."""
    global LAUNCHES
    bf, f32 = torch.bfloat16, torch.float32
    npl, m, kp = a_planes.shape
    n = b_planes.shape[1]
    if b_planes.shape[0] != npl or b_planes.shape[2] != kp:
        raise ValueError(f"gemm_planes: A planes {tuple(a_planes.shape)} vs B planes {tuple(b_planes.shape)}")
    if out is None:
        out = torch.empty(m, n, dtype=f32, device=a_planes.device)
    split = int(lib().is_gemm_tma_split_k(_i64(m), _i64(n), _i64(kp)))
    ws = torch.empty(split * m * n, dtype=f32, device=a_planes.device) if split > 1 else None
    cp, ldc = _rows(out, "out")
    _call("is_gemm_planes_tma", _t(a_planes, bf, "A planes"), _i64(m), _t(b_planes, bf, "B planes"), _i64(n), _i64(kp),
          _i32(npl), _t(a_flag, torch.int32, "a_flag"), _t(b_flag, torch.int32, "b_flag"), _t(bias, f32, "bias"),
          _i32(1 if relu else 0), cp, ldc, _i32(split), _t(ws, f32, "workspace"), _stream())
    if split > 1:
        LAUNCHES += 1
    return out
