"""Stress run of the warp-specialised edge forward kernel: every variant (precision x coordinate branch x SiLU form x A-operand
variant) over several batch shapes and in-degrees, 30 launches each back to back; every launch must reproduce the first one bit
for bit and agree with the lock-step first-generation kernel.  Then the fp16x2 layer kernel (the same kernel with the node tail) in
each of its instances, 30 launches each, every one equal to the two-launch path bit for bit.  Exits non-zero on any CUDA error or mismatch."""
import sys
import torch
sys.path.insert(0, ".")
from immunostruct_b200 import _C
from immunostruct_b200.graph import GraphBatch
from immunostruct_b200.synthetic import synthetic_graph_arrays

dev = "cuda"
g = torch.Generator(device=dev).manual_seed(0)
r = lambda *s: torch.randn(*s, device=dev, generator=g) * 0.2
W1, b1, W2, b2, W3, b3, w4 = r(64, 130), r(64), r(64, 64), r(64), r(64, 64), r(64), r(1, 64)
n_fail = 0
for n_graphs, n_nodes, k in ((1, 200, 10), (7, 37, 3), (64, 200, 10), (300, 190, 12), (512, 200, 10), (40, 120, 30)):
    arr = synthetic_graph_arrays(n_graphs, n_nodes, k, seed=n_graphs, device=dev)
    gb = GraphBatch.from_arrays(*(arr[kk] for kk in ("x", "src", "dst", "edge_attr", "node_counts", "edge_counts")), max_nodes=n_nodes)
    n = gb.n_nodes
    PQ, x = r(n, 128), arr["x"][:, 20:]
    for prec, tol in ((_C.PREC_BF16X3, 2e-5), (_C.PREC_FP16X2, 2e-5), (_C.PREC_BF16, 3e-2)):
        for upd in (True, False):
            ref_hn, ref_x = torch.zeros(n, 64, device=dev), torch.zeros(n, 3, device=dev)
            _C.egnn_edge_fwd_tc(gb, PQ, x, arr["edge_attr"], 64, W1, W2, b2, W3, b3, w4, upd,
                                (_C.PREC_BF16X3 if prec == _C.PREC_FP16X2 else prec) | 16, ref_hn, ref_x, fast_act=False)
            for fast in (True, False):
                for var in (0, 1):
                    _C.set_ws_variant(var)
                    first = None
                    for it in range(30):
                        hn, xo = torch.full((n, 64), float("nan"), device=dev), torch.full((n, 3), float("nan"), device=dev)
                        _C.egnn_edge_fwd_tc(gb, PQ, x, arr["edge_attr"], 64, W1, W2, b2, W3, b3, w4, upd, prec, hn, xo, fast_act=fast)
                        if first is None:
                            first = (hn, xo)
                        elif not (torch.equal(hn, first[0]) and (not upd or torch.equal(xo, first[1]))):
                            print("NOT REPRODUCIBLE", n_graphs, prec, upd, fast, var, it); n_fail += 1; break
                    torch.cuda.synchronize()
                    e_h = float((first[0] - ref_hn).abs().max() / ref_hn.abs().max())
                    e_x = float(((first[1] - x) - (ref_x - x)).abs().max() / (ref_x - x).abs().max().clamp_min(1e-30)) if upd else 0.0
                    ok = e_h < tol and e_x < tol and bool(torch.isfinite(first[0]).all())
                    n_fail += 0 if ok else 1
                    print(f"graphs {n_graphs:4d} n {n_nodes} k {k:2d} prec {prec} coords {int(upd)} fast {int(fast)} var {var}: hn {e_h:.1e} x {e_x:.1e} {'ok' if ok else 'MISMATCH'}", flush=True)
_C.set_ws_variant(1)

# the fp16x2 layer kernel with the node tail (egnn_layer_fwd_fp16x2), every instance: coordinates + next P'/Q', no coordinates +
# QKV, no coordinates + h' only.  30 launches each; every output must equal the two-launch path (edge, then node kernel) bit for bit.
W5, b5, W6, b6, W1n, b1n, Wq, bq = r(64, 128), r(64), r(64, 64), r(64), r(64, 130), r(64), r(192, 64), r(192)
for n_graphs, n_nodes, k in ((1, 200, 10), (7, 37, 3), (64, 200, 10), (300, 190, 12), (512, 200, 10), (40, 120, 30)):
    arr = synthetic_graph_arrays(n_graphs, n_nodes, k, seed=n_graphs, device=dev)
    gb = GraphBatch.from_arrays(*(arr[kk] for kk in ("x", "src", "dst", "edge_attr", "node_counts", "edge_counts")), max_nodes=n_nodes)
    n = gb.n_nodes
    PQ, x, h = r(n, 128), arr["x"][:, 20:], r(n, 64)
    for upd, kind, wn, bn, cols in ((True, 1, W1n, b1n, 128), (False, 2, Wq, bq, 192), (False, 1, None, None, 0)):
        ref_hn, ref_h = torch.zeros(n, 64, device=dev), torch.zeros(n, 64, device=dev)
        ref_x = torch.zeros(n, 3, device=dev) if upd else None
        ref_pq = torch.zeros(n, cols, device=dev) if cols else None
        _C.egnn_edge_fwd_tc(gb, PQ, x, arr["edge_attr"], 64, W1, W2, b2, W3, b3, w4, upd, _C.PREC_FP16X2, ref_hn, ref_x, fast_act=True)
        _C.egnn_node_post_pre_tc(h, ref_hn, W5, b5, W6, b6, ref_h, wn, bn, ref_pq, _C.PREC_FP16X2, next_kind=kind)
        bad = None
        for it in range(30):
            nan = lambda c: torch.full((n, c), float("nan"), device=dev)
            hn, ho, xo, pq = nan(64), nan(64), nan(3) if upd else None, nan(cols) if cols else None
            _C.egnn_layer_fwd_fp16x2(gb, PQ, x, arr["edge_attr"], W1, W2, b2, W3, b3, w4, upd, hn, xo, h, W5, b5, W6, b6, ho,
                                     wn, bn, pq, next_kind=kind)
            same = torch.equal(hn, ref_hn) and torch.equal(ho, ref_h) and (not upd or torch.equal(xo, ref_x)) and \
                (not cols or torch.equal(pq, ref_pq))
            if not same:
                bad = it
                break
        torch.cuda.synchronize()
        ok = bad is None and bool(torch.isfinite(ref_h).all())
        n_fail += 0 if ok else 1
        print(f"layer kernel graphs {n_graphs:4d} n {n_nodes} k {k:2d} coords {int(upd)} next_kind {kind} next {int(cols > 0)}: "
              f"{'ok' if ok else f'DIFFERS from the two-launch path at launch {bad}'}", flush=True)
print("failures:", n_fail)
sys.exit(1 if n_fail else 0)
