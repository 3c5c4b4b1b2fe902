"""The persistent kernels past their first pass, against fp64 runs of their CPU contracts.

Most hot-path kernels launch min(work units, CTA cap) CTAs and loop ``for (t = blockIdx.x; t < n; t += gridDim.x)``.
The second and later passes run code the first never does: weight-gradient MMAs that accumulate onto the previous
tile's (``accumulate = started``), waits on the previous tile's in-flight MMA, the prefetched next CSC run, mbarrier
phases carried from one tile or graph to the next, shared memory and TMEM reused by a graph of another size.  The
sizes below are derived from the SM count and each launcher's grid formula (R rows per pass, at most C CTAs):
  one_pass          M = R C            every CTA runs exactly one pass (the boundary);
  cta0_second_pass  M = R C + 1        only CTA 0 takes a second pass, with one valid row;
  multi_pass        M = R (2C + 5) + 77  every CTA runs two or three passes, the last tile is ragged;
  bench             M = 102 400        the benchmark's training batch (512 graphs x 200 nodes).
The reference is the kernel's contract (oracle/kernel_contracts.py) run in fp64.  Elementwise outputs are compared per
segment (a 128-row tile, or a graph), reduced weight gradients by the rule of conftest.assert_grads_close.  Every output
and partial buffer starts as NaN, so a row or partial block that no CTA wrote fails."""
import contextlib
import time

import pytest
import torch

import immunostruct_b200 as I
from immunostruct_b200 import _C
from immunostruct_b200.synthetic import synthetic_graph_arrays
from oracle import kernel_contracts as KC

from conftest import assert_grads_close, rel_err
from helpers import (close_per_segment, concat_graphs, fp64_default, graph_batch, graph_segments, inject_eps, log_error,
                     named_grads, oracle_training_step, tile_segments)
from test_kernels_gpu import cpu_graph, egnn_weights, out_hub_arrays, random_multigraph_arrays, rnd, to_dev
from test_models_gpu import _bench_shape_case

pytestmark = pytest.mark.gpu
DEV = "cuda"
TOL = 1e-5
TOL_PEAKED = 3e-5          # x6 scores (magnitude ~100): one fp32 ulp of a score is 7.6e-6 of exp(score) (DESIGN.md section 2)
SIZES = ("one_pass", "cta0_second_pass", "multi_pass", "bench")
BENCH_NODES = 102400


def rows_for(size, r, c):
    return {"one_pass": r * c, "cta0_second_pass": r * c + 1, "multi_pass": r * (2 * c + 5) + 77,
            "bench": BENCH_NODES}[size]


def nan(*shape):
    return torch.full(shape, float("nan"), device=DEV)


def dev(*ts):
    return [t.to(DEV) if t is not None else None for t in ts]


def contract(dtype):
    """Run a contract in ``dtype``: fp64 needs the default dtype switched, fp32 is the default."""
    return fp64_default() if dtype is torch.float64 else contextlib.nullcontext()


def reduced_grads_close(got_flat, ref32_flat, ref64_flat, layout, what):
    """Reduced weight gradients (one flat partial row): within max(1e-5 scale, 3 |contract_fp32 - contract_fp64|)."""
    got = {n: got_flat[a:b] for n, a, b in layout}
    r32 = {n: ref32_flat[a:b] for n, a, b in layout}
    r64 = {n: ref64_flat[a:b] for n, a, b in layout}
    assert bool(torch.isfinite(got_flat).all()), what
    assert_grads_close(got, r32, TOL, truth=r64)


def ragged_batch(m, seed):
    """Ragged graphs of {1, 2, 17, 37, 64, 128, 129, 150, 200} nodes (isolated nodes, multi-edges) whose node counts sum
    to ``m``; the last 141 nodes are out_hub_arrays (out-degree-100 and -40 sources, a trailing 1-node graph)."""
    hub = out_hub_arrays(seed)
    rest, counts, sizes = m - int(hub["node_counts"].sum()), [], (1, 2, 37, 150, 200, 64, 17, 128, 129)
    while rest > 0:
        counts.append(min(sizes[len(counts) % len(sizes)], rest))
        rest -= counts[-1]
    return concat_graphs(random_multigraph_arrays(seed, counts, 4.0), hub)


# ---- 1. node backward ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("f", [20, 64])
@pytest.mark.parametrize("size", SIZES)
def test_node_backward_past_the_first_tile(size, f):
    """egnn_node_post_bwd(_tc) and egnn_node_pre_bwd(_tc) at 128 rows per pass and one CTA per SM: ghn, gh_direct, gh and
    gx per tile, the reduced gW5 gb5 gW6 gb6 / gWs gWd gb1, and bit-identical reruns of the tensor-core kernels."""
    sms = _C.num_sms()
    m = rows_for(size, 128, sms)
    grid = _C.egnn_node_grid(m)
    assert grid == min((m + 127) // 128, sms)
    arrays = ragged_batch(m, seed=61 + f)
    gb = to_dev(arrays)
    cg = cpu_graph(gb)
    assert gb.n_nodes == m
    e = gb.n_edges
    gen = torch.Generator().manual_seed(67)
    w = egnn_weights(gen, f)
    x23, h64 = rnd(gen, m, 23), rnd(gen, m, 64)
    h = x23[:, :20] if f == 20 else h64
    h_d = x23.to(DEV)[:, :20] if f == 20 else h64.to(DEV)          # the 20-wide layer reads a strided view of x23
    hn, gh_out = rnd(gen, m, 64, scale=3.0), rnd(gen, m, 64)
    gz1, gQ, gD, gxd = rnd(gen, e, 64), rnd(gen, m, 64), rnd(gen, e, 3), rnd(gen, m, 3)
    gx_out, gh_direct = rnd(gen, m, 3), rnd(gen, m, f)
    tiles = tile_segments(m)
    k = f + 64
    W5, b5, W6, W1 = w["W5"], w["b5"], w["W6"], w["W1"]
    d = dict(zip(("gh_out", "hn", "W5", "b5", "W6", "W1", "gz1", "gQ", "gD", "gxd", "gx_out", "gh_direct"),
                 dev(gh_out, hn, W5, b5, W6, W1, gz1, gQ, gD, gxd, gx_out, gh_direct)))

    # node_post backward
    post_layout = (("gW5", 0, 64 * k), ("gb5", 64 * k, 64 * k + 64), ("gW6", 64 * k + 64, 64 * k + 64 + 4096),
                   ("gb6", 64 * k + 64 + 4096, 64 * k + 128 + 4096))
    stride = 64 * k + 128 + 4096
    for want_direct in (True, False):
        ref = {}
        for dt in (torch.float32, torch.float64):
            with contract(dt):
                ghd, ghn, pp = (torch.empty(m, f, dtype=dt) if want_direct else None), torch.empty(m, 64, dtype=dt), \
                    torch.empty(1, stride, dtype=dt)
                KC.egnn_node_post_bwd(*(t.to(dt) for t in (gh_out, h, hn, W5, b5, W6)), ghd, ghn, pp)
            ref[dt] = (ghd, ghn, pp[0])
        for name, kern, reps in (("tc", _C.egnn_node_post_bwd_tc, 2), ("simt", _C.egnn_node_post_bwd, 1)):
            runs = []
            for _ in range(reps):
                ghd_d, ghn_d, pp_d = (nan(m, f) if want_direct else None), nan(m, 64), nan(grid, stride)
                kern(d["gh_out"], h_d, d["hn"], d["W5"], d["b5"], d["W6"], ghd_d, ghn_d, pp_d)
                runs.append([t for t in (ghd_d, ghn_d, pp_d) if t is not None])
            if reps == 2:
                assert all(torch.equal(a, b) for a, b in zip(*runs)), f"node_post_bwd_tc is not reproducible ({size})"
            ghd_d, ghn_d, pp_d = (runs[0] if want_direct else [None] + runs[0])
            what = f"node_post_bwd {name} {size} M={m} f={f} direct={want_direct}"
            close_per_segment(ghn_d, ref[torch.float64][1], tiles, TOL, what=what + " ghn")
            if want_direct:
                close_per_segment(ghd_d, ref[torch.float64][0], tiles, TOL, what=what + " gh_direct")
            assert bool(torch.isfinite(pp_d).all()), what + ": a partial block was not written"
            red = torch.empty(stride, device=DEV)
            _C.reduce_partials(pp_d, red)
            reduced_grads_close(red.cpu(), ref[torch.float32][2], ref[torch.float64][2], post_layout, what)

    # node_pre backward
    pre_layout = (("gWs", 0, 64 * f), ("gWd", 64 * f, 128 * f), ("gb1", 128 * f, 128 * f + 64))
    stride = 128 * f + 64
    for use_direct, use_gxo, want_gh in ((True, True, True), (False, False, True), (False, True, False)):
        ref = {}
        for dt in (torch.float32, torch.float64):
            with contract(dt):
                gh, gx, p3 = (torch.empty(m, f, dtype=dt) if want_gh else None), torch.empty(m, 3, dtype=dt), \
                    torch.empty(1, stride, dtype=dt)
                KC.egnn_node_pre_bwd(gz1.to(dt), gQ.to(dt), gD.to(dt), gxd.to(dt), gx_out.to(dt) if use_gxo else None,
                                     gh_direct.to(dt) if use_direct else None, cg, h.to(dt), W1.to(dt), gh, gx, p3)
            ref[dt] = (gh, gx, p3[0])
        for name, kern, reps in (("tc", _C.egnn_node_pre_bwd_tc, 2), ("simt", _C.egnn_node_pre_bwd, 1)):
            runs = []
            for _ in range(reps):
                gh_d, gx_d, p3_d = (nan(m, f) if want_gh else None), nan(m, 3), nan(grid, stride)
                kern(d["gz1"], d["gQ"], d["gD"], d["gxd"], d["gx_out"] if use_gxo else None,
                     d["gh_direct"] if use_direct else None, gb, h_d, d["W1"], gh_d, gx_d, p3_d)
                runs.append([t for t in (gh_d, gx_d, p3_d) if t is not None])
            if reps == 2:
                assert all(torch.equal(a, b) for a, b in zip(*runs)), f"node_pre_bwd_tc is not reproducible ({size})"
            gh_d, gx_d, p3_d = (runs[0] if want_gh else [None] + runs[0])
            what = f"node_pre_bwd {name} {size} M={m} f={f} direct={use_direct} gx_out={use_gxo} gh={want_gh}"
            close_per_segment(gx_d, ref[torch.float64][1], tiles, TOL, what=what + " gx")
            if want_gh:
                close_per_segment(gh_d, ref[torch.float64][0], tiles, TOL, what=what + " gh")
            assert bool(torch.isfinite(p3_d).all()), what + ": a partial block was not written"
            red = torch.empty(stride, device=DEV)
            _C.reduce_partials(p3_d, red)
            reduced_grads_close(red.cpu(), ref[torch.float32][2], ref[torch.float64][2], pre_layout, what)
    assert int(gb.status.item()) == 0


# ---- 2. node forward -------------------------------------------------------------------------------------------------
NODE_TC_PRECS = [pytest.param(_C.PREC_BF16X3, True, TOL, id="bf16x3"),
                 pytest.param(_C.PREC_BF16X3, False, TOL, id="bf16x3_accurate_silu"),      # the training forward
                 pytest.param(_C.PREC_FP16X2, True, TOL, id="fp16x2"),
                 pytest.param(_C.PREC_BF16, True, 1e-2, id="bf16")]


@pytest.mark.parametrize("prec,fast,tol", NODE_TC_PRECS)
@pytest.mark.parametrize("f,next_kind", [(20, 1), (64, 1), (64, 2), (64, None)])
@pytest.mark.parametrize("size", SIZES)
def test_node_post_pre_tc_past_the_first_tile(size, f, next_kind, prec, fast, tol):
    """Fused node_post(l) + node_pre(l+1) / QKV / nothing: fp16x2 with next_kind 1 hands over 256 rows (two tiles) per
    pass, bf16 runs two CTAs per SM; h' and PQ' / QKV per 128-row tile."""
    sms = _C.num_sms()
    r = 256 if prec == _C.PREC_FP16X2 and next_kind != 2 else 128
    m = rows_for(size, r, 2 * sms if prec == _C.PREC_BF16 else sms)
    gen = torch.Generator().manual_seed(71)
    w = egnn_weights(gen, f)
    x23, h64 = rnd(gen, m, 23), rnd(gen, m, 64)
    h = x23[:, :20] if f == 20 else h64
    h_d = x23.to(DEV)[:, :20] if f == 20 else h64.to(DEV)
    hn = rnd(gen, m, 64, scale=3.0)
    if next_kind == 2:
        Wn, bn, width = rnd(gen, 192, 64, scale=0.3), rnd(gen, 192, scale=0.3), 192
    else:
        wn = egnn_weights(gen, 64)
        Wn, bn, width = wn["W1"], wn["b1"], 128
    if next_kind is None:
        Wn = bn = None
    with fp64_default():
        ho = torch.empty(m, 64, dtype=torch.float64)
        PQn = torch.empty(m, width, dtype=torch.float64) if Wn is not None else None
        KC.egnn_node_post_pre_tc(h.double(), hn.double(), *(w[k].double() for k in ("W5", "b5", "W6", "b6")), ho,
                                 Wn.double() if Wn is not None else None, bn.double() if bn is not None else None, PQn,
                                 prec, next_kind=next_kind or 1)
    ho_d, PQn_d = nan(m, 64), (nan(m, width) if Wn is not None else None)
    _C.egnn_node_post_pre_tc(h_d, hn.to(DEV), *dev(w["W5"], w["b5"], w["W6"], w["b6"]), ho_d, *dev(Wn, bn), PQn_d, prec,
                             fast_act=fast, next_kind=next_kind or 1)
    tiles = tile_segments(m)
    what = f"node_post_pre_tc {size} M={m} f={f} next={next_kind} prec={prec} fast={fast}"
    close_per_segment(ho_d, ho, tiles, tol, what=what + " h'")
    if Wn is not None:
        close_per_segment(PQn_d, PQn, tiles, tol, what=what + (" QKV" if next_kind == 2 else " PQ'"))


@pytest.mark.parametrize("f", [20, 64])
@pytest.mark.parametrize("size", SIZES)
def test_simt_node_forward_past_the_first_tile(size, f):
    """fp32-mode node kernels: node_pre_fwd runs up to four CTAs per SM, node_post_fwd one (egnn_node_grid)."""
    sms = _C.num_sms()
    gen = torch.Generator().manual_seed(73)
    w = egnn_weights(gen, f)
    for kernel, cap in (("egnn_node_pre_fwd", 4 * sms), ("egnn_node_post_fwd", sms)):
        m = rows_for(size, 128, cap)
        x23, h64, hn = rnd(gen, m, 23), rnd(gen, m, 64), rnd(gen, m, 64, scale=3.0)
        h = x23[:, :20] if f == 20 else h64
        h_d = x23.to(DEV)[:, :20] if f == 20 else h64.to(DEV)
        with fp64_default():
            if kernel == "egnn_node_pre_fwd":
                ref = torch.empty(m, 128, dtype=torch.float64)
                KC.egnn_node_pre_fwd(h.double(), w["W1"].double(), w["b1"].double(), ref)
            else:
                ref = torch.empty(m, 64, dtype=torch.float64)
                KC.egnn_node_post_fwd(h.double(), hn.double(), *(w[k].double() for k in ("W5", "b5", "W6", "b6")), ref)
        got = nan(*ref.shape)
        if kernel == "egnn_node_pre_fwd":
            _C.egnn_node_pre_fwd(h_d, *dev(w["W1"], w["b1"]), got)
        else:
            _C.egnn_node_post_fwd(h_d, hn.to(DEV), *dev(w["W5"], w["b5"], w["W6"], w["b6"]), got)
        close_per_segment(got, ref, tile_segments(m), TOL, what=f"{kernel} {size} M={m} f={f}")


# ---- 3. edge kernels, several tiles per CTA --------------------------------------------------------------------------
def _hub_in_degree(arrays, node=5, degree=128):
    """Graph 0 of a k-NN batch gets an in-degree-``degree`` hub: edges of graph 0 that neither start nor end at ``node``
    are redirected to it (the two-stream edge backward hands such a batch to its lock-step kernel)."""
    dst, src = arrays["dst"].clone(), arrays["src"]
    e0 = int(arrays["edge_counts"][0])
    have = int((dst[:e0] == node).sum())
    cand = torch.nonzero((src[:e0] != node) & (dst[:e0] != node)).flatten()[:degree - have]
    dst[cand] = node
    return dict(arrays, dst=dst)


@pytest.fixture(scope="module", params=["knn", "hub128"])
def edge_batch(request):
    """64 graphs x 200 nodes x 10-NN: 12 800 nodes, 128 000 edges -- every edge CTA walks several tiles."""
    arrays = synthetic_graph_arrays(64, 200, 10, seed=79)
    arrays["edge_attr"] = torch.rand(arrays["edge_attr"].shape, generator=torch.Generator().manual_seed(83)) + 0.5
    if request.param == "hub128":
        arrays = _hub_in_degree(arrays)
    gb = to_dev(arrays)
    if request.param == "hub128":
        assert int(gb.stats[0]) == 128
    return request.param, arrays, gb, cpu_graph(gb)


EDGE_LAYOUT = (("gW2", 0, 4096), ("gW3", 4096, 8192), ("gb2", 8192, 8256), ("gb3", 8256, 8320), ("gw4", 8320, 8384),
               ("gwr", 8384, 8448), ("gwa", 8448, 8512))


@pytest.mark.parametrize("coord", [True, False])
@pytest.mark.parametrize("f", [20, 64])
def test_edge_backward_several_tiles_per_cta(edge_batch, f, coord):
    """egnn_edge_bwd, egnn_edge_bwd_tc and egnn_edge_bwd_ws; coord=False is the last layer of every training step."""
    variant, arrays, gb, cg = edge_batch
    n, e = gb.n_nodes, gb.n_edges
    gen = torch.Generator().manual_seed(89)
    w = egnn_weights(gen, f)
    PQ, ghn, gxo = rnd(gen, n, 128), rnd(gen, n, 64), rnd(gen, n, 3)
    x, ea = arrays["x"][:, 20:].clone(), arrays["edge_attr"].float()
    x_d = arrays["x"].to(DEV)[:, 20:]
    names = ("W1", "W2", "b2", "W3", "b3", "w4")
    ref = {}
    for dt in (torch.float32, torch.float64):
        with contract(dt):
            outs = [torch.empty(e, 64, dtype=dt), torch.empty(n, 64, dtype=dt), torch.empty(e, 3, dtype=dt),
                    torch.empty(n, 3, dtype=dt), torch.empty(1, 8512, dtype=dt)]
            W = [w[k].to(dt) for k in names]
            KC.egnn_edge_bwd(cg, PQ.to(dt), x.to(dt), ea.to(dt), f, *W, ghn.to(dt), gxo.to(dt) if coord else None, *outs)
        ref[dt] = outs
    grid = _C.egnn_edge_bwd_grid(n)
    wd = dev(*(w[k] for k in names))
    edge_rows, node_rows = tile_segments(e), tile_segments(n)
    for kernel in ("egnn_edge_bwd", "egnn_edge_bwd_tc", "egnn_edge_bwd_ws"):
        o = [nan(e, 64), nan(n, 64), nan(e, 3), nan(n, 3), nan(grid, 8512)]
        getattr(_C, kernel)(gb, PQ.to(DEV), x_d, ea.to(DEV), f, *wd, ghn.to(DEV), gxo.to(DEV) if coord else None, *o)
        what = f"{kernel} {variant} f={f} coord={coord}"
        for nm, got, r, seg in zip(("gz1", "gQ", "gD", "gxd"), o[:4], ref[torch.float64][:4],
                                   (edge_rows, node_rows, edge_rows, node_rows)):
            close_per_segment(got, r, seg, TOL, what=f"{what} {nm}")
        assert bool(torch.isfinite(o[4]).all()), what + ": a partial block was not written"
        red = torch.empty(8512, device=DEV)
        _C.reduce_partials(o[4], red)
        reduced_grads_close(red.cpu(), ref[torch.float32][4][0], ref[torch.float64][4][0], EDGE_LAYOUT, what)
    assert int(gb.status.item()) == 0


def test_edge_forward_several_tiles_per_cta(edge_batch):
    """egnn_edge_fwd (fp32) and egnn_edge_fwd_tc (bf16x3 / fp16x2, both SiLU variants), with and without coordinates."""
    variant, arrays, gb, cg = edge_batch
    n = gb.n_nodes
    for f in (20, 64):
        gen = torch.Generator().manual_seed(97 + f)
        w = egnn_weights(gen, f)
        PQ = rnd(gen, n, 128)
        x, ea = arrays["x"][:, 20:].clone(), arrays["edge_attr"].float()
        x_d = arrays["x"].to(DEV)[:, 20:]
        names = ("W1", "W2", "b2", "W3", "b3", "w4")
        wd = dev(*(w[k] for k in names))
        seg = tile_segments(n)
        for upd in (True, False):
            with fp64_default():
                hn, xo = torch.empty(n, 64, dtype=torch.float64), torch.empty(n, 3, dtype=torch.float64)
                KC.egnn_edge_fwd(cg, PQ.double(), x.double(), ea.double(), f, *(w[k].double() for k in names), upd, hn, xo)
            runs = [("simt", None, None)] + [(p, p, fast) for p in ("bf16x3", "fp16x2") for fast in (False, True)]
            for name, prec, fast in runs:
                hn_d, xo_d = nan(n, 64), (nan(n, 3) if upd else None)
                if prec is None:
                    _C.egnn_edge_fwd(gb, PQ.to(DEV), x_d, ea.to(DEV), f, *wd, upd, hn_d, xo_d)
                else:
                    code = {"bf16x3": _C.PREC_BF16X3, "fp16x2": _C.PREC_FP16X2}[prec]
                    _C.egnn_edge_fwd_tc(gb, PQ.to(DEV), x_d, ea.to(DEV), f, *wd, upd, code, hn_d, xo_d, fast_act=fast)
                what = f"edge_fwd {name} {variant} f={f} upd={upd} fast={fast}"
                close_per_segment(hn_d, hn, seg, TOL, what=what + " hn")
                if upd:
                    close_per_segment(xo_d - x_d, xo - x.double(), seg, TOL, what=what + " x'-x")
    assert int(gb.status.item()) == 0


# ---- 4. attention past the first graph -------------------------------------------------------------------------------
ATTN_FAMILIES = {"npad128": (1, 2, 37, 127, 128), "npad256": (1, 2, 129, 200, 255, 256)}
ATTN_GRAPHS = ("S", "S+1", "2S+3", "512")


@pytest.fixture(scope="module", params=[(fam, g) for fam in sorted(ATTN_FAMILIES) for g in ATTN_GRAPHS],
                ids=lambda p: f"{p[0]}-G={p[1]}")
def attn_case(request):
    """Ragged graphs: size[g] = sizes[(g + g // S) % len(sizes)], so the graphs one CTA takes in turn change size."""
    fam, gname = request.param
    sms = _C.num_sms()
    n_graphs = {"S": sms, "S+1": sms + 1, "2S+3": 2 * sms + 3, "512": 512}[gname]
    sizes = ATTN_FAMILIES[fam]
    counts = torch.tensor([sizes[(g + g // sms) % len(sizes)] for g in range(n_graphs)])
    off = torch.zeros(n_graphs + 1, dtype=torch.int64)
    off[1:] = torch.cumsum(counts, 0)
    n = int(off[-1])
    QKV = rnd(torch.Generator().manual_seed(101), n, 192, scale=0.7)
    return f"{fam} G={n_graphs}", QKV, off, int(counts.max())


def _attn_ref(fn, *args, out_shapes):
    with fp64_default():
        outs = [torch.empty(*s, dtype=torch.float64) for s in out_shapes]
        fn(*(a.double() if torch.is_tensor(a) and a.is_floating_point() else a for a in args), *outs)
    return outs


def test_attention_infer_tc_past_the_first_graph(attn_case):
    name, QKV, off, mx = attn_case
    b = off.numel() - 1
    gseg = torch.arange(b)
    off_d = off.to(DEV)
    for mult in (1.0, 6.0):
        ref, = _attn_ref(KC.attn_pool_infer, QKV * mult, off, 1, mx, out_shapes=[(b, 64)])
        for prec, tol in ((_C.PREC_BF16X3, TOL), (_C.PREC_FP16X2, TOL), (_C.PREC_BF16, 1e-2)):
            if mult != 1.0 and prec == _C.PREC_BF16:
                continue          # bf16 Q and K move a score of magnitude ~100 by ~0.4 (test_kernels_gpu.py)
            pooled = nan(b, 64)
            _C.attn_pool_infer_tc(QKV.to(DEV) * mult, off_d, mx, pooled, prec)
            close_per_segment(pooled, ref, gseg, tol if mult == 1.0 else TOL_PEAKED,
                              what=f"attn_pool_infer_tc {name} prec={prec} x{mult}")


def test_attention_bwd_tc_past_the_first_graph(attn_case):
    name, QKV, off, mx = attn_case
    b, n = off.numel() - 1, QKV.shape[0]
    gp = rnd(torch.Generator().manual_seed(103), b, 64)
    nseg = graph_segments(off)
    off_d = off.to(DEV)
    for mult in (1.0, 6.0):
        ref, = _attn_ref(KC.attn_pool_bwd_tc, QKV * mult, off, mx, gp, out_shapes=[(n, 192)])
        runs = []
        for _ in range(2):
            gQKV = nan(n, 192)
            _C.attn_pool_bwd_tc(QKV.to(DEV) * mult, off_d, mx, gp.to(DEV), gQKV)
            runs.append(gQKV)
        assert torch.equal(runs[0], runs[1]), f"attn_pool_bwd_tc is not reproducible ({name})"
        close_per_segment(runs[0], ref, nseg, TOL if mult == 1.0 else TOL_PEAKED,
                          what=f"attn_pool_bwd_tc {name} x{mult}")


@pytest.mark.parametrize("n_head", [1, 8])
def test_attention_simt_past_the_first_graph(attn_case, n_head):
    """fp32-mode attention: attn_pool_fwd (O, LSE, pooled), attn_pool_infer, attn_pool_bwd (pooled / full / both
    upstream gradients, stored and recomputed row statistics)."""
    name, QKV, off, mx = attn_case
    b, n = off.numel() - 1, QKV.shape[0]
    gen = torch.Generator().manual_seed(107)
    g_pooled, gO = rnd(gen, b, 64), rnd(gen, n, 64)
    nseg, gseg = graph_segments(off), torch.arange(b)
    off_d = off.to(DEV)
    for mult in (1.0, 6.0):
        tol = TOL if mult == 1.0 else TOL_PEAKED
        what = f"{name} heads={n_head} x{mult}"
        Q = QKV * mult
        O, LSE, pooled = _attn_ref(KC.attn_pool_fwd, Q, off, n_head, mx, out_shapes=[(n, 64), (n, n_head), (b, 64)])
        O_d, LSE_d, pooled_d = nan(n, 64), nan(n, n_head), nan(b, 64)
        _C.attn_pool_fwd(Q.to(DEV), off_d, n_head, mx, O_d, LSE_d, pooled_d)
        close_per_segment(O_d, O, nseg, tol, what=f"attn_pool_fwd O {what}")
        close_per_segment(LSE_d, LSE, nseg, tol, what=f"attn_pool_fwd LSE {what}")
        close_per_segment(pooled_d, pooled, gseg, tol, what=f"attn_pool_fwd pooled {what}")
        pooled_i = nan(b, 64)
        _C.attn_pool_infer(Q.to(DEV), off_d, n_head, mx, pooled_i)
        close_per_segment(pooled_i, pooled, gseg, tol, what=f"attn_pool_infer {what}")
        for gp, go in ((g_pooled, None), (g_pooled, gO), (None, gO)):
            ref, = _attn_ref(KC.attn_pool_bwd, Q, O, LSE, off, n_head, mx, gp, go, out_shapes=[(n, 192)])
            gQKV = nan(n, 192)
            _C.attn_pool_bwd(Q.to(DEV), O_d, LSE_d, off_d, n_head, mx, *dev(gp, go), gQKV)
            close_per_segment(gQKV, ref, nseg, tol, what=f"attn_pool_bwd {what} pooled={gp is not None} full={go is not None}")
            if go is None:                       # O = None: the kernel recomputes the row statistics
                gQKV_r, lse_r = nan(n, 192), nan(n, n_head)
                _C.attn_pool_bwd(Q.to(DEV), None, lse_r, off_d, n_head, mx, gp.to(DEV), None, gQKV_r)
                close_per_segment(gQKV_r, ref, nseg, tol, what=f"attn_pool_bwd recomputed statistics {what}")
                close_per_segment(lse_r, LSE, nseg, tol, what=f"attn_pool_bwd recomputed LSE {what}")


# ---- 5. reduce_partials3 ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("f", [20, 64])
def test_reduce_partials3_equals_three_reductions_bit_for_bit(f):
    """The one-launch reduction of a training step's three partial buffers (node_post, edge, node_pre) at the benchmark
    batch equals three reduce_partials calls bit for bit: the same CTA order, no other association."""
    nparts = _C.egnn_node_grid(BENCH_NODES)
    strides = (64 * (f + 64) + 128 + 4096, 8512, 128 * f + 64)
    gen = torch.Generator().manual_seed(109)
    # magnitudes over six decades: a different summation order would show in the last bits
    parts = [(rnd(gen, nparts, s) * torch.exp(rnd(gen, nparts, s) * 3.0)).to(DEV) for s in strides]
    outs3 = [nan(s) for s in strides]
    _C.reduce_partials3(parts, outs3)
    for p, o3, s in zip(parts, outs3, strides):
        o1 = nan(s)
        _C.reduce_partials(p, o1)
        assert bool(torch.isfinite(o3).all()) and torch.equal(o3, o1), (f, s)


# ---- 6. the training step at batch 512 -------------------------------------------------------------------------------
TRAIN_BATCH, TRAIN_SEED, ORACLE_CHUNK = 512, 113, 64
# Weight gradients at batch 512 are sums over 102 400 nodes / 1 024 000 edges, accumulated tile by tile per CTA and then
# over the CTAs; the oracle's fp32 run sums them in another blocking, so at this size "3 x the fp32 oracle's own error"
# no longer bounds the product's rounding.  Measured on one NVIDIA B200 (1000 W): 3.5e-5 of the assert_grads_close scale
# in the bf16x3 mode (edge_mlp.2.weight, the 64 x 64 edge-MLP layer), 1.9e-5 in the fp32 mode (the attention key
# projection).  test_edge_kernels_at_benchmark_scale_match_the_simt_kernels already allows 2e-5 between two fp32 orders of
# 512 000-term sums.  A multi-pass defect is far above this: a tile missing from one weight gradient is ~1e-3 of it.
GRAD_TOL_512 = 5e-5


@pytest.fixture(scope="module")
def train_case():
    """HybridModelv2 at the benchmark shape and batch, with the full-model oracle's logits, loss and gradients in fp32
    and fp64, each computed once in chunks of 64 graphs (the 512-graph oracle in one piece would need ~40 GB)."""
    arr, dense, model, eps = _bench_shape_case(TRAIN_BATCH, seed=TRAIN_SEED)
    state = {k: v.cpu() for k, v in model.state_dict().items()}
    t0 = time.time()
    ref = {dt: oracle_training_step(state, arr, dense, eps, dt, chunk=ORACLE_CHUNK) for dt in (torch.float32, torch.float64)}
    log_error(f"batch-512 oracle (fp32 + fp64, chunks of {ORACLE_CHUNK}): {time.time() - t0:.1f} s")
    return arr, dense, model.to(DEV).eval(), eps, ref


@pytest.mark.parametrize("mode", ["default", "fp32"])
def test_training_step_at_batch_512_against_fp64(train_case, mode):
    """The default mode trains on the bf16x3 tensor-core kernels, "fp32" on the SIMT kernels: logits per sample and the
    loss within 1e-5 of fp64, every parameter gradient by the rule of assert_grads_close at GRAD_TOL_512."""
    arr, dense, model, eps, ref = train_case
    out32, _, grads32 = ref[torch.float32]
    out64, loss64, grads64 = ref[torch.float64]
    assert float(out64.std()) > 1e-4 * float(out64.abs().mean())          # outputs do depend on the graph
    default_precision = I.get_precision()
    try:
        if mode != "default":
            I.set_precision(mode)
        model.zero_grad(set_to_none=True)
        inject_eps(model, eps)
        gb = graph_batch(arr, DEV).validate()
        seq, prop, y = (dense[k].to(DEV) for k in ("seq", "prop", "target"))
        recon, mu, logvar, out = model(gb, seq, prop)
        loss = I.Losses(5943, [4.25, 1.0], sequence=True).BCE_loss(recon, seq, mu, logvar, out, y)
        loss.backward()
    finally:
        I.set_precision(default_precision)
    close_per_segment(out.reshape(-1, 1), out64.reshape(-1, 1), torch.arange(TRAIN_BATCH), TOL,
                      what=f"batch-512 logits {mode}")
    log_error(f"batch-512 loss {mode}: rel err {rel_err(loss, loss64):.3e}")
    assert rel_err(loss, loss64) < TOL
    assert_grads_close(named_grads(model), grads32, GRAD_TOL_512, truth=grads64)
