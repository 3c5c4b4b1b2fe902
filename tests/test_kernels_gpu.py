"""Every CUDA kernel, called through the C ABI (ctypes), against its CPU contract
(oracle/kernel_contracts.py) on the same seeded inputs.  Integer outputs bit-exact; fp32 within 1e-5
of the result's scale (the north star's fp32 tolerance)."""
import types

import pytest
import torch

from immunostruct_b200 import _C
from immunostruct_b200.graph import GraphBatch
from immunostruct_b200.synthetic import synthetic_graph_arrays
from oracle import kernel_contracts as KC
from oracle import reference_ops as R

from helpers import close_per_segment, graph_segments

pytestmark = pytest.mark.gpu
DEV = "cuda"
TOL = 1e-5


def close(got, ref, tol=TOL, what=""):
    got, ref = got.detach().double().cpu(), ref.detach().double().cpu()
    assert got.shape == ref.shape, (what, got.shape, ref.shape)
    scale = float(ref.abs().max().clamp_min(1e-6))
    err = float((got - ref).abs().max())
    _log(f"{what}: err {err:.3e} scale {scale:.3e} rel {err / scale:.2e} nan={bool(torch.isnan(got).any())}")
    assert err <= tol * scale, f"{what}: max abs err {err:.3e} vs scale {scale:.3e} (rel {err / scale:.2e})"


def _log(msg):
    import os
    os.makedirs("gpurun_out", exist_ok=True)
    test = os.environ.get("PYTEST_CURRENT_TEST", "").split("::")[-1]
    with open("gpurun_out/kernel_errors.txt", "a") as f:
        f.write(f"{test} | {msg}\n")


def random_multigraph_arrays(seed, node_counts, mean_deg):
    """Ragged batch with multi-edges, self-free random endpoints, isolated nodes and varying in-degree."""
    gen = torch.Generator().manual_seed(seed)
    xs, srcs, dsts, ecs = [], [], [], []
    for n in node_counts:
        e = int(n * mean_deg) if n > 1 else 0
        dst = torch.randint(0, max(n - 2, 1), (e,), generator=gen)        # last two nodes get no in-edges
        src = (dst + 1 + torch.randint(0, max(n - 1, 1), (e,), generator=gen)) % n  # never a self loop
        x = torch.zeros(n, 23)
        x[torch.arange(n), torch.randint(0, 20, (n,), generator=gen)] = 1.0
        x[:, 20:] = torch.randn(n, 3, generator=gen) * 4.0
        xs.append(x); srcs.append(src); dsts.append(dst); ecs.append(e)
    return {"x": torch.cat(xs), "src": torch.cat(srcs), "dst": torch.cat(dsts),
            "edge_attr": torch.rand(sum(ecs), 1, generator=gen) + 0.5,
            "node_counts": torch.tensor(node_counts), "edge_counts": torch.tensor(ecs)}


def hub_and_isolated_arrays(seed, hub=128):
    """Edge cases of the tile walk: a run of 80 isolated nodes (edge-less tiles), hubs with in-degree 128 (the tile
    limit; hub=112: the limit of the two-stream edge backward, which hands larger batches to the lock-step kernel) and
    100, many in-degree-1 nodes (32-node tiles far below 128 edges), a graph without any edge."""
    gen = torch.Generator().manual_seed(seed)
    n0, n1 = 150, 90
    dst = torch.cat([torch.full((hub,), 80), torch.full((100,), 81), torch.arange(82, 150),
                     torch.randint(82, 150, (70,), generator=gen)])
    src = (dst + 1 + torch.randint(0, n0 - 1, (dst.numel(),), generator=gen)) % n0
    x = torch.zeros(n0 + n1, 23)
    x[torch.arange(n0 + n1), torch.randint(0, 20, (n0 + n1,), generator=gen)] = 1.0
    x[:, 20:] = torch.randn(n0 + n1, 3, generator=gen) * 4.0
    perm = torch.randperm(dst.numel(), generator=gen)                      # unsorted edge list
    return {"x": x, "src": src[perm], "dst": dst[perm], "edge_attr": torch.rand(dst.numel(), 1, generator=gen) + 0.5,
            "node_counts": torch.tensor([n0, n1]), "edge_counts": torch.tensor([dst.numel(), 0])}


def out_hub_arrays(seed):
    """Edge cases of the source-side (CSC) walk: out-degrees 100 and 40 (one node's run spans several 32-position
    chunks and 16-row batches), nodes without out-edges next to them, a trailing graph of a single node."""
    gen = torch.Generator().manual_seed(seed)
    n0 = 140
    src = torch.cat([torch.full((100,), 3), torch.full((40,), 4), torch.randint(8, n0, (200,), generator=gen)])
    dst = torch.cat([torch.arange(10, 110), torch.arange(60, 100), torch.randint(0, n0, (200,), generator=gen)])
    dst = torch.where(dst == src, (dst + 1) % n0, dst)
    x = torch.zeros(n0 + 1, 23)
    x[torch.arange(n0 + 1), torch.randint(0, 20, (n0 + 1,), generator=gen)] = 1.0
    x[:, 20:] = torch.randn(n0 + 1, 3, generator=gen) * 4.0
    perm = torch.randperm(src.numel(), generator=gen)
    return {"x": x, "src": src[perm], "dst": dst[perm], "edge_attr": torch.rand(src.numel(), 1, generator=gen) + 0.5,
            "node_counts": torch.tensor([n0, 1]), "edge_counts": torch.tensor([src.numel(), 0])}


CASES = {
    "hubs_isolated": lambda: hub_and_isolated_arrays(7),
    "out_hubs": lambda: out_hub_arrays(11),
    "knn_small": lambda: synthetic_graph_arrays(5, 37, 6, seed=3, n_pad=4, coord_scale=4.0),
    "knn_200": lambda: synthetic_graph_arrays(3, 200, 10, seed=4, n_pad=10),
    "ragged_multi": lambda: random_multigraph_arrays(5, [17, 1, 64, 33, 150, 2], 7.5),
}


def to_dev(arrays):
    return GraphBatch.from_arrays(*(arrays[k].to(DEV) for k in
                                    ("x", "src", "dst", "edge_attr", "node_counts", "edge_counts")))


def cpu_graph(gb):
    ns = types.SimpleNamespace()
    for f in ("indptr", "csr_src", "csr_dst", "csr_eid", "outptr", "csc_pos", "node_off"):
        setattr(ns, f, getattr(gb, f).cpu())
    ns.n_edges, ns.n_graphs, ns.max_nodes = gb.n_edges, gb.n_graphs, gb.max_nodes
    return ns


@pytest.fixture(params=sorted(CASES))
def case(request):
    arrays = CASES[request.param]()
    gb = to_dev(arrays)
    return arrays, gb, cpu_graph(gb)


# the backward tests add the tile limit of the two-stream edge backward (in-degree 112; "hubs_isolated" with its
# in-degree-128 hub exercises the device-side hand-over to the lock-step kernel)
BWD_CASES = dict(CASES, hubs_112=lambda: hub_and_isolated_arrays(9, hub=112))


@pytest.fixture(params=sorted(BWD_CASES))
def bwd_case(request):
    arrays = BWD_CASES[request.param]()
    gb = to_dev(arrays)
    return arrays, gb, cpu_graph(gb)


def rnd(gen, *shape, scale=1.0):
    return torch.randn(*shape, generator=gen) * scale


def egnn_weights(gen, f):
    s = 0.25
    return dict(W1=rnd(gen, 64, 2 * f + 2, scale=s), b1=rnd(gen, 64, scale=s), W2=rnd(gen, 64, 64, scale=s),
                b2=rnd(gen, 64, scale=s), W3=rnd(gen, 64, 64, scale=s), b3=rnd(gen, 64, scale=s),
                w4=rnd(gen, 1, 64, scale=s), W5=rnd(gen, 64, f + 64, scale=s), b5=rnd(gen, 64, scale=s),
                W6=rnd(gen, 64, 64, scale=s), b6=rnd(gen, 64, scale=s))


def dev(*ts):
    return [t.to(DEV) if t is not None else None for t in ts]


# ---- collation: bit exact ----------------------------------------------------------------------
def test_collate_bit_exact(case):
    arrays, gb, _ = case
    from immunostruct_b200.synthetic import split_graphs
    ref = R.dgl_batch(split_graphs(arrays))
    csr = R.csr_from_coo(ref["src"], ref["dst"], ref["num_nodes"])
    assert torch.equal(gb.edge_index.cpu(), torch.stack([ref["src"], ref["dst"]]))
    assert torch.equal(gb.batch.cpu(), R.batch_vector(ref["batch_num_nodes"]))
    off = torch.zeros(gb.n_graphs + 1, dtype=torch.int64)
    off[1:] = torch.cumsum(ref["batch_num_nodes"], 0)
    assert torch.equal(gb.node_off.cpu(), off)
    for k in ("indptr", "csr_src", "csr_dst", "csr_eid", "outptr", "csc_pos"):
        assert torch.equal(getattr(gb, k).cpu(), csr[k]), k
    deg = torch.bincount(ref["dst"], minlength=ref["num_nodes"])
    assert gb.stats.cpu().tolist()[:2] == [int(deg.max()), 0]
    gb.validate()


def test_collate_bit_exact_large_and_mixed_graphs():
    """Graphs above and below the shared-memory cursor capacity of the collation kernel (512 nodes) in one batch."""
    from immunostruct_b200.synthetic import split_graphs
    arrays = random_multigraph_arrays(13, [700, 3, 512, 513, 40], 6.0)
    gb = to_dev(arrays)
    ref = R.dgl_batch(split_graphs(arrays))
    csr = R.csr_from_coo(ref["src"], ref["dst"], ref["num_nodes"])
    assert torch.equal(gb.edge_index.cpu(), torch.stack([ref["src"], ref["dst"]]))
    for k in ("indptr", "csr_src", "csr_dst", "csr_eid", "outptr", "csc_pos"):
        assert torch.equal(getattr(gb, k).cpu(), csr[k]), k


def test_collate_flags_bad_endpoints():
    arrays = CASES["knn_small"]()
    arrays["src"][5] = 1000
    with pytest.raises(ValueError, match="outside"):        # at construction (first batch of a process) or at validate()
        to_dev(arrays).validate()


def test_cpu_tensors_are_rejected():
    with pytest.raises((RuntimeError, ValueError), match="CUDA"):
        _C.egnn_node_pre_fwd(torch.zeros(4, 64), torch.zeros(64, 130), torch.zeros(64), torch.zeros(4, 128))


# ---- EGNN forward ------------------------------------------------------------------------------
@pytest.mark.parametrize("f", [20, 64])
def test_egnn_forward_kernels(case, f):
    arrays, gb, cg = case
    gen = torch.Generator().manual_seed(11)
    n = gb.n_nodes
    w = egnn_weights(gen, f)
    h = arrays["x"][:, :20].clone() if f == 20 else rnd(gen, n, 64)
    x = arrays["x"][:, 20:].clone()
    ea = arrays["edge_attr"].float()
    # strided views for the 20-wide layer, exactly as the model slices ndata['x']
    x23 = arrays["x"].to(DEV)
    h_d = x23[:, :20] if f == 20 else h.to(DEV)
    x_d = x23[:, 20:]
    wd = {k: v.to(DEV) for k, v in w.items()}
    PQ_d, PQ = torch.empty(n, 128, device=DEV), torch.empty(n, 128)
    _C.egnn_node_pre_fwd(h_d, wd["W1"], wd["b1"], PQ_d)
    KC.egnn_node_pre_fwd(h, w["W1"], w["b1"], PQ)
    close(PQ_d, PQ, what="PQ")
    for upd in (True, False):
        hn_d, xo_d = torch.empty(n, 64, device=DEV), torch.empty(n, 3, device=DEV)
        hn, xo = torch.empty(n, 64), torch.empty(n, 3)
        _C.egnn_edge_fwd(gb, PQ_d, x_d, ea.to(DEV), f, wd["W1"], wd["W2"], wd["b2"], wd["W3"], wd["b3"], wd["w4"],
                         upd, hn_d, xo_d if upd else None)
        KC.egnn_edge_fwd(cg, PQ, x, ea, f, w["W1"], w["W2"], w["b2"], w["W3"], w["b3"], w["w4"], upd, hn, xo)
        close(hn_d, hn, what=f"hn upd={upd}")
        if upd:
            close(xo_d - x_d, xo - x, what="x' - x")
            close(xo_d, xo, what="x'")
    ho_d, ho = torch.empty(n, 64, device=DEV), torch.empty(n, 64)
    _C.egnn_node_post_fwd(h_d, hn_d, wd["W5"], wd["b5"], wd["W6"], wd["b6"], ho_d)
    KC.egnn_node_post_fwd(h, hn, w["W5"], w["b5"], w["W6"], w["b6"], ho)
    close(ho_d, ho, what="h'")
    assert int(gb.status.item()) == 0


@pytest.mark.parametrize("prec,tol", [(_C.PREC_BF16X3, 1e-5), (_C.PREC_TF32X3, 1e-5), (_C.PREC_BF16, 1e-2), (_C.PREC_FP16X2, 1e-5),
                                      (_C.PREC_BF16X3 | 16, 1e-5), (_C.PREC_BF16 | 16, 1e-2)])
@pytest.mark.parametrize("f", [20, 64])
def test_egnn_edge_forward_tensor_core(case, f, prec, tol):
    """tcgen05 edge kernels vs the same CPU contract: bf16x3 / 3xTF32 at the fp32 tolerance, bf16 at the north star's 1e-2.
    Default = the warp-specialised kernel; ``prec | 16`` = the lock-step first-generation kernel (SIMT
    destination-side sums), kept for A/B timing."""
    arrays, gb, cg = case
    gen = torch.Generator().manual_seed(37)
    n = gb.n_nodes
    w = egnn_weights(gen, f)
    wd = {k: v.to(DEV) for k, v in w.items()}
    PQ = rnd(gen, n, 128)
    x = arrays["x"][:, 20:].clone()
    ea = arrays["edge_attr"].float()
    x_d = arrays["x"].to(DEV)[:, 20:]
    for upd in (True, False):
        hn_d, xo_d = torch.empty(n, 64, device=DEV), torch.empty(n, 3, device=DEV)
        hn, xo = torch.empty(n, 64), torch.empty(n, 3)
        KC.egnn_edge_fwd(cg, PQ, x, ea, f, w["W1"], w["W2"], w["b2"], w["W3"], w["b3"], w["w4"], upd, hn, xo)
        for fast in (False, True):
            _C.egnn_edge_fwd_tc(gb, PQ.to(DEV), x_d, ea.to(DEV), f, wd["W1"], wd["W2"], wd["b2"], wd["W3"], wd["b3"],
                                wd["w4"], upd, prec, hn_d, xo_d if upd else None, fast_act=fast)
            close(hn_d, hn, tol, what=f"tc hn prec={prec} upd={upd} fast={fast}")
            if upd:
                close(xo_d - x_d, xo - x, tol, what=f"tc x'-x prec={prec} fast={fast}")
    assert int(gb.status.item()) == 0


def test_edge_kernels_at_benchmark_scale_match_the_simt_kernels():
    """Size-independent property at the benchmark shape (256 graphs x 200 nodes x 10-NN: 512 000 edges, every CTA walks
    ~30 tiles, both tile streams of the backward kernel busy): the tensor-core edge forward (bf16x3, both SiLU variants)
    and the two-stream edge backward reproduce the fp32 SIMT kernels of csrc/egnn.cu -- a different schedule, tile size and
    arithmetic path over the same CSR -- at the fp32 tolerance.  Catches wrong-row gathers that only appear at scale."""
    from immunostruct_b200.synthetic import synthetic_graph_arrays
    arr = synthetic_graph_arrays(256, 200, 10, seed=21, device=DEV)
    gb = GraphBatch.from_arrays(*(arr[k] for k in ("x", "src", "dst", "edge_attr", "node_counts", "edge_counts")), max_nodes=200)
    n, e = gb.n_nodes, gb.n_edges
    gen = torch.Generator().manual_seed(43)
    w = {k: v.to(DEV) for k, v in egnn_weights(gen, 64).items()}
    PQ, ghn, gxo = dev(rnd(gen, n, 128), rnd(gen, n, 64), rnd(gen, n, 3))
    x_d, ea = arr["x"][:, 20:], arr["edge_attr"].float()
    ref_hn, ref_x = torch.empty(n, 64, device=DEV), torch.empty(n, 3, device=DEV)
    _C.egnn_edge_fwd(gb, PQ, x_d, ea, 64, w["W1"], w["W2"], w["b2"], w["W3"], w["b3"], w["w4"], True, ref_hn, ref_x)
    for fast in (False, True):
        hn, xo = torch.full((n, 64), float("nan"), device=DEV), torch.full((n, 3), float("nan"), device=DEV)
        _C.egnn_edge_fwd_tc(gb, PQ, x_d, ea, 64, w["W1"], w["W2"], w["b2"], w["W3"], w["b3"], w["w4"], True, _C.PREC_BF16X3,
                            hn, xo, fast_act=fast)
        close(hn, ref_hn.cpu(), 1e-5, what=f"scale hn fast={fast}")
        close(xo - x_d, (ref_x - x_d).cpu(), 1e-5, what=f"scale x'-x fast={fast}")
    grid = _C.egnn_edge_bwd_grid(n)
    outs = {}
    for name in ("egnn_edge_bwd", "egnn_edge_bwd_ws"):
        o = [torch.full((e, 64), float("nan"), device=DEV), torch.full((n, 64), float("nan"), device=DEV),
             torch.full((e, 3), float("nan"), device=DEV), torch.full((n, 3), float("nan"), device=DEV),
             torch.full((grid, 8512), float("nan"), device=DEV)]        # a partial block no CTA writes stays NaN
        getattr(_C, name)(gb, PQ, x_d, ea, 64, w["W1"], w["W2"], w["b2"], w["W3"], w["b3"], w["w4"], ghn, gxo, *o)
        assert bool(torch.isfinite(o[4]).all()), name
        red = torch.empty(8512, device=DEV)
        _C.reduce_partials(o[4], red)
        outs[name] = o[:4] + [red]
    for nm, a, b in zip(("gz1", "gQ", "gD", "gxd"), outs["egnn_edge_bwd_ws"], outs["egnn_edge_bwd"]):
        close(a, b.cpu(), 1e-5, what=f"scale {nm}")
    ra, rb = outs["egnn_edge_bwd_ws"][4], outs["egnn_edge_bwd"][4].cpu()
    for nm, lo, hi in (("gW2", 0, 4096), ("gW3", 4096, 8192), ("gb2", 8192, 8256), ("gb3", 8256, 8320), ("gw4", 8320, 8384),
                       ("gwr", 8384, 8448), ("gwa", 8448, 8512)):
        close(ra[lo:hi], rb[lo:hi], 2e-5, what=f"scale {nm}")       # 512 000-term fp32 sums in two different orders
    assert int(gb.status.item()) == 0


@pytest.mark.parametrize("prec,tol,fast", [pytest.param(_C.PREC_BF16X3, 1e-5, True, id="3-1e-05"),
                                           pytest.param(_C.PREC_BF16, 1e-2, True, id="0-0.01"),
                                           pytest.param(_C.PREC_FP16X2, 1e-5, True, id="4-1e-05"),
                                           pytest.param(_C.PREC_BF16X3, 1e-5, False, id="3-1e-05-accurate_silu")])
@pytest.mark.parametrize("f,with_next", [(20, True), (64, True), (64, False)])
def test_egnn_node_post_pre_tensor_core(case, f, with_next, prec, tol, fast):
    """Fused node_post(l) + node_pre(l+1) tcgen05 kernel vs the CPU contracts of the two SIMT kernels; fast=False is the
    accurate-SiLU instance the training forward runs."""
    arrays, gb, _ = case
    gen = torch.Generator().manual_seed(41)
    n = gb.n_nodes
    w, wn = egnn_weights(gen, f), egnn_weights(gen, 64)
    h = arrays["x"][:, :20].clone() if f == 20 else rnd(gen, n, 64)
    hn = rnd(gen, n, 64, scale=3.0)
    h_d = arrays["x"].to(DEV)[:, :20] if f == 20 else h.to(DEV)
    ho, PQn = torch.empty(n, 64), torch.empty(n, 128)
    ho_d, PQn_d = torch.full((n, 64), float("nan"), device=DEV), torch.full((n, 128), float("nan"), device=DEV)
    KC.egnn_node_post_pre_tc(h, hn, w["W5"], w["b5"], w["W6"], w["b6"], ho, wn["W1"] if with_next else None,
                             wn["b1"] if with_next else None, PQn if with_next else None, prec)
    _C.egnn_node_post_pre_tc(h_d, hn.to(DEV), *dev(w["W5"], w["b5"], w["W6"], w["b6"]), ho_d,
                             *(dev(wn["W1"], wn["b1"]) if with_next else (None, None)),
                             PQn_d if with_next else None, prec, fast_act=fast)
    close(ho_d, ho, tol, what=f"node tc h' prec={prec} f={f} fast={fast}")
    if with_next:
        close(PQn_d, PQn, tol, what=f"node tc PQ' prec={prec} f={f} fast={fast}")


@pytest.mark.parametrize("prec,tol", [(_C.PREC_BF16X3, 1e-5), (_C.PREC_BF16, 1e-2), (_C.PREC_FP16X2, 1e-5)])
def test_egnn_node_post_qkv_tensor_core(case, prec, tol):
    """Last-layer node kernel with the attention projections fused (next_kind = 2): h' and QKV = h' [Wq;Wk;Wv]^T + b."""
    arrays, gb, _ = case
    gen = torch.Generator().manual_seed(43)
    n = gb.n_nodes
    w = egnn_weights(gen, 64)
    h, hn = rnd(gen, n, 64), rnd(gen, n, 64, scale=3.0)
    Wqkv, bqkv = rnd(gen, 192, 64, scale=0.3), rnd(gen, 192, scale=0.3)
    ho, QKV = torch.empty(n, 64), torch.empty(n, 192)
    ho_d, QKV_d = torch.full((n, 64), float("nan"), device=DEV), torch.full((n, 192), float("nan"), device=DEV)
    KC.egnn_node_post_pre_tc(h, hn, w["W5"], w["b5"], w["W6"], w["b6"], ho, Wqkv, bqkv, QKV, prec, next_kind=2)
    _C.egnn_node_post_pre_tc(h.to(DEV), hn.to(DEV), *dev(w["W5"], w["b5"], w["W6"], w["b6"]), ho_d,
                             *dev(Wqkv, bqkv), QKV_d, prec, next_kind=2)
    close(ho_d, ho, tol, what=f"node tc (qkv tail) h' prec={prec}")
    close(QKV_d, QKV, tol, what=f"node tc QKV prec={prec}")


@pytest.mark.parametrize("prec,tol", [(_C.PREC_BF16X3, 1e-5), (_C.PREC_BF16, 1e-2)])
@pytest.mark.parametrize("m,n,k,relu,bias", [(512, 512, 5943, True, True),      # vae_fc1: split-K, unaligned rows
                                              (512, 5943, 512, False, True),     # vae_fc4: ragged N
                                              (376, 32, 512, False, True),       # vae_fc21 on the last partial batch
                                              (7, 130, 40, True, False),         # tiny, ragged everything
                                              (129, 129, 65, False, True)])
def test_linear_tensor_core(m, n, k, relu, bias, prec, tol):
    """tcgen05 Linear vs the fp64 product: bf16x3 at the fp32 tolerance, bf16 at 1e-2 (of the result's scale)."""
    gen = torch.Generator().manual_seed(47)
    x, w = rnd(gen, m, k), rnd(gen, n, k, scale=0.3)
    b = rnd(gen, n) if bias else None
    ref = x.double() @ w.double().T + (b.double() if bias else 0.0)
    ref = torch.relu(ref) if relu else ref
    out = _C.linear_tc(x.to(DEV), w.to(DEV), b.to(DEV) if bias else None, relu=relu, precision=prec)
    close(out, ref.float(), tol, what=f"linear_tc {m}x{n}x{k} prec={prec}")
    # one-hot rows (the real vae_fc1 input) and a strided input view
    if k == 5943:
        oh = torch.zeros(m, 283, 21)
        oh.scatter_(2, torch.randint(0, 21, (m, 283, 1), generator=gen), 1.0)
        oh = oh.reshape(m, k)
        ref = torch.relu(oh.double() @ w.double().T + b.double())
        close(_C.linear_tc(oh.to(DEV), w.to(DEV), b.to(DEV), relu=True, precision=prec), ref.float(), tol, what="linear_tc one-hot")
    big = rnd(gen, m, k + 5).to(DEV)
    ref = big[:, 2:2 + k].double().cpu() @ w.double().T
    close(_C.linear_tc(big[:, 2:2 + k], w.to(DEV), None, precision=prec), ref.float(), tol, what="linear_tc strided view")


@pytest.mark.parametrize("b", [512, 5])
def test_vae_mid_and_head_kernels(b):
    """Eval-mode small-layer fusions (csrc/head.cu) vs their torch contracts."""
    gen = torch.Generator().manual_seed(53)
    h1, prop, eps = rnd(gen, b, 512).abs(), torch.rand(b, 2, generator=gen), rnd(gen, b, 32)
    ws = dict(Wp0=rnd(gen, 32, 2), bp0=rnd(gen, 32), Wp3=rnd(gen, 8, 32), bp3=rnd(gen, 8), W21=rnd(gen, 32, 512, scale=0.1),
              b21=rnd(gen, 32), W22=rnd(gen, 32, 512, scale=0.05), b22=rnd(gen, 32), W3=rnd(gen, 512, 40), b3=rnd(gen, 512))
    ref = KC.vae_mid_infer(h1, prop, eps, *ws.values())
    got = _C.vae_mid_infer(h1.to(DEV), prop.to(DEV), eps.to(DEV), *(v.to(DEV) for v in ws.values()))
    for name, r, g_ in zip(("mu", "logvar", "z_vae", "h3"), ref, got):
        close(g_, r, what=f"vae_mid {name}")
    pooled, zv = rnd(gen, b, 64), ref[2]
    Wc, bc, coef = rnd(gen, 64, 64, scale=0.3), rnd(gen, 64), rnd(gen, 33, scale=0.5)
    W1, b1, W2, b2 = rnd(gen, 32, 104, scale=0.3), rnd(gen, 32), rnd(gen, 1, 32), rnd(gen, 1)
    for use_wc, use_coef, use_w2 in ((True, True, True), (False, False, True), (True, True, False)):
        args = (pooled, Wc if use_wc else None, bc if use_wc else None, zv, coef if use_coef else None, 8, W1, b1,
                W2 if use_w2 else None, b2 if use_w2 else None)
        rx, ro = KC.head_infer(*args)
        gx, go = _C.head_infer(*(a.to(DEV) if torch.is_tensor(a) else a for a in args))
        close(gx, rx, what="head x_gat"); close(go, ro, what=f"head out wc={use_wc} fusion={use_coef} out={use_w2}")


# ---- EGNN backward -----------------------------------------------------------------------------
@pytest.mark.parametrize("tc", [False, True, "ws"])
@pytest.mark.parametrize("f,coord", [(64, True), (64, False), (20, True)])
def test_egnn_backward_kernels(bwd_case, f, coord, tc):
    """tc=True: the tcgen05 edge backward (bf16x3) against the same contract at the same tolerance; "ws": its two-stream
    successor (112-edge tiles; the in-degree-128 case exercises the device-side hand-over to the lock-step kernel)."""
    arrays, gb, cg = bwd_case
    edge_bwd = {False: _C.egnn_edge_bwd, True: _C.egnn_edge_bwd_tc, "ws": _C.egnn_edge_bwd_ws}[tc]
    gen = torch.Generator().manual_seed(13)
    n, e = gb.n_nodes, gb.n_edges
    w = egnn_weights(gen, f)
    wd = {k: v.to(DEV) for k, v in w.items()}
    h = arrays["x"][:, :20].clone() if f == 20 else rnd(gen, n, 64)
    x = arrays["x"][:, 20:].clone()
    ea = arrays["edge_attr"].float()
    x23 = arrays["x"].to(DEV)
    h_d = x23[:, :20] if f == 20 else h.to(DEV)
    x_d = x23[:, 20:]
    PQ, hn = torch.empty(n, 128), torch.empty(n, 64)
    KC.egnn_node_pre_fwd(h, w["W1"], w["b1"], PQ)
    KC.egnn_edge_fwd(cg, PQ, x, ea, f, w["W1"], w["W2"], w["b2"], w["W3"], w["b3"], w["w4"], False, hn, None)
    PQ_d, hn_d = PQ.to(DEV), hn.to(DEV)
    gh_out, gx_out = rnd(gen, n, 64), (rnd(gen, n, 3) if coord else None)
    need_gh = f == 64
    k = f + 64
    # node_post backward
    grid_n = _C.egnn_node_grid(n)
    ghd_d = torch.empty(n, 64, device=DEV) if need_gh else None
    ghn_d, pp_d = torch.empty(n, 64, device=DEV), torch.empty(grid_n, 64 * k + 64 + 4096 + 64, device=DEV)
    ghd = torch.empty(n, 64) if need_gh else None
    ghn, pp = torch.empty(n, 64), torch.empty(KC.FAKE_GRID, 64 * k + 64 + 4096 + 64)
    node_post_bwd = _C.egnn_node_post_bwd_tc if tc else _C.egnn_node_post_bwd
    node_post_bwd(gh_out.to(DEV), h_d, hn_d, wd["W5"], wd["b5"], wd["W6"], ghd_d, ghn_d, pp_d)
    KC.egnn_node_post_bwd(gh_out, h, hn, w["W5"], w["b5"], w["W6"], ghd, ghn, pp)
    close(ghn_d, ghn, what="ghn")
    if need_gh:
        close(ghd_d, ghd, what="gh_direct")
    rp_d = torch.empty(pp_d.shape[1], device=DEV)
    _C.reduce_partials(pp_d, rp_d)
    rp = pp.sum(0)
    for name, a, b in (("gW5", 0, 64 * k), ("gb5", 64 * k, 64 * k + 64), ("gW6", 64 * k + 64, 64 * k + 64 + 4096),
                       ("gb6", 64 * k + 64 + 4096, 64 * k + 128 + 4096)):
        close(rp_d[a:b], rp[a:b], what=name)
    # edge backward
    grid_e = _C.egnn_edge_bwd_grid(n)
    outs_d = [torch.empty(e, 64, device=DEV), torch.empty(n, 64, device=DEV), torch.empty(e, 3, device=DEV),
              torch.empty(n, 3, device=DEV), torch.empty(grid_e, 8512, device=DEV)]
    outs = [torch.empty(e, 64), torch.empty(n, 64), torch.empty(e, 3), torch.empty(n, 3), torch.empty(KC.FAKE_GRID, 8512)]
    # (each kernel is checked in isolation: it consumes the CONTRACT's upstream values, not the device's)
    edge_bwd(gb, PQ_d, x_d, ea.to(DEV), f, wd["W1"], wd["W2"], wd["b2"], wd["W3"], wd["b3"], wd["w4"],
             ghn.to(DEV), gx_out.to(DEV) if coord else None, *outs_d)
    KC.egnn_edge_bwd(cg, PQ, x, ea, f, w["W1"], w["W2"], w["b2"], w["W3"], w["b3"], w["w4"], ghn, gx_out, *outs)
    for name, a, b in zip(("gz1", "gQ", "gD", "gxd"), outs_d[:4], outs[:4]):
        close(a, b, what=name)
    re_d = torch.empty(8512, device=DEV)
    _C.reduce_partials(outs_d[4], re_d)
    re = outs[4].sum(0)
    names = [("gW2", 0, 4096), ("gb2", 8192, 8256), ("gwr", 8384, 8448), ("gwa", 8448, 8512)]
    if coord:
        names += [("gW3", 4096, 8192), ("gb3", 8256, 8320), ("gw4", 8320, 8384)]
    for name, a, b in names:
        close(re_d[a:b], re[a:b], what=name)
    # node_pre backward
    gz1_d, gQ_d, gD_d, gxd_d = outs_d[:4]
    gz1, gQ, gD, gxd = outs[:4]
    gh_d = torch.empty(n, 64, device=DEV) if need_gh else None
    gx_d = torch.empty(n, 3, device=DEV)
    p3_d = torch.empty(grid_n, 2 * 64 * f + 64, device=DEV)
    gh = torch.empty(n, 64) if need_gh else None
    gx, p3 = torch.empty(n, 3), torch.empty(KC.FAKE_GRID, 2 * 64 * f + 64)
    node_pre_bwd = _C.egnn_node_pre_bwd_tc if tc else _C.egnn_node_pre_bwd
    node_pre_bwd(gz1.to(DEV), gQ.to(DEV), gD.to(DEV), gxd.to(DEV), gx_out.to(DEV) if coord else None,
                 ghd.to(DEV) if need_gh else None, gb, h_d, wd["W1"], gh_d, gx_d, p3_d)
    KC.egnn_node_pre_bwd(gz1, gQ, gD, gxd, gx_out, ghd, cg, h, w["W1"], gh, gx, p3)
    close(gx_d, gx, what="gx")
    if need_gh:
        close(gh_d, gh, what="gh")
    r3_d = torch.empty(p3_d.shape[1], device=DEV)
    _C.reduce_partials(p3_d, r3_d)
    r3 = p3.sum(0)
    for name, a, b in (("gWs", 0, 64 * f), ("gWd", 64 * f, 128 * f), ("gb1", 128 * f, 128 * f + 64)):
        close(r3_d[a:b], r3[a:b], what=name)
    assert int(gb.status.item()) == 0


@pytest.mark.parametrize("kernel", ["egnn_edge_bwd", "egnn_edge_bwd_ws"])
def test_backward_is_deterministic(bwd_case, kernel):
    """Same inputs twice -> bit-identical gradients (no floating-point atomics anywhere; the two tile streams of the
    ws kernel accumulate into separate TMEM blocks that are added in a fixed order)."""
    arrays, gb, _ = bwd_case
    gen = torch.Generator().manual_seed(17)
    n, e = gb.n_nodes, gb.n_edges
    w = {k: v.to(DEV) for k, v in egnn_weights(gen, 64).items()}
    PQ, ghn, gx_out = dev(rnd(gen, n, 128), rnd(gen, n, 64), rnd(gen, n, 3))
    x_d, ea = arrays["x"].to(DEV)[:, 20:], arrays["edge_attr"].float().to(DEV)
    res = []
    for _ in range(2):
        outs = [torch.empty(e, 64, device=DEV), torch.empty(n, 64, device=DEV), torch.empty(e, 3, device=DEV),
                torch.empty(n, 3, device=DEV), torch.empty(_C.egnn_edge_bwd_grid(n), 8512, device=DEV)]
        getattr(_C, kernel)(gb, PQ, x_d, ea, 64, w["W1"], w["W2"], w["b2"], w["W3"], w["b3"], w["w4"], ghn, gx_out, *outs)
        red = torch.empty(8512, device=DEV)
        _C.reduce_partials(outs[4], red)
        res.append([o.clone() for o in outs[:4]] + [red])
    for a, b in zip(*res):
        assert torch.equal(a, b)


# ---- attention + pooling -----------------------------------------------------------------------
@pytest.mark.parametrize("n_head", [1, 8])
def test_attention_pool_kernels(case, n_head):
    """Pooled rows and gQKV are compared per graph (helpers.close_per_segment): the input gradient of a graph scales
    with 1 / its node count, so against the scale of the whole tensor a 150-node graph next to 1-node graphs would be
    checked at ~1e-3 of its own size."""
    arrays, gb, cg = case
    gen = torch.Generator().manual_seed(19)
    n, b = gb.n_nodes, gb.n_graphs
    gseg, nseg = torch.arange(b), graph_segments(cg.node_off)
    QKV = rnd(gen, n, 192, scale=0.7)
    O, LSE, pooled = torch.empty(n, 64), torch.empty(n, n_head), torch.empty(b, 64)
    O_d, LSE_d, pooled_d = (torch.empty_like(t, device=DEV) for t in (O, LSE, pooled))
    _C.attn_pool_fwd(QKV.to(DEV), gb.node_off, n_head, gb.max_nodes, O_d, LSE_d, pooled_d)
    KC.attn_pool_fwd(QKV, cg.node_off, n_head, gb.max_nodes, O, LSE, pooled)
    close(O_d, O, what="O"); close(LSE_d, LSE, what="LSE")
    close_per_segment(pooled_d, pooled, gseg, TOL, what="pooled")
    pooled_i = torch.full((b, 64), float("nan"), device=DEV)
    _C.attn_pool_infer(QKV.to(DEV), gb.node_off, n_head, gb.max_nodes, pooled_i)
    close_per_segment(pooled_i, pooled, gseg, TOL, what="pooled (inference kernel)")
    if n_head == 1:
        for prec, tol in ((_C.PREC_BF16X3, 1e-5), (_C.PREC_FP16X2, 1e-5), (_C.PREC_BF16, 1e-2)):
            pooled_t = torch.full((b, 64), float("nan"), device=DEV)
            _C.attn_pool_infer_tc(QKV.to(DEV), gb.node_off, gb.max_nodes, pooled_t, prec)
            close_per_segment(pooled_t, pooled, gseg, tol, what=f"pooled (tensor-core inference kernel, prec={prec})")
            if prec == _C.PREC_BF16:
                # (no peaked-softmax case for plain bf16: with scores of magnitude ~100 the bf16 rounding of Q and K
                #  alone moves a score by ~0.4, i.e. a probability by tens of percent -- a property of the input
                #  format, not of the kernel; the 1e-2 bound is a statement about well-scaled activations)
                continue
            big = QKV.to(DEV) * 6.0                 # peaked softmax rows
            ref_big = torch.empty(b, 64)
            KC.attn_pool_infer(QKV * 6.0, cg.node_off, 1, gb.max_nodes, ref_big)
            _C.attn_pool_infer_tc(big, gb.node_off, gb.max_nodes, pooled_t, prec)
            close_per_segment(pooled_t, ref_big, gseg, tol, what=f"pooled tc peaked prec={prec}")
    g_pooled, gO = rnd(gen, b, 64), rnd(gen, n, 64)
    for gp, go in ((g_pooled, None), (g_pooled, gO), (None, gO)):
        gQKV, gQKV_d = torch.empty(n, 192), torch.empty(n, 192, device=DEV)
        _C.attn_pool_bwd(QKV.to(DEV), O_d, LSE_d, gb.node_off, n_head, gb.max_nodes,
                         gp.to(DEV) if gp is not None else None, go.to(DEV) if go is not None else None, gQKV_d)
        KC.attn_pool_bwd(QKV, O, LSE, cg.node_off, n_head, gb.max_nodes, gp, go, gQKV)
        close_per_segment(gQKV_d, gQKV, nseg, TOL, what=f"gQKV pooled={gp is not None} full={go is not None}")
        if gp is not None and go is None:                    # O = None: row statistics recomputed inside the kernel
            gQKV_r, lse_r = torch.full((n, 192), float("nan"), device=DEV), torch.empty(n, n_head, device=DEV)
            _C.attn_pool_bwd(QKV.to(DEV), None, lse_r, gb.node_off, n_head, gb.max_nodes, gp.to(DEV), None, gQKV_r)
            close_per_segment(gQKV_r, gQKV, nseg, TOL, what="gQKV pooled-only, recomputed statistics")
            close(lse_r, LSE, what="recomputed LSE")
            if n_head == 1:                                  # tensor-core backward (bf16x3): same contract
                for mult in (1.0, 6.0):                      # 6.0: peaked softmax rows
                    gQKV_t = torch.full((n, 192), float("nan"), device=DEV)
                    _C.attn_pool_bwd_tc(QKV.to(DEV) * mult, gb.node_off, gb.max_nodes, gp.to(DEV), gQKV_t)
                    ref_t = torch.empty(n, 192)
                    O_m, LSE_m, pooled_m = torch.empty(n, 64), torch.empty(n, 1), torch.empty(b, 64)
                    KC.attn_pool_fwd(QKV * mult, cg.node_off, 1, gb.max_nodes, O_m, LSE_m, pooled_m)
                    KC.attn_pool_bwd(QKV * mult, O_m, LSE_m, cg.node_off, 1, gb.max_nodes, gp, None, ref_t)
                    # x6: scores of magnitude ~100, where ONE fp32 ulp of a score (7.6e-6) is already a relative error
                    # of 7.6e-6 in exp(score) -- the fp32 oracle itself is no closer to the exact gradient than that
                    close_per_segment(gQKV_t, ref_t, nseg, 1e-5 if mult == 1.0 else 3e-5,
                                      what=f"gQKV tensor-core backward x{mult}")


def test_attention_weights_output():
    arrays = CASES["knn_small"]()
    gb = to_dev(arrays)
    gen = torch.Generator().manual_seed(23)
    n, b, m, hh = gb.n_nodes, gb.n_graphs, gb.max_nodes, 8
    QKV = rnd(gen, n, 192)
    attn_d = torch.empty(b, hh, m, m, device=DEV)
    off = torch.arange(b, device=DEV, dtype=torch.int64) * (hh * m * m)
    O_d, LSE_d, pooled_d = torch.empty(n, 64, device=DEV), torch.empty(n, hh, device=DEV), torch.empty(b, 64, device=DEV)
    _C.attn_pool_fwd(QKV.to(DEV), gb.node_off, hh, m, O_d, LSE_d, pooled_d, attn_d, off)
    ref = torch.stack([KC._attn_graph(QKV[i * m:(i + 1) * m], hh)[1] for i in range(b)])
    close(attn_d, ref, what="attention weights")


# ---- fusion attention --------------------------------------------------------------------------
@pytest.mark.parametrize("L,H", [(104, 8), (208, 8), (7, 2)])
def test_fusion_attention_kernels(L, H):
    gen = torch.Generator().manual_seed(29)
    b = 9
    c, coef, gout = rnd(gen, b, L), rnd(gen, 4 * H + 1, scale=0.8), rnd(gen, b, L)
    out, out_d = torch.empty(b, L), torch.empty(b, L, device=DEV)
    _C.fusion_attn_fwd(c.to(DEV), H, coef.to(DEV), out_d)
    KC.fusion_attn_fwd(c, H, coef, out)
    close(out_d, out, what="fusion out")
    gc, gp = torch.empty(b, L), torch.empty(b, 4 * H)
    gc_d, gp_d = torch.empty(b, L, device=DEV), torch.empty(b, 4 * H, device=DEV)
    _C.fusion_attn_bwd(c.to(DEV), H, coef.to(DEV), gout.to(DEV), gc_d, gp_d)
    KC.fusion_attn_bwd(c, H, coef, gout, gc, gp)
    close(gc_d, gc, what="fusion gc")
    close(gp_d.sum(0), gp.sum(0), what="fusion gcoef")


# ---- losses ------------------------------------------------------------------------------------
@pytest.mark.parametrize("mode,seqflag,b", [pytest.param(mode, seqflag, b, id=f"{mode}-{seqflag}" + ("" if b == 37 else f"-b{b}"))
                                           for b in (37, 512, 511)
                                           for mode, seqflag in ((0, True), (1, True), (0, False), (1, False))])
def test_loss_kernels(mode, seqflag, b):
    """b = 37: each of the recon kernels' 592 CTAs makes less than one pass over the float4 groups; b = 512 (the
    benchmark batch): several passes; b = 511: several passes and a tail that is not a multiple of 4."""
    gen = torch.Generator().manual_seed(31)
    s, z = 5943, 32
    recon, seq = rnd(gen, b, s), (torch.rand(b, s, generator=gen) < 0.05).float()
    mu, lv, logits = rnd(gen, b, z), rnd(gen, b, z, scale=0.3), rnd(gen, b, scale=2.0)
    y = (torch.rand(b, generator=gen) < 0.3).float() if mode == 0 else rnd(gen, b)
    wts = ((5.0, 0.1, 0.1) if mode == 0 else (2.0, 0.5, 0.5)) if seqflag else (1.0, 0.0, 0.0)
    args = (recon, seq, mu, lv) if seqflag else (None, None, None, None)
    out, out_d = torch.empty(4), torch.empty(4, device=DEV)
    part = torch.empty(_C.loss_num_partials(), device=DEV)
    _C.loss_fwd(*dev(*args), logits.to(DEV), y.to(DEV), mode, 4.25, *wts, part, out_d)
    KC.loss_fwd(*args, logits, y, mode, 4.25, *wts, None, out)
    close(out_d[:1], out[:1], what="loss")
    close(out_d, out, what="loss components")
    gout = torch.tensor([0.7])
    g = [torch.empty(b, s), torch.empty(b, z), torch.empty(b, z), torch.empty(b)]
    g_d = [torch.empty_like(t, device=DEV) for t in g]
    if not seqflag:
        g[:3], g_d[:3] = [None] * 3, [None] * 3
    _C.loss_bwd(*dev(*args), logits.to(DEV), y.to(DEV), mode, 4.25, *wts, gout.to(DEV), *g_d)
    KC.loss_bwd(*args, logits, y, mode, 4.25, *wts, gout, *g)
    for name, a, bb in zip(("g_recon", "g_mu", "g_logvar", "g_logits"), g_d, g):
        if a is not None:
            close(a, bb, what=name)
