"""Predictive mean and spread over the reparameterisation draw on the B200: the multi-draw head kernel
(is_head_mc_infer) against its contract, bit-identity of every draw with the fused eval forward, the fp64 oracle per
draw, independence of the number of draws and of the chunking, the statistics, one trunk pass whatever K, and no side
effects on parameter gradients."""
import pytest
import torch

import immunostruct_b200 as I
from immunostruct_b200 import _C
from immunostruct_b200.predictive import predictive, predictive_pair
from immunostruct_b200.synthetic import split_graphs, synthetic_dense, synthetic_graph_arrays
from oracle import reference_ops as R

from helpers import graph_batch, inject_eps
from test_predictive_host import head_mc_infer_contract

pytestmark = pytest.mark.gpu
DEV = "cuda"
TOL = 1e-5


@pytest.fixture
def precision(request):
    prev = I.get_precision()
    I.set_precision(request.param)
    yield request.param
    I.set_precision(prev)


def _close(got, ref, tol=TOL):
    ref = ref.detach().double().cpu()
    err = float((got.detach().double().cpu() - ref).abs().max())
    assert err <= tol * max(float(ref.abs().max()), 1e-30), (err, float(ref.abs().max()))


def _gen(seed):
    return torch.Generator().manual_seed(seed)


# ---- the kernel against its contract -------------------------------------------------------------------------------
def _kernel_case(b, k, n_items, heads, with_wc, seed=0):
    g = _gen(seed)
    r = lambda *s: torch.randn(*s, generator=g)
    items = [(r(b, 64), r(b, 32) * 0.5, r(b, 32) * 0.5, r(b, 40).abs(), r(k, b, 32)) for _ in range(n_items)]
    L = n_items * 104
    Wc, bc = (r(64, 64) * 0.125, r(64) * 0.1) if with_wc else (None, None)
    coef = torch.cat([r(2 * heads) * 0.3, r(2 * heads), r(1)]) if heads else None
    return items, (Wc, bc, coef, heads, r(32, L) * 0.1, r(32) * 0.1, r(1, 32) * 0.2, r(1) * 0.1)


def _run_kernel(items, params):
    return _C.head_mc_infer([tuple(t.to(DEV) for t in it) for it in items],
                            *[p if p is None or isinstance(p, int) else p.to(DEV) for p in params])


def _check_against_contract(items, params, logits, bs, ks):
    """The contract in fp64 on the samples ``bs`` and the draws ``ks`` (a logit depends on (sample, eps[k]) only)."""
    sub = [tuple(t[bs].double() for t in it[:4]) + (it[4][ks][:, bs].double(),) for it in items]
    p64 = [p if isinstance(p, int) or p is None else p.double() for p in params]
    ref, _, _ = head_mc_infer_contract(sub, *p64)
    _close(logits.cpu()[bs][:, ks], ref)


def _check_stats(logits, mean, std):
    p = torch.sigmoid(logits.double())
    assert float((mean.double() - p.mean(1)).abs().max()) <= 1e-7
    assert float((std.double() - p.std(1, unbiased=False)).abs().max()) <= 1e-7


@pytest.mark.parametrize("b", [1, 5, 512])
@pytest.mark.parametrize("k", [1, 3, 64, 257])
@pytest.mark.parametrize("n_items", [1, 2])
def test_head_mc_kernel_against_contract(b, k, n_items):
    assert hasattr(_C.lib(), "is_head_mc_infer")
    for heads, with_wc in ((0, False), (0, True), (8, False), (8, True)):
        items, params = _kernel_case(b, k, n_items, heads, with_wc, seed=b * 1000 + k + n_items)
        logits, mean, std = _run_kernel(items, params)
        assert logits.shape == (b, k) and mean.shape == (b,) and std.shape == (b,)
        bs = sorted({0, b // 2, b - 1, *torch.randint(0, b, (5,), generator=_gen(k)).tolist()})
        ks = sorted({0, k // 2, k - 1, *torch.randint(0, k, (5,), generator=_gen(b)).tolist()})
        _check_against_contract(items, params, logits, bs, ks)
        _check_stats(logits, mean, std)
        again = _run_kernel(items, params)
        assert all(torch.equal(x, y) for x, y in zip((logits, mean, std), again))


def test_head_mc_kernel_draw_and_chunk_independence():
    items, params = _kernel_case(512, 257, 2, 8, True, seed=3)
    full = _run_kernel(items, params)
    eight = _run_kernel([it[:4] + (it[4][:8],) for it in items], params)
    assert torch.equal(full[0][:, :8], eight[0])
    one = _run_kernel([it[:4] + (it[4][:1],) for it in items], params)
    assert torch.equal(one[0][:, 0], full[0][:, 0]) and torch.equal(one[2], torch.zeros_like(one[2]))
    big, bparams = _kernel_case(1, 4096, 1, 8, True, seed=4)
    logits, mean, std = _run_kernel(big, bparams)
    ks = sorted({0, 7, 8, 2047, 4095, *torch.randint(0, 4096, (12,), generator=_gen(9)).tolist()})
    _check_against_contract(big, bparams, logits, [0], ks)
    _check_stats(logits, mean, std)


# ---- full models ------------------------------------------------------------------------------------------------------
def _case(b, seed, name, n_pad=10, **kw):
    arr = synthetic_graph_arrays(b, 200, 10, seed=seed, n_pad=n_pad)
    dense = synthetic_dense(b, seed=seed)
    torch.manual_seed(seed)
    model = I.model_map[name](vae_input_dim=5943, device=DEV, **kw).to(DEV).eval()
    return graph_batch(arr, DEV), arr, dense["seq"].to(DEV), dense["prop"].to(DEV), model


def _eps(k, b, seed):
    return torch.randn(k, b, 32, generator=_gen(seed)).to(DEV)


@pytest.mark.parametrize("precision", ["fp16x2", "bf16x3", "bf16"], indirect=True)
@pytest.mark.parametrize("name", ["HybridModel", "HybridModelv2", "HybridModel_SSL", "HybridModelv2_SSL"])
def test_draws_equal_the_fused_forward(precision, name):
    g, _, seq, prop, model = _case(512, 41, name)
    eps = _eps(6, 512, 42)
    res = predictive(model, g, seq, prop, eps=eps)
    for k in (0, 2, 5):
        inject_eps(model, eps[k])
        with torch.no_grad():
            ref = model(g, seq, prop)[3].reshape(-1)
        if name.endswith("_SSL"):            # the last Linear of the SSL forward runs in torch, after the fused head
            _close(res.logits[:, k], ref)
        else:
            assert torch.equal(res.logits[:, k], ref), (k, float((res.logits[:, k] - ref).abs().max()))


def _state64(model):
    return {k: v.detach().double().cpu() for k, v in model.state_dict().items()}


def _og64(arr):
    og = R.dgl_batch(split_graphs(arr))
    return dict(og, x=og["x"].double(), edge_attr=og["edge_attr"].double())


@pytest.mark.parametrize("precision", ["fp16x2", "bf16x3", "fp32", "bf16"], indirect=True)
@pytest.mark.parametrize("name,version", [("HybridModel", "v1"), ("HybridModelv2", "v2")])
def test_hybrid_draws_match_fp64_oracle(precision, name, version):
    g, arr, seq, prop, model = _case(6, 51, name)
    eps = _eps(3, 6, 52)
    res = predictive(model, g, seq, prop, eps=eps)
    p, og = _state64(model), _og64(arr)
    ref = torch.stack([R.hybrid_forward(p, og, seq.double().cpu(), prop.double().cpu(), eps[k].double().cpu(),
                                        version=version)[3].reshape(-1) for k in range(3)], 1)
    _close(res.logits, ref, 1e-2 if precision == "bf16" else TOL)
    _check_stats(res.logits, res.prob_mean, res.prob_std)


@pytest.mark.parametrize("precision", ["fp16x2", "bf16x3", "fp32", "bf16"], indirect=True)
@pytest.mark.parametrize("use_wt", [True, False])
def test_comparative_draws_match_fp64_oracle_and_forward(precision, use_wt):
    gc, arr_c, seq_c, prop_c, model = _case(5, 61, "HybridModelv2_Comparative", use_wt_for_downstream=use_wt)
    arr_w = synthetic_graph_arrays(5, 200, 10, seed=62, n_pad=10)
    dw = synthetic_dense(5, seed=62)
    gw, seq_w, prop_w = graph_batch(arr_w, DEV), dw["seq"].to(DEV), dw["prop"].to(DEV)
    eps_c, eps_w = _eps(3, 5, 63), _eps(3, 5, 64)
    tol = 1e-2 if precision == "bf16" else TOL
    res = predictive_pair(model, (gc, gw), (seq_c, seq_w), (prop_c, prop_w), eps=(eps_c, eps_w))
    p, ogs = _state64(model), (_og64(arr_c), _og64(arr_w))
    cpu = lambda t: t.double().cpu()
    ref = torch.stack([R.comparative_forward(p, ogs, (cpu(seq_c), cpu(seq_w)), (cpu(prop_c), cpu(prop_w)),
                                             (cpu(eps_c[k]), cpu(eps_w[k])), use_wt=use_wt)[4].reshape(-1)
                       for k in range(3)], 1)
    _close(res.logits, ref, tol)
    fwd = []
    for k in range(3):
        inject_eps(model, eps_c[k], eps_w[k])
        with torch.no_grad():
            fwd.append(model.forward_comparative((gc, gw), (seq_c, seq_w), (prop_c, prop_w))[4].reshape(-1))
    _close(res.logits, torch.stack(fwd, 1), tol)
    single = predictive(model, gc, seq_c, prop_c, eps=eps_c)
    ref1 = torch.stack([R.comparative_single_forward(p, ogs[0], cpu(seq_c), cpu(prop_c), cpu(eps_c[k]),
                                                     use_wt=use_wt)[3].reshape(-1) for k in range(3)], 1)
    _close(single.logits, ref1, tol)
    _check_stats(res.logits, res.prob_mean, res.prob_std)


def test_draw_count_independence_and_statistics():
    g, _, seq, prop, model = _case(512, 71, "HybridModelv2")
    eps = _eps(257, 512, 72)
    full = predictive(model, g, seq, prop, eps=eps)
    eight = predictive(model, g, seq, prop, eps=eps[:8])
    assert torch.equal(full.logits[:, :8], eight.logits)
    one = predictive(model, g, seq, prop, eps=eps[:1])
    assert torch.equal(one.prob_std, torch.zeros_like(one.prob_std))
    _check_stats(full.logits, full.prob_mean, full.prob_std)
    assert float(full.prob_std.min()) > 0
    g1, _, seq1, prop1, _ = _case(1, 71, "HybridModelv2")
    single = predictive(model, g1, seq1, prop1, samples=4096)
    assert single.logits.shape == (1, 4096)
    _check_stats(single.logits, single.prob_mean, single.prob_std)


def _kernel_names(fn):
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    return [e.name for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA
            and "memcpy" not in e.name.lower() and "memset" not in e.name.lower()]


def test_trunk_runs_once_whatever_the_number_of_draws():
    g, _, seq, prop, model = _case(512, 81, "HybridModelv2")
    predictive(model, g, seq, prop, samples=256)                         # warm-up (module loads, cached weights)
    k1 = _kernel_names(lambda: predictive(model, g, seq, prop, samples=1))
    k256 = _kernel_names(lambda: predictive(model, g, seq, prop, samples=256))
    assert len(k1) == len(k256)
    assert sum("head_mc_infer_kernel" in n for n in k256) == 1
    with torch.no_grad():
        fwd = _kernel_names(lambda: model(g, seq, prop))
    gemm = lambda names: sum("gemm" in n.lower() for n in names)
    assert 1 <= gemm(k256) < gemm(fwd)                                   # vae_fc1 only: no vae_fc4 GEMM


@pytest.mark.parametrize("grad_mode", [torch.enable_grad, torch.no_grad])
def test_no_side_effects_on_gradients(grad_mode):
    g, _, seq, prop, model = _case(8, 91, "HybridModelv2")
    params = list(model.parameters())
    for i, q in enumerate(params[::3]):
        q.grad = torch.full_like(q, float(i + 1))
    before = [None if q.grad is None else q.grad.clone() for q in params]
    with grad_mode():
        res = predictive(model, g, seq, prop, samples=4)
    assert not res.logits.requires_grad
    for q, b in zip(params, before):
        assert (q.grad is None) == (b is None) and (b is None or torch.equal(q.grad, b))
    model.train()
    with pytest.raises(RuntimeError, match="eval"):
        predictive(model, g, seq, prop)
