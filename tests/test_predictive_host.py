"""Predictive mean and spread over the reparameterisation draw (immunostruct_b200/predictive.py), host logic on CPU:
``immunostruct_b200._C`` is patched with the per-kernel contracts (oracle/kernel_contracts.py) plus the contract of the
multi-draw head kernel defined here, and every draw is compared with the fp64 oracle's forward on that draw, on the
golden graphs.  The device kernel is checked in tests/test_predictive_gpu.py, which shares ``head_mc_infer_contract``."""
import pytest
import torch
import torch.nn.functional as F

import immunostruct_b200 as I
from immunostruct_b200 import _C, predictive as P, trunk
from immunostruct_b200.predictive import predictive, predictive_pair
from oracle import kernel_contracts as KC
from oracle import reference_ops as R

from conftest import load_golden, oracle_graph, rel_err
from helpers import build_model, graph_batch

TOL = 1e-4
K = 3


def head_mc_infer_contract(items, Wc, bc, coef, n_head, W1, b1, W2, b2):
    """Contract of is_head_mc_infer (signature of ``_C.head_mc_infer``): per draw k the tokens are, item after item,
    [x_gat | mu + eps[k] exp(0.5 logvar) | prop] (x_gat = Wc pooled + bc, or pooled), then the closed-form fusion
    attention (coef None: none) and the classifier.  -> (logits [B,K], mean and population std of sigmoid(logit))."""
    toks = []
    for pooled, mu, logvar, zv, eps in items:
        k, ld = eps.shape[0], mu.shape[1]
        x_gat = F.linear(pooled, Wc, bc) if Wc is not None else pooled
        z = mu + eps * torch.exp(0.5 * logvar)
        toks.append(torch.cat([x_gat.expand(k, -1, -1), z, zv[:, ld:].expand(k, -1, -1)], -1))
    c = torch.cat(toks, -1)
    k, b, L = c.shape
    flat = c.reshape(k * b, L)
    if coef is not None:
        flat = KC._fusion(flat, coef, n_head)
    logits = F.linear(torch.relu(F.linear(flat, W1, b1)), W2, b2).reshape(k, b).t().contiguous()
    p = torch.sigmoid(logits.double())
    return logits, p.mean(1).to(logits.dtype), p.std(1, unbiased=False).to(logits.dtype)


@pytest.fixture
def cpu_backend(monkeypatch):
    for name in KC.ALL:
        monkeypatch.setattr(_C, name, getattr(KC, name))
    monkeypatch.setattr(_C, "head_mc_infer", head_mc_infer_contract)
    monkeypatch.setattr(trunk, "_require_device_batch", lambda g: None)
    yield


def _eps(k, b, seed, ld=32):
    return torch.randn(k, b, ld, generator=torch.Generator().manual_seed(seed))


def _og64(arrays):
    g = oracle_graph(arrays)
    return dict(g, x=g["x"].double(), edge_attr=g["edge_attr"].double())


def _p64(model):
    return {k: v.detach().double() for k, v in model.state_dict().items()}


def _check_stats(res):
    p = torch.sigmoid(res.logits.double())
    assert float((res.prob_mean.double() - p.mean(1)).abs().max()) < 1e-7
    assert float((res.prob_std.double() - p.std(1, unbiased=False)).abs().max()) < 1e-7


def _comparative(use_wt, gd):
    """HybridModelv2_Comparative with the golden weights; without use_wt the classifier takes the cancer half of the
    golden first layer."""
    meta = gd["meta"]
    model = I.model_map["HybridModelv2_Comparative"](vae_input_dim=231, device="cpu", gcn_layers=int(meta["gcn_layers"]) - 1,
                                                     vae_hidden_dim=32, use_wt_for_downstream=use_wt)
    w = dict(gd["weights"])
    if not use_wt:
        w["classifier.1.weight"] = w["classifier.1.weight"][:, :104].clone()
    model.load_state_dict(w, strict=True)
    return model.eval()


@pytest.mark.parametrize("name,cls,version", [("hybrid_v2", "HybridModelv2", "v2"), ("hybrid_v1", "HybridModel", "v1")])
def test_predictive_draws_match_fp64_oracle(cpu_backend, name, cls, version):
    gd = load_golden(name)
    model = build_model(cls, gd)
    d = gd["dense"]
    eps = _eps(K, 3, 1)
    res = predictive(model, graph_batch(gd["graph"]), d["seq"], d["prop"], eps=eps)
    assert res.logits.shape == (3, K) and res.prob_mean.shape == (3,) and res.prob_std.shape == (3,)
    og, p = _og64(gd["graph"]), _p64(model)
    for k in range(K):
        ref = R.hybrid_forward(p, og, d["seq"].double(), d["prop"].double(), eps[k].double(), version=version,
                               n_layers=int(gd["meta"]["gcn_layers"]))[3].reshape(-1)
        assert rel_err(res.logits[:, k], ref) < TOL, k
    _check_stats(res)
    assert all(q.grad is None for q in model.parameters())


@pytest.mark.parametrize("use_wt", [True, False])
def test_predictive_pair_draws_match_fp64_oracle(cpu_backend, use_wt):
    gd = load_golden("comparative_v2")
    model = _comparative(use_wt, gd)
    d = gd["dense"]
    gc, gw = graph_batch(gd["graph_c"]), graph_batch(gd["graph_w"])
    eps_c, eps_w = _eps(K, 4, 2), _eps(K, 4, 3)
    res = predictive_pair(model, (gc, gw), (d["seq_c"], d["seq_w"]), (d["prop_c"], d["prop_w"]), eps=(eps_c, eps_w))
    ogs, p = (_og64(gd["graph_c"]), _og64(gd["graph_w"])), _p64(model)
    for k in range(K):
        ref = R.comparative_forward(p, ogs, (d["seq_c"].double(), d["seq_w"].double()),
                                    (d["prop_c"].double(), d["prop_w"].double()), (eps_c[k].double(), eps_w[k].double()),
                                    n_layers=int(gd["meta"]["gcn_layers"]), use_wt=use_wt)[4].reshape(-1)
        assert rel_err(res.logits[:, k], ref) < TOL, k
    _check_stats(res)


@pytest.mark.parametrize("use_wt", [True, False])
def test_predictive_comparative_single_graph_matches_fp64_oracle(cpu_backend, use_wt):
    gd = load_golden("comparative_v2")
    model = _comparative(use_wt, gd)
    d = gd["dense"]
    eps = _eps(K, 4, 4)
    res = predictive(model, graph_batch(gd["graph_c"]), d["seq_c"], d["prop_c"], eps=eps)
    og, p = _og64(gd["graph_c"]), _p64(model)
    for k in range(K):
        ref = R.comparative_single_forward(p, og, d["seq_c"].double(), d["prop_c"].double(), eps[k].double(),
                                           n_layers=int(gd["meta"]["gcn_layers"]), use_wt=use_wt)[3].reshape(-1)
        assert rel_err(res.logits[:, k], ref) < TOL, k
    _check_stats(res)


def test_default_draws_come_from_sample_eps_once_per_item_cancer_first(cpu_backend, monkeypatch):
    gd = load_golden("comparative_v2")
    model = _comparative(True, gd)
    d = gd["dense"]
    gc, gw = graph_batch(gd["graph_c"]), graph_batch(gd["graph_w"])
    calls = []

    def sample_eps(like):
        calls.append(torch.randn(like.shape, generator=torch.Generator().manual_seed(10 + len(calls))))
        return calls[-1]

    model.sample_eps = sample_eps
    layers = []
    monkeypatch.setattr(P, "_tc_linear", lambda layer, x, relu=False: layers.append(layer) or trunk._tc_linear(layer, x, relu))
    args = ((gc, gw), (d["seq_c"], d["seq_w"]), (d["prop_c"], d["prop_w"]))
    res = predictive_pair(model, *args, samples=5)
    assert [tuple(c.shape) for c in calls] == [(5 * 4, 32), (5 * 4, 32)]
    assert all(layer is model.vae_fc1 for layer in layers) and len(layers) == 2        # no vae_fc4 (decoder)
    again = predictive_pair(model, *args, eps=(calls[0].reshape(5, 4, 32), calls[1].reshape(5, 4, 32)))
    assert torch.equal(res.logits, again.logits)                                       # first call = cancer item
    calls.clear()
    single = predictive(model, gc, d["seq_c"], d["prop_c"], samples=2)
    assert [tuple(c.shape) for c in calls] == [(2 * 4, 32)] and single.logits.shape == (4, 2)
    calls.clear()
    cancer_only = _comparative(False, gd)
    cancer_only.sample_eps = sample_eps
    predictive_pair(cancer_only, *args, samples=3)
    assert [tuple(c.shape) for c in calls] == [(3 * 4, 32)]                             # the wild type does not enter


def test_predictive_errors(cpu_backend):
    gd = load_golden("hybrid_v2")
    model = build_model("HybridModelv2", gd)
    g, d = graph_batch(gd["graph"]), gd["dense"]
    args = (g, d["seq"], d["prop"])
    with pytest.raises(ValueError, match="samples"):
        predictive(model, *args, samples=0)
    for bad in (_eps(2, 4, 0), _eps(2, 3, 0, ld=31), torch.randn(3, 32)):
        with pytest.raises(ValueError, match="eps"):
            predictive(model, *args, eps=bad)
    with pytest.raises(NotImplementedError, match="HybridModel_Comparative"):
        predictive_pair(model, (g, g), (d["seq"], d["seq"]), (d["prop"], d["prop"]))
    model.train()
    with pytest.raises(RuntimeError, match="eval"):
        predictive(model, *args)
    for name in ("StructureModel", "StructureModelv2", "StructureModel_SSL", "SequenceModel", "SequenceFpModel", "DualModel"):
        other = I.model_map[name](vae_input_dim=231, device="cpu").eval()
        with pytest.raises(NotImplementedError, match="HybridModelv2_SSL"):
            predictive(other, *args)
    # (a trunk width other than 64 is refused by EGNNConv itself)
    for kw in ({"mlp_features": 16}, {"combined_attention_heads": 16}, {"vae_latent_dim": 200}):
        other = I.model_map["HybridModelv2"](vae_input_dim=231, device="cpu", **kw).eval()
        with pytest.raises(NotImplementedError):
            predictive(other, *args)
    gdc = load_golden("comparative_v2")
    pair = _comparative(True, gdc)
    dc = gdc["dense"]
    pargs = ((graph_batch(gdc["graph_c"]), graph_batch(gdc["graph_w"])), (dc["seq_c"], dc["seq_w"]), (dc["prop_c"], dc["prop_w"]))
    for bad in (_eps(2, 4, 0), (_eps(2, 4, 0), None), (_eps(2, 4, 0), _eps(3, 4, 0)), (_eps(2, 5, 0), _eps(2, 5, 0))):
        with pytest.raises(ValueError):
            predictive_pair(pair, *pargs, eps=bad)


@pytest.mark.parametrize("grad_mode", [torch.enable_grad, torch.no_grad])
def test_predictive_leaves_grads_untouched(cpu_backend, grad_mode):
    gd = load_golden("hybrid_v2")
    model = build_model("HybridModelv2", gd)
    params = list(model.parameters())
    for i, q in enumerate(params[::2]):
        q.grad = torch.full_like(q, float(i))
    before = [None if q.grad is None else q.grad.clone() for q in params]
    with grad_mode():
        res = predictive(model, graph_batch(gd["graph"]), gd["dense"]["seq"], gd["dense"]["prop"], samples=2)
    assert not res.logits.requires_grad
    for q, b in zip(params, before):
        assert (q.grad is None) == (b is None) and (b is None or torch.equal(q.grad, b))
