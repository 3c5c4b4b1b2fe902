"""Input gradients through the EGNN stack and integrated-gradients attribution (immunostruct_b200/attribution.py), host
logic on CPU: ``immunostruct_b200._C`` is patched with the per-kernel contracts (oracle/kernel_contracts.py) and the
product is compared with the full-model oracle's autograd on the hybrid_v2 golden graph.  The device kernels are checked
in tests/test_attribution_gpu.py.  ``oracle_ig``, ``oracle_input_grads`` and the contract of the edge-feature
gradient kernel are shared with that file."""
import pytest
import torch

import immunostruct_b200 as I
from immunostruct_b200 import _C, trunk
from immunostruct_b200.attribution import integrated_gradients
from oracle import kernel_contracts as KC
from oracle import reference_ops as R

from conftest import load_golden, oracle_graph, rel_err
from helpers import build_model, graph_batch, inject_eps

TOL = 1e-4


def egnn_edge_attr_grad_contract(gz1, g, W1, f, g_attr, accumulate):
    """Contract of is_egnn_edge_attr_grad (signature of ``_C.egnn_edge_attr_grad``): g_attr[csr_eid[p]] (+)= gz1[p] .
    W1[:, 2f+1] -- a_e enters the first edge-MLP layer as a_e W1[:, 2f+1]."""
    v = torch.zeros(gz1.shape[0], dtype=gz1.dtype).index_copy_(0, g.csr_eid.long(), gz1 @ W1[:, 2 * f + 1])
    flat = g_attr.view(-1)
    if accumulate:
        flat += v
    else:
        flat.copy_(v)


@pytest.fixture
def cpu_backend(monkeypatch):
    for name in KC.ALL:
        monkeypatch.setattr(_C, name, getattr(KC, name))
    monkeypatch.setattr(_C, "egnn_edge_attr_grad", egnn_edge_attr_grad_contract)
    monkeypatch.setattr(trunk, "_require_device_batch", lambda g: None)
    yield


def _leaf(t, dtype):
    return t.detach().to(dtype).clone().requires_grad_(True)


def oracle_input_grads(weights, g, seq, prop, eps, dtype, forward=R.hybrid_forward, objective=None, **kw):
    """Gradients of sum(logit) (or of ``objective(outputs)``) with respect to x23 and edge_attr, by autograd through the
    oracle in ``dtype``."""
    p = {k: v.detach().to(dtype) for k, v in weights.items()}
    x, ea = _leaf(g["x"], dtype), _leaf(g["edge_attr"], dtype)
    outs = forward(p, dict(g, x=x, edge_attr=ea), seq.to(dtype), prop.to(dtype), eps.to(dtype), **kw)
    obj = outs[3].sum() if objective is None else objective(outs, dtype)
    return torch.autograd.grad(obj, [x, ea])


def oracle_ig(weights, g, seq, prop, eps, steps, dtype, forward=R.hybrid_forward, **kw):
    """Integrated gradients of the oracle's logit on the midpoint grid, all-zero baseline, coordinates held at the input:
    -> (residue [N, 20], edge [E], sequence, property, logit [B], baseline logit [B], completeness gap [B])."""
    p = {k: v.detach().to(dtype) for k, v in weights.items()}
    x, ea, s, pr, ep = (t.detach().to(dtype) for t in (g["x"], g["edge_attr"], seq, prop, eps))

    def f(a, grad):
        xa = x.clone()
        xa[:, :20] *= a
        leaves = [t.requires_grad_(grad) for t in (xa, ea * a, s * a, pr * a)]
        out = forward(p, dict(g, x=leaves[0], edge_attr=leaves[1]), leaves[2], leaves[3], ep, **kw)[3].reshape(-1)
        if not grad:
            return out.detach(), None
        return out.detach(), torch.autograd.grad(out.sum(), leaves, allow_unused=True)

    tot = None
    for k in range(steps):
        _, gr = f((k + 0.5) / steps, True)
        gr = [torch.zeros_like(t) if gg is None else gg for gg, t in zip(gr, (x, ea, s, pr))]
        tot = gr if tot is None else [a + b for a, b in zip(tot, gr)]
    res = x[:, :20] * tot[0][:, :20] / steps
    edge = (ea * tot[1] / steps).reshape(-1)
    sq, pp = s * tot[2] / steps, pr * tot[3] / steps
    logit, base = f(1.0, False)[0], f(0.0, False)[0]
    bvec = R.batch_vector(g["batch_num_nodes"])
    ebvec = R.batch_vector(g["batch_num_edges"])
    b = logit.numel()
    per = (torch.zeros(b, dtype=dtype).index_add_(0, bvec, res.sum(1)) + torch.zeros(b, dtype=dtype).index_add_(0, ebvec, edge)
           + sq.reshape(b, -1).sum(1) + pp.reshape(b, -1).sum(1))
    return res, edge, sq, pp, logit, base, logit - base - per


def test_input_gradients_match_oracle_autograd(cpu_backend):
    gd = load_golden("hybrid_v2")
    model = build_model("HybridModelv2", gd)
    g = graph_batch(gd["graph"])
    d = gd["dense"]
    x, ea = g.ndata["x"].detach().clone().requires_grad_(True), g.edata["edge_attr"].detach().clone().requires_grad_(True)
    g.ndata["x"], g.edata["edge_attr"] = x, ea
    inject_eps(model, d["eps"])
    model(g, d["seq"], d["prop"])[3].sum().backward()
    og = oracle_graph(gd["graph"])
    gx64, ge64 = oracle_input_grads(gd["weights"], og, d["seq"], d["prop"], d["eps"], torch.float64, n_layers=6)
    assert x.grad is not None and ea.grad is not None and ea.grad.shape == ea.shape
    assert rel_err(x.grad, gx64) < TOL and rel_err(ea.grad, ge64) < TOL
    assert float(gx64[:, 20:].abs().max()) > 0 and float(gx64[:, :20].abs().max()) > 0


def test_standalone_egnnconv_input_gradients(cpu_backend):
    gd = load_golden("hybrid_v2")
    g = graph_batch(gd["graph"])
    torch.manual_seed(0)
    conv = I.EGNNConv(20, 64, 64, 1)
    h = g.ndata["x"][:, :20].detach().clone().requires_grad_(True)
    xc = g.ndata["x"][:, 20:].detach().clone().requires_grad_(True)
    ea = g.edata["edge_attr"].detach().clone().requires_grad_(True)
    ho, xo = conv(g, h, xc, ea)
    (ho.pow(2).sum() + xo.pow(2).sum()).backward()
    p = {"c." + k: v.detach().double() for k, v in conv.state_dict().items()}
    og = oracle_graph(gd["graph"])
    leaves = [_leaf(t, torch.float64) for t in (h, xc, ea)]
    ho64, xo64 = R.egnn_conv(p, "c.", og["src"], og["dst"], *leaves)
    ref = torch.autograd.grad(ho64.pow(2).sum() + xo64.pow(2).sum(), leaves)
    for got, r in zip((h.grad, xc.grad, ea.grad), ref):
        assert got is not None and rel_err(got, r) < TOL


def test_integrated_gradients_match_oracle(cpu_backend):
    gd = load_golden("hybrid_v2")
    model = build_model("HybridModelv2", gd)
    g = graph_batch(gd["graph"])
    d = gd["dense"]
    res = integrated_gradients(model, g, d["seq"], d["prop"], steps=4, eps=d["eps"], max_graphs=6)
    ref = oracle_ig(gd["weights"], oracle_graph(gd["graph"]), d["seq"], d["prop"], d["eps"], 4, torch.float64, n_layers=6)
    got = (res.residue_features, res.edge_attr, res.sequence, res.peptide_property, res.logit, res.baseline_logit)
    for a, r in zip(got, ref[:6]):
        assert a.shape == r.shape and rel_err(a, r) < TOL
    assert float((res.completeness_gap - ref[6]).abs().max()) < TOL * float(res.logit.abs().max())
    assert all(p.grad is None for p in model.parameters())
    assert "sample_eps" not in model.__dict__


def test_integrated_gradients_refuse_training_mode(cpu_backend):
    gd = load_golden("hybrid_v2")
    model = build_model("HybridModelv2", gd).train()
    with pytest.raises(RuntimeError, match="eval"):
        integrated_gradients(model, graph_batch(gd["graph"]), gd["dense"]["seq"], gd["dense"]["prop"])
