"""The oracle against (1) the committed golden vectors produced by the unmodified reference code, at the small
test widths and at the production width, (2) hand-derived known answers for the un-vendored DGL/PyG operators."""
import math

import pytest
import torch

from conftest import assert_grads_close, load_golden, oracle_graph, rel_err
from oracle import reference_ops as R

TOL = 1e-5


@pytest.mark.parametrize("name,version", [("hybrid_v2", "v2"), ("hybrid_v1", "v1")])
def test_hybrid_restatement_matches_golden(name, version):
    gd = load_golden(name)
    g = oracle_graph(gd["graph"])
    p = {k: v.clone().requires_grad_(True) for k, v in gd["weights"].items()}
    d = gd["dense"]
    n_layers = int(gd["meta"]["gcn_layers"])
    recon, mu, logvar, out = R.hybrid_forward(p, g, d["seq"], d["prop"], d["eps"], version=version,
                                              n_layers=n_layers)
    o = gd["out"]
    for got, key in ((recon, "recon"), (mu, "mu"), (logvar, "logvar"), (out, "logits")):
        assert rel_err(got, o[key]) < TOL, key
    emb = R.hybrid_forward(p, g, d["seq"], d["prop"], d["eps"], version=version, n_layers=n_layers,
                           return_embedding=True)[0]
    att = R.hybrid_forward(p, g, d["seq"], d["prop"], d["eps"], version=version, n_layers=n_layers,
                           return_attention=True)[0]
    assert rel_err(emb, o["embedding"]) < TOL
    assert rel_err(att, o["attention"]) < TOL
    loss = R.bce_loss(recon, d["seq"], mu, logvar, out, d["target"], float(gd["meta"]["pos_weight"]))
    assert rel_err(loss, o["loss_bce"]) < TOL
    assert rel_err(R.regression_loss(recon, d["seq"], mu, logvar, out, d["target"] * 0.5 - 0.1),
                   o["loss_reg"]) < TOL
    loss.backward()
    # last-layer coord_mlp: no gradient at all (None), everything else within tolerance
    assert_grads_close({k: v.grad for k, v in p.items()}, gd["grads"], 1e-4)


def test_comparative_restatement_matches_golden():
    gd = load_golden("comparative_v2")
    gc, gw = oracle_graph(gd["graph_c"]), oracle_graph(gd["graph_w"])
    p = {k: v.clone().requires_grad_(True) for k, v in gd["weights"].items()}
    d, o = gd["dense"], gd["out"]
    embs, recons, mus, logvars, out = R.comparative_forward(
        p, (gc, gw), (d["seq_c"], d["seq_w"]), (d["prop_c"], d["prop_w"]), (d["eps_c"], d["eps_w"]),
        n_layers=int(gd["meta"]["gcn_layers"]))
    assert rel_err(out, o["logits"]) < TOL
    assert rel_err(embs[0], o["emb_c"]) < TOL and rel_err(embs[1], o["emb_w"]) < TOL
    pw = float(gd["meta"]["pos_weight"])
    l_c = R.bce_loss(recons[0], d["seq_c"], mus[0], logvars[0], out, d["target"], pw)
    l_w = R.bce_loss(recons[1], d["seq_w"], mus[1], logvars[1], out, d["target"], pw)
    l_con = R.paired_contrastive(gd["projector"], embs[0], embs[1], d["target"])
    assert rel_err(l_con, o["loss_contrastive"]) < TOL
    loss = (l_c + l_w) / 2 + float(gd["meta"]["coeff_contrastive"]) * l_con
    assert rel_err(loss, o["loss"]) < TOL
    loss.backward()
    assert_grads_close({k: v.grad for k, v in p.items()}, gd["grads"], 1e-4)
    single = R.comparative_single_forward(p, gc, d["seq_c"], d["prop_c"], d["eps_c"],
                                          n_layers=int(gd["meta"]["gcn_layers"]))
    assert rel_err(single[3], o["single_logits"]) < TOL


def test_contrastive_returns_zero_without_two_classes():
    gd = load_golden("comparative_v2")
    e = gd["out"]["emb_c"]
    assert R.paired_contrastive(gd["projector"], e, e, torch.ones(e.shape[0])) == 0
    assert R.paired_contrastive(gd["projector"], e, e, torch.linspace(0, 1, e.shape[0])) == 0


# ---- hand-derived known answers for the restated third-party operators ---------------------
def _identity_egnn(in_size=2, hidden=2):
    """Weights chosen so every quantity can be written down by hand."""
    z = torch.zeros
    p = {
        "edge_mlp.0.weight": z(hidden, 2 * in_size + 2), "edge_mlp.0.bias": z(hidden),
        "edge_mlp.2.weight": torch.eye(hidden), "edge_mlp.2.bias": z(hidden),
        "coord_mlp.0.weight": torch.eye(hidden), "coord_mlp.0.bias": z(hidden),
        "coord_mlp.2.weight": torch.ones(1, hidden),
        "node_mlp.0.weight": z(hidden, in_size + hidden), "node_mlp.0.bias": z(hidden),
        "node_mlp.2.weight": torch.eye(hidden), "node_mlp.2.bias": z(hidden),
    }
    return p


def test_egnn_single_edge_known_answer():
    s = lambda v: v / (1 + math.exp(-v))
    p = _identity_egnn()
    # first edge-MLP row picks h_src[0], second picks radial; concat order [h_s, h_d, radial, a]
    p["edge_mlp.0.weight"][0, 0] = 1.0
    p["edge_mlp.0.weight"][1, 4] = 1.0
    p["node_mlp.0.weight"][0, 2] = 1.0      # h_neigh[0]
    p["node_mlp.0.weight"][1, 0] = 1.0      # own h[0]
    h = torch.tensor([[2.0, 0.0], [0.5, 0.0]])
    x = torch.tensor([[3.0, 0.0, 0.0], [0.0, 4.0, 0.0]])
    src, dst = torch.tensor([0]), torch.tensor([1])       # 0 -> 1
    a = torch.ones(1, 1)
    h2, x2 = R.egnn_conv(p, "", src, dst, h, x, a)
    radial = 25.0
    t = [s(2.0), s(radial)]
    m = [s(t[0]), s(t[1])]
    c = s(m[0]) + s(m[1])
    diff = [3 / 5, -4 / 5, 0.0]                            # x_src - x_dst, normalised
    assert torch.allclose(x2[1], torch.tensor([0 + c * diff[0], 4 + c * diff[1], 0.0]), atol=1e-6)
    assert torch.allclose(x2[0], x[0])                     # no in-edges: x unchanged
    assert torch.allclose(h2[1], torch.tensor([s(m[0]), s(0.5)]), atol=1e-6)
    assert torch.allclose(h2[0], torch.tensor([s(0.0), s(2.0)]), atol=1e-6)   # h_neigh = 0


def test_egnn_mean_vs_sum_and_multi_edge():
    p = _identity_egnn()
    p["edge_mlp.0.bias"][:] = 1.0
    h = torch.zeros(3, 2)
    x = torch.tensor([[1.0, 0, 0], [0.0, 0, 0], [0.0, 2.0, 0]])
    src, dst = torch.tensor([0, 2, 0]), torch.tensor([1, 1, 1])    # duplicate edge 0->1
    a = torch.zeros(3, 1)
    p["node_mlp.0.weight"][0, 2] = 1.0
    h2, x2 = R.egnn_conv(p, "", src, dst, h, x, a)
    s = lambda v: v / (1 + math.exp(-v))
    m = s(s(1.0))
    c = 2 * s(m)
    assert math.isclose(float(h2[1, 0]), s(3 * m), rel_tol=1e-6)            # features: SUM of 3
    exp_x = torch.tensor([c * (1 + 1) / 3, c * 2.0 / 2.0 / 3 * 1.0, 0.0])   # coords: MEAN of 3
    exp_x[1] = c * 1.0 / 3
    assert torch.allclose(x2[1], exp_x, atol=1e-6)


def test_pooling_known_answer():
    x = torch.tensor([[1.0, -1.0], [3.0, 5.0], [10.0, 0.0]])
    b = torch.tensor([0, 0, 1])
    assert torch.equal(R.global_mean_pool(x, b), torch.tensor([[2.0, 2.0], [10.0, 0.0]]))
    assert torch.equal(R.global_max_pool(x, b), torch.tensor([[3.0, 5.0], [10.0, 0.0]]))


def test_batch_and_csr_known_answer():
    g0 = {"src": torch.tensor([1, 2, 0]), "dst": torch.tensor([0, 0, 2]), "num_nodes": 3,
          "x": torch.zeros(3, 23), "edge_attr": torch.ones(3, 1)}
    g1 = {"src": torch.tensor([1, 0]), "dst": torch.tensor([0, 1]), "num_nodes": 2,
          "x": torch.ones(2, 23), "edge_attr": torch.ones(2, 1)}
    b = R.dgl_batch([g0, g1])
    assert b["src"].tolist() == [1, 2, 0, 4, 3] and b["dst"].tolist() == [0, 0, 2, 3, 4]
    assert R.batch_vector(b["batch_num_nodes"]).tolist() == [0, 0, 0, 1, 1]
    c = R.csr_from_coo(b["src"], b["dst"], 5)
    assert c["indptr"].tolist() == [0, 2, 2, 3, 4, 5]
    assert c["csr_src"].tolist() == [1, 2, 0, 4, 3]
    assert c["csr_eid"].tolist() == [0, 1, 2, 3, 4]
    assert c["outptr"].tolist() == [0, 1, 2, 3, 4, 5]
    assert c["csc_pos"].tolist() == [2, 0, 1, 4, 3]


def test_restatement_matches_reference_code_production_width():
    """HybridModelv2 at the production width (vae_input_dim 5943, vae_hidden_dim 512) against the outputs of the
    reference's own class stored in r2_big_hybrid_v2.npz (tests/golden/make_golden_r2.py); the weights are regenerated
    from the same name-keyed seed."""
    import immunostruct_b200 as I
    from golden_util import sample_big, seeded_state_dict
    gd = load_golden("r2_big_hybrid_v2")
    n_layers = int(gd["meta"]["gcn_layers"])
    model = I.model_map["HybridModelv2"](vae_input_dim=5943, device="cpu", gcn_layers=n_layers - 1)
    p = seeded_state_dict(model, int(gd["meta"]["seed"]))
    d, o = gd["dense"], gd["out"]
    seq = torch.nn.functional.one_hot(d["seq_tokens"].long(), 21).float()
    recon, mu, logvar, out = R.hybrid_forward(p, oracle_graph(gd["graph"]), seq, d["prop"], d["eps"], n_layers=n_layers)
    assert rel_err(out, o["logits"]) < TOL and rel_err(out, o["logits64"]) < TOL
    assert rel_err(mu, o["mu"]) < TOL and rel_err(logvar, o["logvar"]) < TOL
    r = sample_big(recon)
    assert rel_err(r[1:], o["recon_sample"][1:]) < TOL
    assert abs(float(r[0]) - float(o["recon_sample"][0])) < TOL * float(o["recon_sample"][0])
    loss = R.bce_loss(recon, seq, mu, logvar, out, d["target"], float(gd["meta"]["pos_weight"]))
    assert rel_err(loss, o["loss"]) < TOL and rel_err(loss, o["loss64"]) < TOL


def test_pooled_only_attention_backward_closed_form():
    """The algebra csrc/attn_pool_bwd_tc.cu implements (its header comment), checked in fp64 against autograd of the
    oracle's attention + mean pool: with g0 = g_pooled / n every row of gO equals g0, so c_j = V_j . g0,
    D_i = sum_j P_ij c_j, G_ij = P_ij (c_j - D_i), gQ = G K / 8, gK = G^T Q / 8, gV_j = (sum_i P_ij) g0."""
    from oracle import kernel_contracts as KC
    gen = torch.Generator().manual_seed(3)
    for n in (1, 7, 130):
        qkv = torch.randn(n, 192, generator=gen, dtype=torch.float64).requires_grad_(True)
        gp = torch.randn(64, generator=gen, dtype=torch.float64)
        o, _, _ = KC._attn_graph(qkv, 1)
        (ref,) = torch.autograd.grad(o.mean(0), qkv, gp)
        Q, K, V = (qkv.detach()[:, 64 * i:64 * i + 64] for i in range(3))
        P = torch.softmax(Q @ K.T / 8.0, dim=1)
        g0 = gp / n
        c = V @ g0
        G = P * (c[None, :] - (P @ c)[:, None])
        closed = torch.cat([G @ K / 8.0, G.T @ Q / 8.0, P.sum(0)[:, None] * g0[None, :]], dim=1)
        assert rel_err(closed, ref) < 1e-12
        assert float(G.sum(1).abs().max()) < 1e-14          # shift invariance: every row of G sums to zero
