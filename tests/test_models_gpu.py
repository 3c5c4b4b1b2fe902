"""End-to-end parity of the product models on the GPU: golden vectors produced by the unmodified
reference code, the full-model CPU oracle at the benchmark's graph shape, and size-independent
properties (determinism, edge-order invariance, padding semantics) at full batch sizes.
Tolerances: 1e-5 relative on logits / loss (north star, fp32), gradients 1e-5 of the parameter's
scale with a floor (conftest.assert_grads_close)."""
import pytest
import torch

import immunostruct_b200 as I
from immunostruct_b200.synthetic import synthetic_dense, synthetic_graph_arrays, split_graphs
from oracle import reference_ops as R

from conftest import assert_grads_close, load_golden, rel_err
from helpers import build_model, graph_batch, inject_eps, named_grads

pytestmark = pytest.mark.gpu
DEV = "cuda"
TOL = 1e-5


def _d(t):
    return t.to(DEV)


@pytest.mark.parametrize("name,cls", [("hybrid_v2", "HybridModelv2"), ("hybrid_v1", "HybridModel")])
def test_hybrid_golden(name, cls):
    gd = load_golden(name)
    model = build_model(cls, gd, device=DEV)
    g = graph_batch(gd["graph"], DEV).validate()
    d, o = gd["dense"], gd["out"]
    inject_eps(model, d["eps"], d["eps"], d["eps"])
    recon, mu, logvar, out = model(g, _d(d["seq"]), _d(d["prop"]))
    for got, key in ((recon, "recon"), (mu, "mu"), (logvar, "logvar"), (out, "logits")):
        assert rel_err(got, o[key]) < TOL, key
    # closer to the fp64 run of the reference than 1e-5 as well
    assert rel_err(out, o["logits64"]) < TOL
    losses = I.Losses(231, [float(gd["meta"]["pos_weight"]), 1.0], sequence=True)
    loss = losses.BCE_loss(recon, _d(d["seq"]), mu, logvar, out, _d(d["target"]))
    assert rel_err(loss, o["loss_bce"]) < TOL
    assert rel_err(losses.regression_loss(recon, _d(d["seq"]), mu, logvar, out, _d(d["target"] * 0.5 - 0.1)),
                   o["loss_reg"]) < TOL
    loss.backward()
    assert_grads_close(named_grads(model), gd["grads"], TOL, truth=gd["grads64"])
    inject_eps(model, d["eps"], d["eps"], d["eps"])
    with torch.no_grad():                         # inference path: fused stack + pooled-only attention
        r_ng = model(g, _d(d["seq"]), _d(d["prop"]))
    assert rel_err(r_ng[3], o["logits"]) < TOL and rel_err(r_ng[0], o["recon"]) < TOL
    emb = model(g, _d(d["seq"]), _d(d["prop"]), return_embedding=True)[0]
    att = model(g, _d(d["seq"]), _d(d["prop"]), return_attention=True)[0]
    assert rel_err(emb, o["embedding"]) < TOL
    assert att.shape == o["attention"].shape and rel_err(att, o["attention"]) < TOL


def test_comparative_golden():
    gd = load_golden("comparative_v2")
    model = build_model("HybridModelv2_Comparative", gd, device=DEV)
    gc, gw = graph_batch(gd["graph_c"], DEV), graph_batch(gd["graph_w"], DEV)
    d, o = gd["dense"], gd["out"]
    inject_eps(model, d["eps_c"], d["eps_w"], d["eps_c"])
    embs, recons, mus, logvars, out = model.forward_comparative(
        (gc, gw), (_d(d["seq_c"]), _d(d["seq_w"])), (_d(d["prop_c"]), _d(d["prop_w"])))
    assert rel_err(out, o["logits"]) < TOL
    assert rel_err(embs[0], o["emb_c"]) < TOL and rel_err(embs[1], o["emb_w"]) < TOL
    losses = I.Losses(231, [float(gd["meta"]["pos_weight"]), 1.0], sequence=True)
    pcl = I.PairedContrastiveLoss(embedding_dim=104, device=DEV)
    pcl.load_state_dict(gd["projector"])
    y = _d(d["target"])
    l_c = losses.BCE_loss(recons[0], _d(d["seq_c"]), mus[0], logvars[0], out, y)
    l_w = losses.BCE_loss(recons[1], _d(d["seq_w"]), mus[1], logvars[1], out, y)
    l_con = pcl(embs[0], embs[1], y)
    assert rel_err(l_con, o["loss_contrastive"]) < 5e-5      # B x B and 128 x 128 sums of squares
    loss = (l_c + l_w) / 2 + float(gd["meta"]["coeff_contrastive"]) * l_con
    assert rel_err(loss, o["loss"]) < TOL
    loss.backward()
    assert_grads_close(named_grads(model), gd["grads"], TOL, truth=gd["grads64"])
    assert rel_err(model(gc, _d(d["seq_c"]), _d(d["prop_c"]))[3], o["single_logits"]) < TOL


def test_structure_v2_golden():
    gd = load_golden("structure_v2")
    model = I.model_map["StructureModelv2"](vae_input_dim=231, device=DEV, gcn_layers=1)
    model.load_state_dict(gd["weights"])
    model.to(DEV).eval()
    g = graph_batch(gd["graph"], DEV)
    _, _, _, out, node_pred = model(g, _d(gd["dense"]["seq"]), _d(gd["dense"]["prop"]))
    assert rel_err(out, gd["out"]["logits"]) < TOL and rel_err(node_pred, gd["out"]["node_pred"]) < TOL
    (out.sum() + node_pred.pow(2).sum()).backward()
    assert_grads_close(named_grads(model), gd["grads"], TOL)


def _bench_shape_case(b, seed, n_pad=0, scale=1.0, device=DEV):
    """HybridModelv2 at the BASELINE shape with default initialisation (at 200 nodes / in-degree 10 the
    logits already differ between graphs in the 2nd digit; scaling the EGNN weights up saturates the
    per-graph softmax and, from about 2x, overflows fp32 through the six un-normalised
    sum-aggregations in reference and product alike)."""
    arr = synthetic_graph_arrays(b, 200, 10, seed=seed, n_pad=n_pad)
    dense = synthetic_dense(b, seed=seed)
    torch.manual_seed(seed)
    model = I.model_map["HybridModelv2"](vae_input_dim=5943, device=device)
    with torch.no_grad():
        for k, p in model.named_parameters():
            if k.startswith("GCN_layers") and k.endswith("weight"):
                p.mul_(scale)
    eps = torch.randn(b, 32, generator=torch.Generator().manual_seed(seed + 3))
    return arr, dense, model, eps


def _oracle_run(state, arr, dense, eps, dtype):
    p = {k: v.detach().clone().to(dtype).requires_grad_(True) for k, v in state.items()}
    g = R.dgl_batch(split_graphs(arr))
    g = dict(g, x=g["x"].to(dtype), edge_attr=g["edge_attr"].to(dtype))
    recon, mu, logvar, out = R.hybrid_forward(p, g, dense["seq"].to(dtype), dense["prop"].to(dtype), eps.to(dtype))
    loss = R.bce_loss(recon, dense["seq"].to(dtype), mu, logvar, out, dense["target"].to(dtype), 4.25)
    loss.backward()
    return recon, out, loss, {k: v.grad for k, v in p.items()}


def test_benchmark_shape_against_full_model_oracle():
    """N = 200, k = 10, vae_input_dim 5943 (BASELINE config shape), padded variant: logits, loss and
    every parameter gradient against the CPU oracle (fp32 = the reference's arithmetic, fp64 = truth)."""
    b = 6
    arr, dense, model, eps = _bench_shape_case(b, seed=5, n_pad=10)
    state = {k: v.cpu() for k, v in model.state_dict().items()}
    recon, out, loss_ref, grads32 = _oracle_run(state, arr, dense, eps, torch.float32)
    _, out64, _, grads64 = _oracle_run(state, arr, dense, eps, torch.float64)
    assert float(out.std()) > 1e-4 * float(out.abs().mean())          # outputs do depend on the graph
    model = model.to(DEV).eval()
    inject_eps(model, eps)
    gb = graph_batch(arr, DEV).validate()
    r2, m2, lv2, o2 = model(gb, _d(dense["seq"]), _d(dense["prop"]))
    losses = I.Losses(5943, [4.25, 1.0], sequence=True)
    loss = losses.BCE_loss(r2, _d(dense["seq"]), m2, lv2, o2, _d(dense["target"]))
    assert rel_err(o2, out) < TOL and rel_err(r2, recon) < TOL and rel_err(loss, loss_ref) < TOL
    assert rel_err(o2, out64) < TOL
    loss.backward()
    assert_grads_close(named_grads(model), grads32, TOL, truth=grads64)


def test_bf16_mode_within_1e_2_of_fp32_reference():
    """bf16 tensor-core mode (north star: 1e-2 relative): logits and loss at the benchmark shape against
    the fp32 CPU oracle, inference path and training-forward path; gradients against the ORACLE's fp32 gradients
    (the backward always recomputes in fp32, so only the forward activations carry bf16 rounding)."""
    b = 8
    arr, dense, model, eps = _bench_shape_case(b, seed=21)
    state = {k: v.cpu() for k, v in model.state_dict().items()}
    recon, out, loss_ref, grads_oracle = _oracle_run(state, arr, dense, eps, torch.float32)
    model = model.to(DEV).eval()
    gb = graph_batch(arr, DEV)
    losses = I.Losses(5943, [4.25, 1.0], sequence=True)
    grads = {}
    default_precision = I.get_precision()
    try:
        for prec in ("bf16x3", "tf32x3", "fp32", "fp16x2", "bf16"):
            I.set_precision(prec)
            inject_eps(model, eps, eps)
            with torch.no_grad():
                o_inf = model(gb, _d(dense["seq"]), _d(dense["prop"]))[3]
            model.zero_grad()
            r2, m2, lv2, o2 = model(gb, _d(dense["seq"]), _d(dense["prop"]))
            loss = losses.BCE_loss(r2, _d(dense["seq"]), m2, lv2, o2, _d(dense["target"]))
            loss.backward()
            grads[prec] = {k: v.clone() for k, v in named_grads(model).items() if v is not None}
            tol = 1e-2 if prec == "bf16" else TOL
            assert rel_err(o_inf, out) < tol and rel_err(o2, out) < tol and rel_err(loss, loss_ref) < tol, prec
    finally:
        I.set_precision(default_precision)
    ref_grads = {k: v for k, v in grads_oracle.items() if v is not None}
    gmax = max(float(v.abs().max()) for v in ref_grads.values())
    worst = ("", 0.0)
    for k, ref in ref_grads.items():
        err = float((grads["bf16"][k].cpu() - ref).abs().max())
        ratio = err / max(float(ref.abs().max()), 1e-2 * gmax)
        worst = max(worst, (k, ratio), key=lambda t: t[1])
    import os
    os.makedirs("gpurun_out", exist_ok=True)
    with open("gpurun_out/kernel_errors.txt", "a") as f:
        f.write(f"test_bf16_mode | worst bf16 gradient vs oracle: {worst[0]} rel {worst[1]:.3e}\n")
    assert worst[1] <= 1e-2, worst


def test_precision_modes_agree_at_the_full_batch():
    """Batch 512 (the benchmark batch), no-grad forward: the default fp16x2 arithmetic, bf16x3, tf32x3 and the fp32 SIMT
    kernels are four independent roundings of the same computation -- logits, reconstruction and latent statistics of all
    512 graphs must agree within the fp32 tolerance (the oracle comparison above runs at batch 8)."""
    b = 512
    arr, dense, model, eps = _bench_shape_case(b, seed=13)
    model = model.to(DEV).eval()
    seq, prop = _d(dense["seq"]), _d(dense["prop"])
    gb = graph_batch(arr, DEV)
    default_precision = I.get_precision()
    outs = {}
    try:
        with torch.no_grad():
            for prec in ("fp32", "fp16x2", "bf16x3", "tf32x3"):
                I.set_precision(prec)
                inject_eps(model, eps)
                outs[prec] = [t.clone() for t in model(gb, seq, prop)]
    finally:
        I.set_precision(default_precision)
    for prec in ("fp16x2", "bf16x3", "tf32x3"):
        for a, ref, what in zip(outs[prec], outs["fp32"], ("recon", "mu", "logvar", "logits")):
            assert bool(torch.isfinite(a).all())
            assert rel_err(a, ref) < TOL, (prec, what, rel_err(a, ref))


def test_full_batch_properties():
    """Batch 512 (BASELINE inference batch): bit-determinism, edge-order invariance within tolerance,
    per-graph independence (a graph's output does not depend on its batch neighbours)."""
    b = 512
    arr, dense, model, eps = _bench_shape_case(b, seed=9)
    model = model.to(DEV).eval()
    seq, prop = _d(dense["seq"]), _d(dense["prop"])
    with torch.no_grad():
        outs = []
        for _ in range(2):
            inject_eps(model, eps)
            outs.append(model(graph_batch(arr, DEV), seq, prop))
        for a, c in zip(outs[0], outs[1]):
            assert torch.equal(a, c)
        # shuffle the edge order inside every graph: sums are re-associated, nothing else changes
        e = int(arr["edge_counts"][0])
        perm = torch.stack([torch.randperm(e) + i * e for i in range(b)]).reshape(-1)
        arr2 = dict(arr, src=arr["src"][perm], dst=arr["dst"][perm], edge_attr=arr["edge_attr"][perm])
        inject_eps(model, eps)
        shuffled = model(graph_batch(arr2, DEV), seq, prop)
        assert rel_err(shuffled[3], outs[0][3]) < TOL
        # the first 8 graphs alone give the same logits as inside the batch of 512
        sub = synthetic_graph_arrays(b, 200, 10, seed=9)
        n8, e8 = 8 * 200, 8 * e
        arr8 = {"x": sub["x"][:n8], "src": sub["src"][:e8], "dst": sub["dst"][:e8], "edge_attr": sub["edge_attr"][:e8],
                "node_counts": sub["node_counts"][:8], "edge_counts": sub["edge_counts"][:8]}
        inject_eps(model, eps[:8])
        small = model(graph_batch(arr8, DEV), seq[:8], prop[:8])
        assert rel_err(small[3], outs[0][3][:8]) < TOL
    assert torch.isfinite(outs[0][3]).all()


def test_last_layer_coord_mlp_has_no_grad_and_training_step_runs():
    """Reference behaviour (SURVEY 8(a) row 4): layer-5 coord_mlp parameters keep grad None, so
    Adam/AdamW skip them.  Also runs two optimiser steps in train mode (dropout + randn_like live)."""
    b = 16
    arr, dense, model, _ = _bench_shape_case(b, seed=13)
    model = model.to(DEV).train()
    opt = torch.optim.Adam(model.parameters(), lr=1e-3)
    losses = I.Losses(5943, [4.25, 1.0], sequence=True)
    gb = graph_batch(arr, DEV)
    vals = []
    for _ in range(2):
        opt.zero_grad()
        recon, mu, logvar, out = model(gb, _d(dense["seq"]), _d(dense["prop"]))
        loss = losses.BCE_loss(recon, _d(dense["seq"]), mu, logvar, out, _d(dense["target"]))
        loss.backward()
        opt.step()
        vals.append(float(loss))
    last = len(model.GCN_layers) - 1
    for k, p in model.named_parameters():
        if k.startswith(f"GCN_layers.{last}.coord_mlp"):
            assert p.grad is None, k
        else:
            assert p.grad is not None and torch.isfinite(p.grad).all(), k
    assert all(v == v for v in vals)


def test_contrastive_gate_on_device():
    pcl = I.PairedContrastiveLoss(embedding_dim=104, device=DEV)
    e1, e2 = torch.randn(8, 104, device=DEV), torch.randn(8, 104, device=DEV)
    assert float(pcl(e1, e2, torch.ones(8, device=DEV))) == 0.0
    assert float(pcl(e1, e2, torch.tensor([0., 1, 0, 1, 1, 0, 0, 1], device=DEV))) > 0.0


def test_device_prefetcher_matches_direct_path():
    """Overlapped H2D + collation (DevicePrefetcher) yields the same batches / logits as `.to(device)`."""
    from immunostruct_b200.graph import GraphBatch
    arr, dense, model, eps = _bench_shape_case(12, seed=17)
    model = model.to(DEV).eval()
    keys = ("x", "src", "dst", "edge_attr", "node_counts", "edge_counts")

    def host_batches():
        for lo in (0, 4, 8):
            n0, e0 = lo * 200, lo * 2000
            sub = {"x": arr["x"][n0:n0 + 800], "src": arr["src"][e0:e0 + 8000], "dst": arr["dst"][e0:e0 + 8000],
                   "edge_attr": arr["edge_attr"][e0:e0 + 8000], "node_counts": arr["node_counts"][lo:lo + 4],
                   "edge_counts": arr["edge_counts"][lo:lo + 4]}
            yield (GraphBatch.from_arrays(*(sub[k] for k in keys), max_nodes=200), dense["seq"][lo:lo + 4],
                   dense["target"][lo:lo + 4], dense["prop"][lo:lo + 4])

    direct, fetched = [], []
    with torch.no_grad():
        for i, (g, seq, y, prop) in enumerate(host_batches()):
            inject_eps(model, eps[4 * i:4 * i + 4])
            direct.append(model(g.to(DEV), seq.to(DEV), prop.to(DEV))[3])
        for i, (g, seq, y, prop) in enumerate(I.DevicePrefetcher(host_batches(), DEV)):
            assert g.device.type == "cuda" and seq.is_cuda and y.is_cuda and g.to(DEV) is g
            inject_eps(model, eps[4 * i:4 * i + 4])
            fetched.append(model(g, seq, prop)[3])
    assert len(fetched) == 3
    for a, b in zip(direct, fetched):
        assert torch.equal(a, b)


@pytest.mark.gpu
def test_packed_batches_expand_bit_exactly_and_prefetch():
    """Compact input format: device expansion == the dense batch (bit-exact arrays, CSR and logits), through
    `.to(device)` and through the DevicePrefetcher; non-unit edge_attr travels explicitly."""
    from immunostruct_b200.graph import GraphBatch
    arr, dense, model, eps = _bench_shape_case(8, seed=23, n_pad=10)
    model = model.to(DEV).eval()
    keys = ("x", "src", "dst", "edge_attr", "node_counts", "edge_counts")
    host = GraphBatch.from_arrays(*(arr[k] for k in keys), max_nodes=200)
    pk, ps = I.pack_graph_batch(host), I.pack_sequence(dense["seq"])
    assert pk.nbytes * 3 < sum(arr[k].numel() * arr[k].element_size() for k in keys)
    g_dense, g_packed = host.to(DEV), pk.to(DEV)
    for f in ("indptr", "csr_src", "csr_dst", "csr_eid", "outptr", "csc_pos", "node_off", "edge_off"):
        assert torch.equal(getattr(g_dense, f), getattr(g_packed, f)), f
    assert torch.equal(g_dense.ndata["x"], g_packed.ndata["x"]) and torch.equal(g_dense.edata["edge_attr"], g_packed.edata["edge_attr"])
    seq_d = ps.to(DEV)
    assert torch.equal(seq_d, dense["seq"].to(DEV))
    with torch.no_grad():
        inject_eps(model, eps)
        ref = model(g_dense, dense["seq"].to(DEV), dense["prop"].to(DEV))[3]
        inject_eps(model, eps)
        got = model(g_packed, seq_d, dense["prop"].to(DEV))[3]
        assert torch.equal(ref, got)
        for g, seq, prop in I.DevicePrefetcher([(pk.pin_memory(), ps.pin_memory(), dense["prop"])], DEV):
            assert isinstance(g, GraphBatch) and g.device.type == "cuda" and seq.shape == (8, 283, 21)
            inject_eps(model, eps)
            assert torch.equal(model(g, seq, prop)[3], ref)
    arr2 = dict(arr, edge_attr=torch.rand_like(arr["edge_attr"]) + 0.5)
    pk2 = I.pack_graph_batch(GraphBatch.from_arrays(*(arr2[k] for k in keys), max_nodes=200))
    assert pk2.edge_attr is not None and torch.equal(pk2.to(DEV).edata["edge_attr"], arr2["edge_attr"].to(DEV))
