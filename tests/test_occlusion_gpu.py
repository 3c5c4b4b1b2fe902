"""Structural occlusion on the B200: the expansion kernel (is_occlusion_expand) against its contract bit for bit, every
entry against the fused eval forward of the host-built occluded batch and against the fp64 oracle, independence of the
pass size, ``base`` against ``predictive``, the launches of each pass, the pair form, gradients and argument rules.

An entry is held to 1e-6 relative against the same graph run in another batch: where a graph sits in a batch changes two
summation orders of the eval path (tests/test_mutscan_gpu.py, DESIGN 4.4c)."""
import pytest
import torch

import immunostruct_b200 as I
from immunostruct_b200 import _C
from immunostruct_b200.occlusion import (_contact_tables, _residue_tables, occlude_contacts, occlude_contacts_pair,
                                         occlude_residues, occlude_residues_pair)
from immunostruct_b200.predictive import predictive, predictive_pair
from immunostruct_b200.resident import variant_passes
from immunostruct_b200.synthetic import synthetic_dense
from oracle import reference_ops as R

from helpers import concat_graphs, graph_batch, inject_eps, log_error
from test_occlusion_host import _explicit, _offsets, hand_case, occlusion_expand_contract
from test_variants_gpu import _arrays, _case, _mutants, _og64

pytestmark = pytest.mark.gpu
DEV = "cuda"
TOL = 1e-5
BATCH_TOL = 1e-6          # the same graph in another batch: summation order only (module docstring)


@pytest.fixture
def precision(request):
    prev = I.get_precision()
    I.set_precision(request.param)
    yield request.param
    I.set_precision(prev)


def _close(got, ref, tol=TOL, what="occlusion"):
    ref = ref.detach().double().cpu()
    err = float((got.detach().double().cpu() - ref).abs().max())
    lim = tol * max(float(ref.abs().max()), 1e-30)
    log_error(f"{what}: err {err:.3e} err/bound {err / lim:.3f} (tol {tol:.0e})")
    assert err <= lim, (err, float(ref.abs().max()))


def _eps(k, b, seed):
    return torch.randn(k, b, 32, generator=torch.Generator().manual_seed(seed)).to(DEV)


def _rows(arr, rows):
    """bool [ΣN]: graph-local rows ``rows`` of every graph that has them."""
    off = _offsets(arr["node_counts"].cpu())
    sel = torch.zeros(int(off[-1]), dtype=torch.bool)
    for s, n in enumerate(arr["node_counts"].tolist()):
        sel[off[s] + torch.tensor([r for r in rows if r < n], dtype=torch.int64)] = True
    return sel


def _bits(t):
    """Bit pattern of an output (the NaN prefill of a block the kernel did not write compares equal to itself)."""
    return t.view(torch.int32) if t.dtype == torch.float32 else t


def _variants(tables):
    return [tuple(t) for t in torch.stack(tables[:3], 1).tolist()]


def _occluded(c, variants):
    """The host-built occluded batch: (device batch, sequences, properties, sample index on the device)."""
    arr = _explicit(c["arr"], variants)
    samples = torch.tensor([v[0] for v in variants], device=DEV)
    return graph_batch(arr, DEV), c["seq"][samples], c["prop"][samples], samples, arr


# ---- the kernel against its contract -----------------------------------------------------------------------------------
@pytest.mark.parametrize("mode", ["residues", "contacts"])
def test_expand_kernel_against_contract(mode):
    arr = concat_graphs(_arrays(48, 5, big=True), hand_case(4))     # ragged, a 256-node graph, multi-edges, self-loops
    assert int(arr["node_counts"][0]) == 256
    g = graph_batch(arr, DEV)
    nodes = None if mode == "residues" else _rows(arr, range(0, 256, 9))
    tables = (_residue_tables if mode == "residues" else _contact_tables)(g, nodes, 4096)[0]
    smp, na, nb, nv, kept, ncs, ecs, passes, node_tot, edge_tot, c = tables
    assert len(passes) >= 2 and 2 * 4096 > 10 * 4 * _C.num_sms()        # every CTA loops over many (variant, part) units
    off, eoff = _offsets(arr["node_counts"]), _offsets(arr["edge_counts"])
    for (j, r), n_p, e_p in zip(passes, node_tot, edge_tot):
        outs = []
        for dev in (DEV, "cpu"):
            t = lambda x: x.to(dev)
            xo, eo = torch.full((n_p, 23), float("nan"), device=dev), torch.full((e_p, 1), float("nan"), device=dev)
            so, do = (torch.full((e_p,), -7, dtype=torch.int64, device=dev) for _ in range(2))
            flag = torch.zeros(1, dtype=torch.int32, device=dev)
            fn = _C.occlusion_expand if dev == DEV else occlusion_expand_contract
            fn(t(arr["x"]), t(off), t(eoff), t(arr["src"]), t(arr["dst"]), t(arr["edge_attr"]), t(smp[j:j + r]),
               t(na[j:j + r]), t(nb[j:j + r]), t(ncs[j:j + r + 1] - ncs[j]), t(ecs[j:j + r + 1] - ecs[j]), xo, so, do, eo,
               flag)
            outs.append([x.cpu() for x in (xo, so, do, eo, flag)])
        for a, b_ in zip(*outs):
            assert torch.equal(_bits(a), _bits(b_))
        assert int(outs[0][4]) == 0


def test_expand_kernel_flags():
    arr = hand_case(5)
    g = graph_batch(arr, DEV)
    lib = [(0, 1, -1), (2, 3, 9), (4, 0, -1), (1, 3, -1), (2, 5, 5), (1, 0, -2), (0, 2, 3)]
    t = torch.tensor(lib).T.contiguous()
    ref = _explicit(arr, [v if i not in (2, 3, 4, 5) else (0, 0, -1) for i, v in enumerate(lib)])
    no, eo = _offsets(ref["node_counts"]), _offsets(ref["edge_counts"])
    eo_bad = eo + torch.tensor([0, 0, 0, 0, 0, 0, 0, 1])              # the last variant's kept count disagrees
    for edge_out in (eo, eo_bad):
        outs = []
        for dev in (DEV, "cpu"):
            xo = torch.full((int(no[-1]), 23), float("nan"), device=dev)
            so, do = (torch.full((int(edge_out[-1]),), -7, dtype=torch.int64, device=dev) for _ in range(2))
            ea = torch.full((int(edge_out[-1]), 1), float("nan"), device=dev)
            flag = torch.zeros(1, dtype=torch.int32, device=dev)
            fn = _C.occlusion_expand if dev == DEV else occlusion_expand_contract
            fn(*(x.to(dev) for x in (arr["x"], g.node_off, g.edge_off, arr["src"], arr["dst"], arr["edge_attr"], t[0], t[1],
                                     t[2], no, edge_out)), xo, so, do, ea, flag)
            outs.append([x.cpu() for x in (xo, so, do, ea, flag)])
        assert int(outs[0][4]) == int(outs[1][4]) == 1
        assert all(torch.equal(_bits(a), _bits(b_)) for a, b_ in zip(*outs))


# ---- entries against the fused eval forward and the fp64 oracle ---------------------------------------------------------
def _fused_forward(c, variants, eps_k):
    """Logits of the fused eval forward of the host-built occluded graphs on draw ``eps_k`` [B, latent], run B graphs at
    a time (the last run padded with repeats of its last variant).  With ``max_graphs`` = B these are the occlusion
    passes' batches: every graph sits at the same batch position and the VAE encoder sees the same row count (B) as in
    the call, so the two summation orders of DESIGN 4.4c agree; test_pass_size_independence_and_base covers other
    positions."""
    b, out = c["b"], []
    for lo in range(0, len(variants), b):
        chunk = variants[lo:lo + b]
        g, seq, prop, samples, _ = _occluded(c, chunk + chunk[-1:] * (b - len(chunk)))
        inject_eps(c["model"], eps_k[samples])
        with torch.no_grad():
            out.append(c["model"](g, seq, prop)[3].reshape(-1)[:len(chunk)])
    del c["model"].sample_eps
    return torch.cat(out)


@pytest.mark.parametrize("precision", ["fp16x2", "bf16x3"], indirect=True)
@pytest.mark.parametrize("name", ["HybridModel", "HybridModelv2"])
@pytest.mark.parametrize("mode", ["residues", "contacts"])
def test_entries_match_the_fused_forward(precision, name, mode):
    c = _case(12, 12, name)
    eps = _eps(3, 12, 14)
    if mode == "residues":
        nodes = _rows(c["arr"], range(14))
        res = occlude_residues(c["model"], c["g"], c["seq"], c["prop"], nodes=nodes, eps=eps, max_graphs=c["b"])
        rows = nodes.nonzero().flatten().to(DEV)
        off = _offsets(c["arr"]["node_counts"])
        smp = torch.searchsorted(off, rows.cpu(), right=True) - 1
        variants = [(int(s), int(r - off[s]), -1) for s, r in zip(smp, rows.cpu())]
        logits, mean = res.logits[rows], res.prob_mean[rows]
        assert torch.isnan(res.logits[~nodes.to(DEV)]).all()
    else:
        res = occlude_contacts(c["model"], c["g"], c["seq"], c["prop"], nodes=_rows(c["arr"], range(5)), eps=eps,
                               max_graphs=c["b"])
        variants = list(zip(res.sample.tolist(), res.u.tolist(), res.v.tolist()))
        logits, mean = res.logits, res.prob_mean
    assert len(variants) > 64
    for k in (0, 2):
        _close(logits[:, k], _fused_forward(c, variants, eps[k]), BATCH_TOL)
    pr = torch.sigmoid(logits.double())
    assert float((mean.double() - pr.mean(-1)).abs().max()) <= 1e-7


@pytest.mark.parametrize("precision", ["fp16x2", "bf16x3"], indirect=True)
def test_entries_match_fp64_oracle(precision):
    c = _case(3, 31, ragged=False)
    eps = _eps(2, 3, 33)
    nodes = _rows(c["arr"], (0, 7, 195))                                   # 195: a padded row, scored as selected
    res = occlude_residues(c["model"], c["g"], c["seq"], c["prop"], nodes=nodes, eps=eps, max_graphs=4)
    con = occlude_contacts(c["model"], c["g"], c["seq"], c["prop"], nodes=_rows(c["arr"], (3,)), eps=eps, max_graphs=5)
    rows = nodes.nonzero().flatten()
    variants = [(int(r) // 200, int(r) % 200, -1) for r in rows]
    variants_c = list(zip(con.sample.tolist(), con.u.tolist(), con.v.tolist()))
    p64 = {k: v.detach().double().cpu() for k, v in c["model"].state_dict().items()}
    for lg, var in ((res.logits[rows.to(DEV)], variants), (con.logits, variants_c)):
        _, seq, _, samples, arr = _occluded(c, var)
        for k in range(2):
            ref = R.hybrid_forward(p64, _og64(arr), seq.double().cpu(), c["prop"][samples].double().cpu(),
                                   eps[k][samples].double().cpu(), version="v2")[3].reshape(-1)
            _close(lg[:, k].cpu(), ref)


# ---- pass size, base, absent rows -------------------------------------------------------------------------------------
def test_pass_size_independence_and_base():
    b = 24
    c = _case(b, 41)
    eps = _eps(2, b, 43)
    runs = [occlude_residues(c["model"], c["g"], c["seq"], c["prop"], eps=eps, max_graphs=m) for m in (4096, 37)]
    assert len(variant_passes(int(torch.isfinite(runs[0].prob_mean).sum()), 37)) > 10
    present = torch.isfinite(runs[0].prob_mean)
    assert torch.equal(present, torch.isfinite(runs[1].prob_mean))
    _close(runs[1].logits[present], runs[0].logits[present], BATCH_TOL)
    stat_lim = BATCH_TOL * float(runs[0].logits[present].abs().max()) / 4   # sigmoid' <= 1/4
    for f in ("prob_mean", "prob_std"):
        assert float((getattr(runs[1], f)[present] - getattr(runs[0], f)[present]).abs().max()) <= stat_lim, f
    cons = [occlude_contacts(c["model"], c["g"], c["seq"], c["prop"], nodes=_rows(c["arr"], range(9)), eps=eps,
                             max_graphs=m) for m in (4096, 37)]
    assert torch.equal(cons[0].edge_contact, cons[1].edge_contact)
    _close(cons[1].logits, cons[0].logits, BATCH_TOL)
    ref = predictive(c["model"], c["g"], c["seq"], c["prop"], eps=eps)
    for run in runs + cons:
        for f in ("logits", "prob_mean", "prob_std"):
            assert torch.equal(getattr(run.base, f), getattr(ref, f)), f
    # the default skips the absent rows (graphs of 200 and 60 nodes end in padded rows); selected, one equals base
    off = _offsets(c["arr"]["node_counts"])
    absent = int(off[1]) - 1
    assert not bool(present[absent])
    nodes = torch.zeros(int(off[-1]), dtype=torch.bool)
    nodes[absent] = True
    one = occlude_residues(c["model"], c["g"], c["seq"], c["prop"], nodes=nodes, eps=eps)
    _close(one.logits[absent], ref.logits[0], BATCH_TOL)


# ---- launches, gradients, argument rules -------------------------------------------------------------------------------
def _names(fn, monkeypatch):
    names = []
    call = _C._call
    monkeypatch.setattr(_C, "_call", lambda name, *a: names.append(name) or call(name, *a))
    out = fn()
    monkeypatch.setattr(_C, "_call", call)
    return names, out


@pytest.mark.parametrize("mode", ["residues", "contacts"])
def test_launches_per_pass_and_gradients(mode, monkeypatch):
    b, max_graphs = 16, 300
    c = _case(b, 51)
    model = c["model"]
    params = list(model.parameters())
    for i, q in enumerate(params[::3]):
        q.grad = torch.full_like(q, float(i + 1))
    before = [None if q.grad is None else q.grad.clone() for q in params]
    eps = _eps(4, b, 53)
    fn = occlude_residues if mode == "residues" else occlude_contacts
    run = lambda: fn(model, c["g"], c["seq"], c["prop"], eps=eps, max_graphs=max_graphs,
                     nodes=None if mode == "residues" else _rows(c["arr"], range(9)))
    res = run()                                                                        # warm-up
    base, _ = _names(lambda: predictive(model, c["g"], c["seq"], c["prop"], eps=eps), monkeypatch)
    g = c["g"]
    tables = (_residue_tables if mode == "residues" else _contact_tables)(g, None if mode == "residues" else
                                                                          _rows(c["arr"], range(9)), max_graphs)[0]
    expected = list(base)
    for j, r in tables[7]:
        g_r, _, _, _, _ = _occluded(c, _variants(tables)[j:j + r])
        with torch.no_grad():
            trunk, _ = _names(lambda: model.structure_embedding(g_r, project=False), monkeypatch)
        expected += ["is_occlusion_expand", "is_collate_csr"] + trunk + ["is_head_mc_infer"]
    assert len(tables[7]) >= 2
    names, res = _names(run, monkeypatch)
    assert names == expected
    assert names.count("is_vae_mid_infer") == 1                                        # the encoder ran once
    for q, b_ in zip(params, before):
        assert (q.grad is None) == (b_ is None) and (b_ is None or torch.equal(q.grad, b_))
    assert not res.logits.requires_grad
    model.train()
    with pytest.raises(RuntimeError, match="eval"):
        run()
    model.eval()
    with pytest.raises(NotImplementedError, match="HybridModelv2_SSL"):
        fn(I.model_map["StructureModelv2"](vae_input_dim=5943, device=DEV).to(DEV).eval(), c["g"], c["seq"], c["prop"])


@pytest.mark.parametrize("mode", ["residues", "contacts"])
@pytest.mark.parametrize("use_wt", [True, False])
def test_pair_against_forward_comparative(use_wt, mode):
    b = 10
    c = _case(b, 61, "HybridModelv2_Comparative", use_wt_for_downstream=use_wt)
    aw = _arrays(b, 62)
    dw = synthetic_dense(b, seed=62)
    gw, seq_w, prop_w = graph_batch(aw, DEV), dw["seq"].to(DEV), dw["prop"].to(DEV)
    args = ((c["g"], gw), (c["seq"], seq_w), (c["prop"], prop_w))
    calls = []
    c["model"].sample_eps = lambda like: calls.append(like.shape[0]) or torch.randn(
        like.shape, generator=torch.Generator().manual_seed(70 + len(calls))).to(like.device)
    nodes = _rows(c["arr"], range(6))
    if mode == "residues":
        res = occlude_residues_pair(c["model"], *args, nodes=nodes, samples=2, max_graphs=25)
        rows = nodes.nonzero().flatten()
        off = _offsets(c["arr"]["node_counts"])
        smp = torch.searchsorted(off, rows, right=True) - 1
        variants = [(int(s), int(r - off[s]), -1) for s, r in zip(smp, rows)]
        logits = res.logits[rows.to(DEV)]
    else:
        res = occlude_contacts_pair(c["model"], *args, nodes=nodes, samples=2, max_graphs=25)
        variants = list(zip(res.sample.tolist(), res.u.tolist(), res.v.tolist()))
        logits = res.logits
    assert calls == [2 * b] * (2 if use_wt else 1)                        # no wild-type draw without use_wt
    draws = [torch.randn(2 * b, 32, generator=torch.Generator().manual_seed(70 + i)).reshape(2, b, 32).to(DEV)
             for i in range(1, 3)]
    g, seq, prop, samples, _ = _occluded(c, variants)
    _, gw_v, seq_wv, _ = _mutants(c, [(v[0], []) for v in variants], arr=aw, seq=dw["seq"])   # the fixed wild type
    for k in range(2):
        inject_eps(c["model"], draws[0][k][samples], draws[1][k][samples] if use_wt else torch.zeros(len(variants), 32))
        with torch.no_grad():
            ref = c["model"].forward_comparative((g, gw_v), (seq, seq_wv), (prop, prop_w[samples]))[4].reshape(-1)
        _close(logits[:, k], ref, BATCH_TOL)
    del c["model"].sample_eps
    ref_base = predictive_pair(c["model"], *args, eps=(draws[0], draws[1] if use_wt else None))
    assert torch.equal(res.base.logits, ref_base.logits)
