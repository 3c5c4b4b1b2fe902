"""Single-residue mutational scan (immunostruct_b200/mutagenesis.py), host logic on CPU: the contract of the expansion
kernel (is_mutscan_expand) against explicit per-copy edits, the copy enumeration and the pass split, every error raised
before a kernel call, and whole scans through the per-kernel contracts against the fp64 oracle's forward on each mutant.
The device kernel is checked in tests/test_mutscan_gpu.py, which shares ``mutscan_expand_contract``."""
import pytest
import torch
import torch.nn.functional as F

import immunostruct_b200 as I
from immunostruct_b200 import _C, trunk
from immunostruct_b200.mutagenesis import mutational_scan, mutational_scan_pair, scan_sites
from immunostruct_b200.resident import scan_passes
from oracle import kernel_contracts as KC
from oracle import reference_ops as R

from conftest import load_golden, oracle_graph, rel_err
from helpers import build_model, graph_batch
from test_predictive_host import _comparative, head_mc_infer_contract

TOL = 1e-4


def mutscan_expand_contract(x23, node_off, node_index, seq, seq_index, seq_columns, sites, x23_out, seq_out, flag):
    """Contract of is_mutscan_expand (signature of ``_C.mutscan_expand``): copy k of the base batch gets sites[k] = (p, c)
    at node row node_off[b] + node_index[b, p] (residue columns one_hot_20(c)) and sequence row seq_index[b, p]
    (one_hot_V(seq_columns[c])) of every sample b with node_index[b, p] >= 0.  flag |= 1 when a patched site's base rows
    are not exactly one-hot or disagree with seq_columns, or when an index is out of range (that graph stays unpatched)."""
    b, _ = node_index.shape
    n, (L, V), r = x23.shape[0], seq.shape[1:], sites.shape[0]
    ps, cs = sites[:, 0].long(), sites[:, 1].long()
    ni, si, sc = node_index[:, ps].t(), seq_index[:, ps].t(), seq_columns.long()[cs]          # [r, b], [r, b], [r]
    counts = (node_off[1:] - node_off[:-1]).unsqueeze(0)
    present = ni >= 0
    ok = present & (ni < counts) & (si >= 0) & (si < L) & ((sc >= 0) & (sc < V)).unsqueeze(1)
    rows = (node_off[:-1].unsqueeze(0) + ni.clamp_min(0)).clamp_max(max(n - 1, 0))
    xr = x23[rows, :20]
    sr = seq[torch.arange(b).unsqueeze(0).expand(r, b), si.clamp(0, L - 1)]
    one_hot = lambda t: ((t == 1).sum(-1) == 1) & ((t != 0).sum(-1) == 1)
    good = one_hot(xr) & one_hot(sr) & (seq_columns.long()[xr.argmax(-1)] == sr.argmax(-1))
    xo, so = x23.repeat(r, 1).reshape(r, n, 23), seq.repeat(r, 1, 1).reshape(r, b, L, V)
    kk, bb = ok.nonzero(as_tuple=True)
    xo[kk, rows[kk, bb], :20] = F.one_hot(cs[kk], 20).to(xo.dtype)
    so[kk, bb, si[kk, bb]] = F.one_hot(sc[kk], V).to(so.dtype)
    x23_out.copy_(xo.reshape(r * n, 23))
    seq_out.copy_(so.reshape(r * b, L, V))
    if bool((present & ~ok).any() | (ok & ~good).any()):
        flag.fill_(1)


def _explicit(x23, node_off, node_index, seq, seq_index, seq_columns, sites):
    """The same pass written as one edit per (copy, sample): (x23_out, seq_out, flag)."""
    r, (b, L, V) = sites.shape[0], seq.shape
    xs, ss, flag = [], [], 0
    for p, c in sites.tolist():
        x, s = x23.clone(), seq.clone()
        for i in range(b):
            ni, si = int(node_index[i, p]), int(seq_index[i, p])
            if ni < 0:
                continue
            n0, nb, sc = int(node_off[i]), int(node_off[i + 1] - node_off[i]), int(seq_columns[c])
            if ni >= nb or not 0 <= si < L or not 0 <= sc < V:
                flag = 1
                continue
            row, srow = x23[n0 + ni, :20], seq[i, si]
            if (sorted(row.tolist()) != [0.0] * 19 + [1.0] or sorted(srow.tolist()) != [0.0] * (V - 1) + [1.0]
                    or int(seq_columns[int(row.argmax())]) != int(srow.argmax())):
                flag = 1
            x[n0 + ni, :20] = 0.0
            x[n0 + ni, c] = 1.0
            s[i, si] = 0.0
            s[i, si, sc] = 1.0
        xs.append(x)
        ss.append(s)
    return torch.cat(xs), torch.cat(ss), flag


def _ragged_case(seed=0, V=21, L=9):
    """Four graphs of 12, 5, 30 and 1 nodes; graphs 0 and 2 end in two all-zero padded rows.  Sites: 3 per sample, the
    last absent for samples 1 and 3; the sequence rows at the sites follow the permuted ``seq_columns``."""
    gen = torch.Generator().manual_seed(seed)
    counts = [12, 5, 30, 1]
    n = sum(counts)
    aa = torch.randint(0, 20, (n,), generator=gen)
    x = torch.cat([F.one_hot(aa, 20).float(), torch.randn(n, 3, generator=gen)], 1)
    off = torch.tensor([0] + counts).cumsum(0)
    for i in (0, 2):
        x[off[i + 1] - 2:off[i + 1], :20] = 0.0
    cols = torch.randperm(V, generator=gen)[:20]
    tok = torch.randint(0, V, (4, L), generator=gen)
    node_index = torch.tensor([[0, 4, 9], [1, 4, -1], [27, 3, 11], [0, 0, -1]])
    seq_index = torch.tensor([[1, 2, 8], [0, 5, -1], [3, 1, 7], [4, 6, -1]])
    for i in range(4):
        for p in range(3):
            if node_index[i, p] >= 0:
                tok[i, seq_index[i, p]] = cols[aa[off[i] + node_index[i, p]]]
    seq = F.one_hot(tok, V).float()
    return x, off, node_index, seq, seq_index, cols


def _run_contract(x, off, ni, seq, si, cols, sites):
    r, n, (b, L, V) = sites.shape[0], x.shape[0], seq.shape
    xo, so = torch.full((r * n, 23), float("nan")), torch.full((r * b, L, V), float("nan"))
    flag = torch.zeros(1, dtype=torch.int32)
    mutscan_expand_contract(x, off, ni, seq, si, cols, sites, xo, so, flag)
    return xo, so, int(flag)


@pytest.mark.parametrize("which", ["all", "first", "one", "tail"])
def test_contract_equals_explicit_edits(which):
    x, off, ni, seq, si, cols = _ragged_case()
    sites = scan_sites(3)
    sites = {"all": sites, "first": sites[:20], "one": sites[37:38], "tail": sites[41:]}[which]
    xo, so, flag = _run_contract(x, off, ni, seq, si, cols, sites)
    ex, es, eflag = _explicit(x, off, ni, seq, si, cols, sites)
    assert torch.equal(xo, ex) and torch.equal(so, es) and flag == eflag == 0
    r = sites.shape[0]
    assert torch.equal(xo.reshape(r, -1, 23)[:, :, 20:], x[:, 20:].expand(r, -1, -1))           # coordinates untouched


def test_contract_flags_bad_rows_and_maps():
    x, off, ni, seq, si, cols = _ragged_case(1)
    sites = scan_sites(3)
    for edit in ("padded", "map", "seq_row", "range"):
        ni2, cols2, seq2 = ni.clone(), cols.clone(), seq.clone()
        if edit == "padded":
            ni2[0, 1] = 10                                       # an all-zero padded row of graph 0
        elif edit == "map":
            cols2 = cols.roll(1)
        elif edit == "seq_row":
            seq2[2, si[2, 0]] = 0.5
        else:
            ni2[1, 0] = 5                                        # graph 1 has 5 nodes
        xo, so, flag = _run_contract(x, off, ni2, seq2, si, cols2, sites)
        ex, es, eflag = _explicit(x, off, ni2, seq2, si, cols2, sites)
        assert flag == eflag == 1, edit
        assert torch.equal(xo, ex) and torch.equal(so, es), edit


@pytest.mark.parametrize("max_graphs", [4, 5, 11, 12, 60, 4096])
def test_copy_enumeration_and_pass_split(max_graphs):
    b, n_sites = 4, 3
    sites = scan_sites(n_sites)
    assert sites.dtype == torch.int32 and sites.shape == (n_sites * 20, 2)
    assert sites.tolist() == [[p, c] for p in range(n_sites) for c in range(20)]
    passes = scan_passes(n_sites * 20, b, max_graphs)
    per = max_graphs // b
    assert all(r == per for _, r in passes[:-1]) and 1 <= passes[-1][1] <= per
    assert [j for j, _ in passes] == list(range(0, 60, per)) and sum(r for _, r in passes) == 60
    assert len({r for _, r in passes}) <= 2
    with pytest.raises(ValueError, match="max_graphs"):
        scan_passes(60, b, b - 1)


# ---- whole scans through the kernel contracts -----------------------------------------------------------------------
@pytest.fixture
def cpu_backend(monkeypatch):
    for name in KC.ALL:
        monkeypatch.setattr(_C, name, getattr(KC, name))
    monkeypatch.setattr(_C, "head_mc_infer", head_mc_infer_contract)
    monkeypatch.setattr(_C, "mutscan_expand", mutscan_expand_contract)
    monkeypatch.setattr(trunk, "_require_device_batch", lambda g: None)
    yield


def _sites_for(graph_arrays, seq, n_sites=2):
    """Sites on real residues (the first rows of each graph), the second absent for sample 1; the sequence rows at the
    sites are rewritten to the residue's column under the reversed alphabet map."""
    cols = torch.arange(20).flip(0)
    counts = graph_arrays["node_counts"]
    off = torch.cat([torch.zeros(1, dtype=torch.int64), counts.cumsum(0)])
    b = counts.numel()
    ni = torch.tensor([[0, 3]] * b)
    si = torch.tensor([[2, 6]] * b)
    ni[1, 1] = si[1, 1] = -1
    seq = seq.clone()
    for i in range(b):
        for p in range(n_sites):
            if ni[i, p] >= 0:
                c = int(graph_arrays["x"][off[i] + ni[i, p], :20].argmax())
                seq[i, si[i, p]] = F.one_hot(cols[c], seq.shape[2]).float()
    return ni, si, cols, seq, off


def _mutant(arrays, seq, off, ni, si, cols, p, c):
    x, s = arrays["x"].clone(), seq.clone()
    for i in range(ni.shape[0]):
        if ni[i, p] >= 0:
            x[off[i] + ni[i, p], :20] = F.one_hot(torch.tensor(c), 20).float()
            s[i, si[i, p]] = F.one_hot(cols[c], s.shape[2]).float()
    return dict(arrays, x=x), s


def _og64(arrays):
    g = oracle_graph(arrays)
    return dict(g, x=g["x"].double(), edge_attr=g["edge_attr"].double())


@pytest.mark.parametrize("max_graphs", [3, 9, 4096])
def test_scan_matches_fp64_oracle_per_mutant(cpu_backend, max_graphs):
    gd = load_golden("hybrid_v2")
    model = build_model("HybridModelv2", gd)
    d = gd["dense"]
    ni, si, cols, seq, off = _sites_for(gd["graph"], d["seq"])
    eps = torch.randn(2, 3, 32, generator=torch.Generator().manual_seed(3))
    res = mutational_scan(model, graph_batch(gd["graph"]), seq, d["prop"], ni, si, seq_columns=cols, eps=eps,
                          max_graphs=max_graphs)
    assert res.logits.shape == (3, 2, 20, 2) and res.prob_mean.shape == res.prob_std.shape == (3, 2, 20)
    assert torch.isnan(res.logits[1, 1]).all() and torch.isnan(res.prob_mean[1, 1]).all()
    assert not torch.isnan(res.logits[0]).any() and res.native[1, 1] == -1
    p64 = {k: v.detach().double() for k, v in model.state_dict().items()}
    for p, c in ((0, 0), (0, 7), (1, 19), (1, int(res.native[0, 1]))):
        arr, s = _mutant(gd["graph"], seq, off, ni, si, cols, p, c)
        for k in range(2):
            ref = R.hybrid_forward(p64, _og64(arr), s.double(), d["prop"].double(), eps[k].double(), version="v2",
                                   n_layers=int(gd["meta"]["gcn_layers"]))[3].reshape(-1)
            got = res.logits[:, p, c, k]
            keep = ni[:, p] >= 0
            assert rel_err(got[keep], ref[keep]) < TOL, (p, c, k)
    for i in range(3):
        for p in range(2):
            if ni[i, p] >= 0:
                assert int(res.native[i, p]) == int(gd["graph"]["x"][off[i] + ni[i, p], :20].argmax())
                assert torch.allclose(res.logits[i, p, int(res.native[i, p])], res.base.logits[i], rtol=0, atol=1e-6)
    pr = torch.sigmoid(res.logits.double())
    keep = ~torch.isnan(pr[..., 0])
    assert float((res.prob_mean.double()[keep] - pr.mean(-1)[keep]).abs().max()) < 1e-7
    assert float((res.prob_std.double()[keep] - pr.std(-1, unbiased=False)[keep]).abs().max()) < 1e-7
    assert all(q.grad is None for q in model.parameters())


@pytest.mark.parametrize("use_wt", [True, False])
def test_pair_scan_matches_fp64_oracle_and_draws_once_per_item(cpu_backend, use_wt):
    gd = load_golden("comparative_v2")
    model = _comparative(use_wt, gd)
    d = gd["dense"]
    ni, si, cols, seq_c, off = _sites_for(gd["graph_c"], d["seq_c"])
    calls = []

    def sample_eps(like):
        calls.append(torch.randn(like.shape, generator=torch.Generator().manual_seed(20 + len(calls))))
        return calls[-1]

    model.sample_eps = sample_eps
    gc, gw = graph_batch(gd["graph_c"]), graph_batch(gd["graph_w"])
    res = mutational_scan_pair(model, (gc, gw), (seq_c, d["seq_w"]), (d["prop_c"], d["prop_w"]), ni, si, seq_columns=cols,
                               samples=2, max_graphs=8)
    assert [tuple(c.shape) for c in calls] == [(2 * 4, 32)] * (2 if use_wt else 1)
    eps_c = calls[0].reshape(2, 4, 32)
    eps_w = calls[1].reshape(2, 4, 32) if use_wt else torch.zeros(2, 4, 32)
    p64 = {k: v.detach().double() for k, v in model.state_dict().items()}
    for p, c in ((0, 5), (1, 0)):
        arr, s = _mutant(gd["graph_c"], seq_c, off, ni, si, cols, p, c)
        for k in range(2):
            ref = R.comparative_forward(p64, (_og64(arr), _og64(gd["graph_w"])), (s.double(), d["seq_w"].double()),
                                        (d["prop_c"].double(), d["prop_w"].double()), (eps_c[k].double(), eps_w[k].double()),
                                        n_layers=int(gd["meta"]["gcn_layers"]), use_wt=use_wt)[4].reshape(-1)
            keep = ni[:, p] >= 0
            assert rel_err(res.logits[:, p, c, k][keep], ref[keep]) < TOL, (p, c, k)


def _hybrid_args(gd):
    d = gd["dense"]
    ni, si, cols, seq, _ = _sites_for(gd["graph"], d["seq"])
    return graph_batch(gd["graph"]), seq, d["prop"], ni, si, cols


def test_errors_before_any_kernel_call(cpu_backend, monkeypatch):
    gd = load_golden("hybrid_v2")
    model = build_model("HybridModelv2", gd)
    g, seq, prop, ni, si, cols = _hybrid_args(gd)
    launched = []
    monkeypatch.setattr(_C, "mutscan_expand", lambda *a: launched.append(1))

    def bad(exc, match, m=model, **kw):
        args = dict(node_index=ni, seq_index=si, seq_columns=cols)
        args.update(kw)
        with pytest.raises(exc, match=match):
            mutational_scan(m, g, seq, prop, args.pop("node_index"), args.pop("seq_index"), **args)

    bad(ValueError, "int64", node_index=ni.int())
    bad(ValueError, "int64", seq_index=si[:2])
    bad(ValueError, "same shape", seq_index=si[:, :1])
    one_sided = si.clone()
    one_sided[0, 0] = -1
    bad(ValueError, "absent", seq_index=one_sided)
    below = ni.clone()
    below[0, 0] = below[0, 0] * 0 - 2
    bad(ValueError, ">= -1", node_index=below, seq_index=torch.where(below < 0, below, si))
    past = ni.clone()
    past[2, 0] = 12                                                     # graph 2 has 12 nodes
    bad(ValueError, "node count", node_index=past)
    bad(ValueError, "sequence length", seq_index=torch.where(si >= 0, si + 5, si))
    bad(ValueError, "seq_columns", seq_columns=cols[:19])
    bad(ValueError, "seq_columns", seq_columns=torch.zeros(20, dtype=torch.int64))
    bad(ValueError, "seq_columns", seq_columns=cols + 2)                # 21 and 22 are past V = 21
    bad(ValueError, "seq_columns", seq_columns=cols.float())
    bad(ValueError, "max_graphs", max_graphs=2)
    bad(ValueError, "samples", samples=0)
    for name in ("StructureModel", "StructureModelv2", "SequenceModel", "DualModel"):
        bad(NotImplementedError, "HybridModelv2_SSL", m=I.model_map[name](vae_input_dim=231, device="cpu").eval())
    with pytest.raises(NotImplementedError, match="HybridModel_Comparative"):
        mutational_scan_pair(model, (g, g), (seq, seq), (prop, prop), ni, si, seq_columns=cols)
    model.train()
    bad(RuntimeError, "eval")
    assert not launched


def test_flag_raises_after_the_passes(cpu_backend):
    gd = load_golden("hybrid_v2")
    model = build_model("HybridModelv2", gd)
    g, seq, prop, ni, si, cols = _hybrid_args(gd)
    padded = ni.clone()
    padded[0, 1] = 11                                                    # rows 10 and 11 of each graph are padding
    with pytest.raises(ValueError, match="one-hot"):
        mutational_scan(model, g, seq, prop, padded, si, seq_columns=cols)
    with pytest.raises(ValueError, match="seq_columns"):
        mutational_scan(model, g, seq, prop, ni, si, seq_columns=cols.roll(3))
