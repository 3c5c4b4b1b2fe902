"""Variant libraries (immunostruct_b200/mutagenesis.py: score_variants), host logic on CPU: the contract of the gather-and-
substitute kernel (is_variant_expand) against explicit per-variant edits, every flag case, every error raised before a
kernel call, the pass split, and whole runs through the per-kernel contracts against the fp64 oracle's forward on each
host-built mutant.  The device kernel is checked in tests/test_variants_gpu.py, which shares ``variant_expand_contract``."""
import pytest
import torch
import torch.nn.functional as F

import immunostruct_b200 as I
from immunostruct_b200 import _C, trunk
from immunostruct_b200.mutagenesis import score_variants, score_variants_pair
from immunostruct_b200.resident import variant_passes
from oracle import kernel_contracts as KC
from oracle import reference_ops as R

from conftest import load_golden, oracle_graph, rel_err
from helpers import build_model, graph_batch
from test_predictive_host import _comparative, head_mc_infer_contract

TOL = 1e-4


def _one_hot_rows(t):
    return ((t == 1).sum(-1) == 1) & ((t != 0).sum(-1) == 1)


def variant_expand_contract(x23, node_off, edge_off, src_local, dst_local, edge_attr, seq, sample, offsets, node_index,
                            seq_index, residue, seq_columns, node_out, edge_out, x23_out, src_out, dst_out, edge_attr_out,
                            seq_out, flag):
    """Contract of is_variant_expand (signature of ``_C.variant_expand``): variant v is base graph b = sample[v] copied to
    node rows node_out[v]..., edges edge_out[v]... (graph-local endpoints) and sequence v, then each substitution s of
    offsets[v] .. offsets[v+1]-1 writes one_hot_20(residue[s]) into the residue columns of node row node_index[s] (>= 0)
    and one_hot_V(seq_columns[residue[s]]) into sequence row seq_index[s].  flag |= 1 for a base row that is not exactly
    one-hot (the x23 row when node_index >= 0, the sequence row always), a sequence column that is not seq_columns[the
    x23 row's column], an index out of range (that substitution is skipped), a sample outside [0, B) or output offsets
    that disagree with the base counts (that variant is not written), or offsets outside [0, S] (copied, nothing
    substituted).  Rows substituted twice within one variant are left to the kernel (the host rejects them)."""
    b, L, V = seq.shape
    r, n_sub = sample.numel(), node_index.numel()
    nc, ec = node_off.diff(), edge_off.diff()
    sb = sample.clamp(0, b - 1)
    ok = ((sample >= 0) & (sample < b) & (node_out[:-1] >= 0) & (node_out.diff() == nc[sb]) &
          (node_out[1:] <= x23_out.shape[0]) & (edge_out[:-1] >= 0) & (edge_out.diff() == ec[sb]) &
          (edge_out[1:] <= src_out.shape[0]))
    v = ok.nonzero().flatten()

    def rows(base_off, out_off, counts):           # (source, destination) rows of every written variant's block
        n = counts[sb[v]]
        within = torch.arange(int(n.sum())) - torch.repeat_interleave(n.cumsum(0) - n, n)
        return (torch.repeat_interleave(base_off[sb[v]], n) + within, torch.repeat_interleave(out_off[v], n) + within)

    s_, d_ = rows(node_off, node_out, nc)
    x23_out[d_] = x23[s_]
    s_, d_ = rows(edge_off, edge_out, ec)
    src_out[d_], dst_out[d_] = src_local[s_], dst_local[s_]
    edge_attr_out.reshape(-1)[d_] = edge_attr.reshape(-1)[s_]
    seq_out[v] = seq[sb[v]]
    subs_ok = ok & (offsets[:-1] >= 0) & (offsets.diff() >= 0) & (offsets[1:] <= n_sub)
    bad = bool((~ok).any() | (ok & ~subs_ok).any())
    v = subs_ok.nonzero().flatten()
    cnt = offsets.diff()[v]
    owner = torch.repeat_interleave(v, cnt)
    s = torch.repeat_interleave(offsets[:-1][v], cnt) + torch.arange(int(cnt.sum())) - torch.repeat_interleave(cnt.cumsum(0) - cnt, cnt)
    ni, si, c, bs = node_index[s], seq_index[s], residue[s], sb[owner]
    in_range = (ni >= -1) & (ni < nc[bs]) & (si >= 0) & (si < L) & (c >= 0) & (c < 20)
    sc = seq_columns[c.clamp(0, 19)]
    in_range &= (sc >= 0) & (sc < V)
    xr = x23[(node_off[bs] + ni.clamp_min(0)).clamp(0, max(x23.shape[0] - 1, 0)), :20]
    sr = seq[bs, si.clamp(0, L - 1)]
    x_ok = (ni < 0) | (_one_hot_rows(xr) & (seq_columns[xr.argmax(-1)] == sr.argmax(-1)))
    good = in_range & _one_hot_rows(sr) & x_ok
    bad |= bool((~good).any())
    node = good & (ni >= 0)
    x23_out[node_out[owner[node]] + ni[node], :20] = F.one_hot(c[node], 20).to(x23_out.dtype)
    seq_out[owner[good], si[good]] = F.one_hot(sc[good], V).to(seq_out.dtype)
    if bad:
        flag.fill_(1)


def _explicit(arr, seq, cols, library):
    """The same pass written as one edit per variant: (x23, src, dst, edge_attr, seq, flag) of the concatenated variants.
    ``library``: a list of (sample, [(node_index, seq_index, residue), ...])."""
    off = torch.cat([torch.zeros(1, dtype=torch.int64), arr["node_counts"].cumsum(0)])
    eoff = torch.cat([torch.zeros(1, dtype=torch.int64), arr["edge_counts"].cumsum(0)])
    L, V = seq.shape[1:]
    xs, srcs, dsts, eas, ss, flag = [], [], [], [], [], 0
    for b, subs in library:
        x, s = arr["x"][off[b]:off[b + 1]].clone(), seq[b].clone()
        for ni, si, c in subs:
            nb = x.shape[0]
            if not (-1 <= ni < nb and 0 <= si < L and 0 <= c < 20 and 0 <= int(cols[c]) < V):
                flag = 1
                continue
            srow = seq[b, si]
            if sorted(srow.tolist()) != [0.0] * (V - 1) + [1.0]:
                flag = 1
                continue
            if ni >= 0:
                row = arr["x"][off[b] + ni, :20]
                if sorted(row.tolist()) != [0.0] * 19 + [1.0] or int(cols[int(row.argmax())]) != int(srow.argmax()):
                    flag = 1
                    continue
                x[ni, :20] = 0.0
                x[ni, c] = 1.0
            s[si] = 0.0
            s[si, int(cols[c])] = 1.0
        xs.append(x)
        srcs.append(arr["src"][eoff[b]:eoff[b + 1]])
        dsts.append(arr["dst"][eoff[b]:eoff[b + 1]])
        eas.append(arr["edge_attr"][eoff[b]:eoff[b + 1]])
        ss.append(s)
    return torch.cat(xs), torch.cat(srcs), torch.cat(dsts), torch.cat(eas), torch.stack(ss), flag


def library_tables(library):
    """(sample [V], offsets [V+1], node_index [S], seq_index [S], residue [S]) of a list of (sample, substitutions)."""
    subs = [t for _, s in library for t in s]
    counts = torch.tensor([len(s) for _, s in library], dtype=torch.int64)
    offsets = torch.cat([torch.zeros(1, dtype=torch.int64), counts.cumsum(0)])
    tab = torch.tensor(subs, dtype=torch.int64).reshape(-1, 3)
    return torch.tensor([b for b, _ in library], dtype=torch.int64), offsets, tab[:, 0].contiguous(), \
        tab[:, 1].contiguous(), tab[:, 2].contiguous()


def run_contract(arr, seq, cols, sample, offsets, ni, si, res, fill=float("nan")):
    """The contract on a graph-array batch, outputs prefilled with ``fill``: (x23, src, dst, edge_attr, seq, flag)."""
    off = torch.cat([torch.zeros(1, dtype=torch.int64), arr["node_counts"].cumsum(0)])
    eoff = torch.cat([torch.zeros(1, dtype=torch.int64), arr["edge_counts"].cumsum(0)])
    sb = sample.clamp(0, arr["node_counts"].numel() - 1)          # an out-of-range sample keeps a block of some graph
    nv, ev = arr["node_counts"][sb], arr["edge_counts"][sb]
    node_out = torch.cat([torch.zeros(1, dtype=torch.int64), nv.cumsum(0)])
    edge_out = torch.cat([torch.zeros(1, dtype=torch.int64), ev.cumsum(0)])
    r, (L, V) = sample.numel(), seq.shape[1:]
    xo = torch.full((int(node_out[-1]), 23), fill)
    so, do = torch.full((int(edge_out[-1]),), -7, dtype=torch.int64), torch.full((int(edge_out[-1]),), -7, dtype=torch.int64)
    eo = torch.full((int(edge_out[-1]), 1), fill)
    sq = torch.full((r, L, V), fill)
    flag = torch.zeros(1, dtype=torch.int32)
    variant_expand_contract(arr["x"], off, eoff, arr["src"], arr["dst"], arr["edge_attr"], seq, sample, offsets, ni, si,
                            res, cols, node_out, edge_out, xo, so, do, eo, sq, flag)
    return xo, so, do, eo, sq, int(flag)


def _ragged_case(seed=0, V=21, L=12):
    """Four graphs of 12, 5, 30 and 1 nodes (graph 3 has no edge); graphs 0 and 2 end in two all-zero padded rows.  The
    sequence rows 0..11 carry the residues of node rows 0..11 under a permuted ``seq_columns`` where the graph holds them
    and random residues past its end."""
    gen = torch.Generator().manual_seed(seed)
    counts = [12, 5, 30, 1]
    ecounts = [40, 9, 100, 0]
    n = sum(counts)
    aa = torch.randint(0, 20, (n,), generator=gen)
    x = torch.cat([F.one_hot(aa, 20).float(), torch.randn(n, 3, generator=gen)], 1)
    off = torch.tensor([0] + counts).cumsum(0)
    for i in (0, 2):
        x[off[i + 1] - 2:off[i + 1], :20] = 0.0
    src = torch.cat([torch.randint(0, max(c, 1), (e,), generator=gen) for c, e in zip(counts, ecounts)])
    dst = torch.cat([torch.randint(0, max(c, 1), (e,), generator=gen) for c, e in zip(counts, ecounts)])
    cols = torch.randperm(V, generator=gen)[:20]
    tok = cols[torch.randint(0, 20, (4, L), generator=gen)]
    for i in range(4):
        for p in range(min(L, counts[i])):
            if x[off[i] + p, :20].any():
                tok[i, p] = cols[aa[off[i] + p]]
    arr = {"x": x, "src": src, "dst": dst, "edge_attr": torch.rand(sum(ecounts), 1, generator=gen),
           "node_counts": torch.tensor(counts), "edge_counts": torch.tensor(ecounts)}
    return arr, F.one_hot(tok, V).float(), cols


# graph 0: rows 10, 11 padded; graph 1: 5 rows; graph 2: rows 28, 29 padded; graph 3: 1 row
LIBRARY = [
    (2, [(0, 0, 3), (5, 5, 17)]),
    (0, []),                                                      # an empty variant: the base sample, as a control
    (0, [(1, 1, 4)]),
    (3, [(0, 0, 9), (-1, 6, 2)]),                                 # the second substitution is in the sequence only
    (2, [(p, p, (3 * p) % 20) for p in range(12)]),               # twelve substitutions
    (1, [(-1, 7, 11), (-1, 8, 0)]),                               # sequence only
    (0, [(1, 1, 4)]),                                             # a repeated variant
    (2, [(9, 9, 19), (2, 2, 0)]),                                 # out of table order
]


@pytest.mark.parametrize("which", ["all", "first", "reversed", "one"])
def test_contract_equals_explicit_edits(which):
    arr, seq, cols = _ragged_case()
    lib = {"all": LIBRARY, "first": LIBRARY[:3], "reversed": LIBRARY[::-1], "one": LIBRARY[4:5]}[which]
    got = run_contract(arr, seq, cols, *library_tables(lib))
    ref = _explicit(arr, seq, cols, lib)
    for a, b in zip(got[:5], ref[:5]):
        assert torch.equal(a, b)
    assert got[5] == ref[5] == 0
    assert torch.equal(got[0][:, 20:], torch.cat([arr["x"][int(arr["node_counts"][:b].sum()):][:int(arr["node_counts"][b])]
                                                   for b, _ in lib])[:, 20:])     # coordinates untouched


def test_contract_flags_bad_rows_maps_and_indices():
    arr, seq, cols = _ragged_case(1)
    cases = {
        "padded": [(0, [(10, 1, 3)])],                            # an all-zero padded row of graph 0
        "map": [(0, [(2, 2, 5)])],                                # sequence row 3 carries the residue of node row 3
        "seq_row": [(1, [(-1, 2, 5)])],                           # sequence row made two-hot below
        "node_range": [(1, [(5, 1, 3)])],                         # graph 1 has 5 nodes
        "below": [(1, [(-2, 1, 3)])],
        "seq_range": [(2, [(1, 12, 3)])],                         # L = 12
        "residue": [(2, [(1, 1, 20)])],
    }
    for edit, lib in cases.items():
        s = seq.clone()
        if edit == "map":
            s[0, 2], s[0, 3] = s[0, 3].clone(), s[0, 2].clone()
            if torch.equal(s[0, 2], seq[0, 2]):
                s[0, 2] = F.one_hot((seq[0, 2].argmax() + 1) % 21, 21).float()
        if edit == "seq_row":
            s[1, 2, (s[1, 2].argmax() + 1) % 21] = 1.0
        lib = [(0, [(1, 1, 4)])] + lib                            # a good variant next to it is still applied
        got = run_contract(arr, s, cols, *library_tables(lib))
        ref = _explicit(arr, s, cols, lib)
        assert got[5] == ref[5] == 1, edit
        for a, b in zip(got[:5], ref[:5]):
            assert torch.equal(a, b), edit
    tables = list(library_tables(LIBRARY[:3]))
    for edit in ("sample", "offsets"):                            # a variant that cannot be read is flagged
        t = [x.clone() for x in tables]
        if edit == "sample":
            t[0][1] = 4
        else:
            t[1][2] = 9
        got = run_contract(arr, seq, cols, *t)
        assert got[5] == 1, edit
        if edit == "sample":
            assert torch.isnan(got[4][1]).all() and not torch.isnan(got[4][0]).any()
        else:                                                     # variant 1 copied, nothing substituted
            assert torch.equal(got[4][1], seq[0])


@pytest.mark.parametrize("max_graphs", [1, 3, 4, 7, 4096])
def test_pass_split(max_graphs):
    passes = variant_passes(10, max_graphs)
    assert [j for j, _ in passes] == list(range(0, 10, max_graphs))
    assert all(r == max_graphs for _, r in passes[:-1]) and 1 <= passes[-1][1] <= max_graphs
    assert sum(r for _, r in passes) == 10
    with pytest.raises(ValueError, match="max_graphs"):
        variant_passes(10, 0)


# ---- whole runs through the kernel contracts ------------------------------------------------------------------------
@pytest.fixture
def cpu_backend(monkeypatch):
    for name in KC.ALL:
        monkeypatch.setattr(_C, name, getattr(KC, name))
    monkeypatch.setattr(_C, "head_mc_infer", head_mc_infer_contract)
    monkeypatch.setattr(_C, "variant_expand", variant_expand_contract)
    monkeypatch.setattr(trunk, "_require_device_batch", lambda g: None)
    yield


def _golden_library(arrays, seq):
    """A library on the golden batch (graphs of 12 nodes, rows 10 and 11 padded): sequence rows 2..7 carry the residues of
    node rows 0..5 under the reversed alphabet map.  -> (cols, seq, list of (sample, substitutions))."""
    cols = torch.arange(20).flip(0)
    off = torch.cat([torch.zeros(1, dtype=torch.int64), arrays["node_counts"].cumsum(0)])
    seq = seq.clone()
    for i in range(arrays["node_counts"].numel()):
        for p in range(6):
            seq[i, 2 + p] = F.one_hot(cols[arrays["x"][off[i] + p, :20].argmax()], seq.shape[2]).float()
    lib = [(1, [(0, 2, 5)]), (0, []), (2, [(0, 2, 0), (3, 5, 19), (-1, 9, 7)]), (0, [(5, 7, 12), (1, 3, 1)]),
           (1, [(0, 2, 5)]), (2, [(4, 6, 8)])]
    return cols, seq, lib


def _mutant_batch(arrays, seq, cols, lib):
    """The host-built mutant batch of a library: graph arrays and sequences of the variants in order."""
    x, src, dst, ea, s, flag = _explicit(arrays, seq, cols, lib)
    samples = torch.tensor([b for b, _ in lib])
    assert flag == 0
    return {"x": x, "src": src, "dst": dst, "edge_attr": ea, "node_counts": arrays["node_counts"][samples],
            "edge_counts": arrays["edge_counts"][samples]}, s, samples


def _og64(arrays):
    g = oracle_graph(arrays)
    return dict(g, x=g["x"].double(), edge_attr=g["edge_attr"].double())


@pytest.mark.parametrize("max_graphs", [1, 4, 4096])
def test_score_variants_matches_fp64_oracle_per_mutant(cpu_backend, max_graphs):
    gd = load_golden("hybrid_v2")
    model = build_model("HybridModelv2", gd)
    d = gd["dense"]
    cols, seq, lib = _golden_library(gd["graph"], d["seq"])
    eps = torch.randn(2, 3, 32, generator=torch.Generator().manual_seed(3))
    res = score_variants(model, graph_batch(gd["graph"]), seq, d["prop"], *library_tables(lib), seq_columns=cols, eps=eps,
                         max_graphs=max_graphs)
    assert res.logits.shape == (6, 2) and res.prob_mean.shape == res.prob_std.shape == (6,)
    arr, s, samples = _mutant_batch(gd["graph"], seq, cols, lib)
    p64 = {k: v.detach().double() for k, v in model.state_dict().items()}
    for k in range(2):
        ref = R.hybrid_forward(p64, _og64(arr), s.double(), d["prop"][samples].double(), eps[k][samples].double(),
                               version="v2", n_layers=int(gd["meta"]["gcn_layers"]))[3].reshape(-1)
        assert rel_err(res.logits[:, k], ref) < TOL, k
    assert torch.allclose(res.logits[1], res.base.logits[0], rtol=0, atol=1e-6)            # the empty variant
    assert torch.allclose(res.logits[0], res.logits[4], rtol=0, atol=1e-6)                 # a repeated variant
    pr = torch.sigmoid(res.logits.double())
    assert float((res.prob_mean.double() - pr.mean(-1)).abs().max()) < 1e-7
    assert float((res.prob_std.double() - pr.std(-1, unbiased=False)).abs().max()) < 1e-7
    assert all(q.grad is None for q in model.parameters())


@pytest.mark.parametrize("use_wt", [True, False])
def test_score_variants_pair_matches_fp64_oracle_and_draws_once_per_item(cpu_backend, use_wt):
    gd = load_golden("comparative_v2")
    model = _comparative(use_wt, gd)
    d = gd["dense"]
    cols, seq_c, lib = _golden_library(gd["graph_c"], d["seq_c"])
    calls = []

    def sample_eps(like):
        calls.append(torch.randn(like.shape, generator=torch.Generator().manual_seed(20 + len(calls))))
        return calls[-1]

    model.sample_eps = sample_eps
    gc, gw = graph_batch(gd["graph_c"]), graph_batch(gd["graph_w"])
    res = score_variants_pair(model, (gc, gw), (seq_c, d["seq_w"]), (d["prop_c"], d["prop_w"]), *library_tables(lib),
                              seq_columns=cols, samples=2, max_graphs=4)
    b = gd["graph_c"]["node_counts"].numel()
    assert [tuple(c.shape) for c in calls] == [(2 * b, 32)] * (2 if use_wt else 1)
    eps_c = calls[0].reshape(2, b, 32)
    eps_w = calls[1].reshape(2, b, 32) if use_wt else torch.zeros(2, b, 32)
    arr, s, samples = _mutant_batch(gd["graph_c"], seq_c, cols, lib)
    wt = {k: v[samples] for k, v in gd["graph_w"].items() if k in ("node_counts", "edge_counts")}
    xw, srcw, dstw, eaw, sw, _ = _explicit(gd["graph_w"], d["seq_w"], torch.arange(20), [(int(i), []) for i in samples])
    arr_w = dict(wt, x=xw, src=srcw, dst=dstw, edge_attr=eaw)
    p64 = {k: v.detach().double() for k, v in model.state_dict().items()}
    for k in range(2):
        ref = R.comparative_forward(p64, (_og64(arr), _og64(arr_w)), (s.double(), sw.double()),
                                    (d["prop_c"][samples].double(), d["prop_w"][samples].double()),
                                    (eps_c[k][samples].double(), eps_w[k][samples].double()),
                                    n_layers=int(gd["meta"]["gcn_layers"]), use_wt=use_wt)[4].reshape(-1)
        assert rel_err(res.logits[:, k], ref) < TOL, k


def _hybrid_args(gd):
    d = gd["dense"]
    cols, seq, lib = _golden_library(gd["graph"], d["seq"])
    return graph_batch(gd["graph"]), seq, d["prop"], cols, library_tables(lib)


def test_errors_before_any_kernel_call(cpu_backend, monkeypatch):
    gd = load_golden("hybrid_v2")
    model = build_model("HybridModelv2", gd)
    g, seq, prop, cols, tables = _hybrid_args(gd)
    launched = []
    for name in ("variant_expand", "head_mc_infer", "collate_csr"):
        monkeypatch.setattr(_C, name, lambda *a, **k: launched.append(1))

    def bad(exc, match, m=model, **kw):
        args = dict(zip(("sample", "offsets", "node_index", "seq_index", "residue"), tables), seq_columns=cols)
        args.update(kw)
        with pytest.raises(exc, match=match):
            score_variants(m, g, seq, prop, *(args.pop(n) for n in ("sample", "offsets", "node_index", "seq_index",
                                                                    "residue")), **args)

    sample, offsets, ni, si, res = tables
    bad(ValueError, "int64", sample=sample.int())
    bad(ValueError, "int64", node_index=ni.reshape(-1, 1))
    bad(ValueError, "at least one variant", sample=sample[:0], offsets=offsets[:1])
    bad(ValueError, "V \\+ 1", offsets=offsets[:-1])
    bad(ValueError, "one entry per substitution", residue=res[:-1])
    bad(ValueError, r"sample must index", sample=torch.where(sample == 2, 3, sample))
    bad(ValueError, r"sample must index", sample=torch.where(sample == 2, -1, sample))
    for o in (offsets + 1, offsets.flip(0), torch.cat([offsets[:-1], offsets[-1:] + 1])):
        bad(ValueError, "offsets must start", offsets=o)
    past = ni.clone()
    past[0] = 12                                                          # graphs have 12 nodes
    bad(ValueError, "node_index", node_index=past)
    below = ni.clone()
    below[0] = -2
    bad(ValueError, "node_index", node_index=below)
    bad(ValueError, "sequence length", seq_index=torch.where(si == 9, seq.shape[1], si))
    bad(ValueError, "sequence length", seq_index=si - 3)
    bad(ValueError, "residue", residue=torch.where(res == 19, 20, res))
    bad(ValueError, "residue", residue=res - 1)
    bad(ValueError, "seq_columns", seq_columns=cols[:19])
    bad(ValueError, "seq_columns", seq_columns=torch.zeros(20, dtype=torch.int64))
    bad(ValueError, "seq_columns", seq_columns=cols + 2)                 # 21 and 22 are past V = 21
    bad(ValueError, "seq_columns", seq_columns=cols.float())
    twice = ni.clone()
    twice[2] = twice[1]                                                   # variant 2 (entries 1..3): node row 0 twice
    bad(ValueError, "same node row twice", node_index=twice)
    twice = si.clone()
    twice[3] = twice[1]                                                   # variant 2: sequence row 2 twice
    bad(ValueError, "same sequence row twice", seq_index=twice)
    bad(ValueError, "max_graphs", max_graphs=0)
    bad(ValueError, "samples", samples=0)
    for name in ("StructureModel", "StructureModelv2", "SequenceModel", "DualModel"):
        bad(NotImplementedError, "HybridModelv2_SSL", m=I.model_map[name](vae_input_dim=231, device="cpu").eval())
    with pytest.raises(NotImplementedError, match="HybridModel_Comparative"):
        score_variants_pair(model, (g, g), (seq, seq), (prop, prop), *tables, seq_columns=cols)
    model.train()
    bad(RuntimeError, "eval")
    assert not launched


def test_rows_shared_across_variants_are_allowed(cpu_backend):
    """The same node row in two variants, and a node row and a sequence row of equal index, are not repeats."""
    gd = load_golden("hybrid_v2")
    model = build_model("HybridModelv2", gd)
    g, seq, prop, cols, _ = _hybrid_args(gd)
    lib = [(0, [(2, 4, 1), (4, 6, 2)]), (0, [(2, 4, 3)])]
    res = score_variants(model, g, seq, prop, *library_tables(lib), seq_columns=cols)
    assert res.logits.shape == (2, 1) and torch.isfinite(res.logits).all()


def test_flag_raises_after_the_passes(cpu_backend):
    gd = load_golden("hybrid_v2")
    model = build_model("HybridModelv2", gd)
    g, seq, prop, cols, tables = _hybrid_args(gd)
    padded = tables[2].clone()
    padded[0] = 11                                                        # rows 10 and 11 of each graph are padding
    with pytest.raises(ValueError, match="one-hot"):
        score_variants(model, g, seq, prop, tables[0], tables[1], padded, *tables[3:], seq_columns=cols, max_graphs=2)
    with pytest.raises(ValueError, match="seq_columns"):
        score_variants(model, g, seq, prop, *tables, seq_columns=cols.roll(3))
