"""Structural occlusion (immunostruct_b200/occlusion.py), host logic on CPU: the contract of the expansion kernel
(is_occlusion_expand) against explicit per-variant boolean-mask edits, every flag case, every error raised before a kernel
call, the pass split, and whole runs through the per-kernel contracts against the fp64 oracle's forward on each host-built
occluded graph, single and pair.  The device kernel is checked in tests/test_occlusion_gpu.py, which shares
``occlusion_expand_contract``."""
import pytest
import torch

import immunostruct_b200 as I
from immunostruct_b200 import _C, trunk
from immunostruct_b200.occlusion import (_contact_tables, _residue_tables, occlude_contacts, occlude_contacts_pair,
                                         occlude_residues, occlude_residues_pair)
from immunostruct_b200.resident import variant_passes
from oracle import kernel_contracts as KC
from oracle import reference_ops as R

from conftest import load_golden, oracle_graph, rel_err
from helpers import build_model, graph_batch
from test_predictive_host import _comparative, head_mc_infer_contract

TOL = 1e-4


def occlusion_expand_contract(x23, node_off, edge_off, src_local, dst_local, edge_attr, sample, node_a, node_b, node_out,
                              edge_out, x23_out, src_out, dst_out, edge_attr_out, flag):
    """Contract of is_occlusion_expand (signature of ``_C.occlusion_expand``): variant v is base graph s = sample[v] with
    row a = node_a[v] zeroed and every edge touching it dropped (node_b[v] == -1), or every edge between a and node_b[v]
    dropped (rows unchanged); rows go to node_out[v]..., the kept edges in base order (graph-local endpoints, attributes)
    to edge_out[v]....  flag |= 1, and the variant is not written, for a sample outside [0, B), a outside [0, n_s),
    node_b outside [-1, n_s) or equal to a, node_out[v+1] - node_out[v] != n_s, a kept count that is not
    edge_out[v+1] - edge_out[v], or offsets past the outputs."""
    b = node_off.numel() - 1
    n_out, e_out = x23_out.shape[0], src_out.shape[0]
    bad = False
    for v in range(sample.numel()):
        s, a, b2 = int(sample[v]), int(node_a[v]), int(node_b[v])
        if not 0 <= s < b:
            bad = True
            continue
        n0, nb = int(node_off[s]), int(node_off[s + 1] - node_off[s])
        e0, eb = int(edge_off[s]), int(edge_off[s + 1] - edge_off[s])
        no, n1, eo, e1 = int(node_out[v]), int(node_out[v + 1]), int(edge_out[v]), int(edge_out[v + 1])
        if not (0 <= a < nb and -1 <= b2 < nb and b2 != a and no >= 0 and n1 - no == nb and n1 <= n_out and eo >= 0
                and e1 >= eo and e1 <= e_out):
            bad = True
            continue
        src, dst = src_local[e0:e0 + eb], dst_local[e0:e0 + eb]
        hit = (src == a) | (dst == a) if b2 < 0 else ((src == a) & (dst == b2)) | ((src == b2) & (dst == a))
        keep = (~hit).nonzero().flatten()
        if keep.numel() != e1 - eo:
            bad = True
            continue
        x23_out[no:n1] = x23[n0:n0 + nb]
        if b2 < 0:
            x23_out[no + a] = 0.0
        src_out[eo:e1], dst_out[eo:e1] = src[keep], dst[keep]
        edge_attr_out.reshape(-1)[eo:e1] = edge_attr.reshape(-1)[e0 + keep]
    if bad:
        flag.fill_(1)


def _offsets(counts):
    return torch.cat([torch.zeros(1, dtype=torch.int64), torch.as_tensor(counts, dtype=torch.int64).cumsum(0)])


def _explicit(arr, variants):
    """The same variants built one by one with a boolean edge mask: graph arrays of the occluded graphs in order.
    ``variants``: a list of (sample, a, b), b = -1 for a residue."""
    off, eoff = _offsets(arr["node_counts"]), _offsets(arr["edge_counts"])
    xs, srcs, dsts, eas, nc, ec = [], [], [], [], [], []
    for s, a, b in variants:
        x = arr["x"][off[s]:off[s + 1]].clone()
        src, dst, ea = (arr[k][eoff[s]:eoff[s + 1]] for k in ("src", "dst", "edge_attr"))
        if b < 0:
            x[a] = 0.0
            mask = (src != a) & (dst != a)
        else:
            mask = ~(((src == a) & (dst == b)) | ((src == b) & (dst == a)))
        xs.append(x)
        srcs.append(src[mask])
        dsts.append(dst[mask])
        eas.append(ea[mask])
        nc.append(x.shape[0])
        ec.append(int(mask.sum()))
    return {"x": torch.cat(xs), "src": torch.cat(srcs), "dst": torch.cat(dsts), "edge_attr": torch.cat(eas),
            "node_counts": torch.tensor(nc), "edge_counts": torch.tensor(ec)}


def run_contract(arr, variants, fill=float("nan"), node_out=None, edge_out=None):
    """The contract on a graph-array batch and a list of (sample, a, b), outputs prefilled with ``fill``; the offsets are
    those of the explicit edits unless given (a variant the kernel must reject gets the block of row 0 of a graph).
    -> (x23, src, dst, edge_attr, flag)."""
    nc = arr["node_counts"].tolist()
    fine = lambda s, a, b: 0 <= s < len(nc) and 0 <= a < nc[s] and -1 <= b < nc[s] and a != b
    ref = _explicit(arr, [v if fine(*v) else (min(max(v[0], 0), len(nc) - 1), 0, -1) for v in variants])
    node_out = _offsets(ref["node_counts"]) if node_out is None else node_out
    edge_out = _offsets(ref["edge_counts"]) if edge_out is None else edge_out
    n, e = int(node_out[-1]), int(edge_out[-1])
    xo, eo = torch.full((n, 23), fill), torch.full((e, 1), fill)
    so, do = torch.full((e,), -7, dtype=torch.int64), torch.full((e,), -7, dtype=torch.int64)
    flag = torch.zeros(1, dtype=torch.int32)
    t = torch.tensor(variants, dtype=torch.int64).reshape(-1, 3)
    occlusion_expand_contract(arr["x"], _offsets(arr["node_counts"]), _offsets(arr["edge_counts"]), arr["src"], arr["dst"],
                              arr["edge_attr"], t[:, 0].contiguous(), t[:, 1].contiguous(), t[:, 2].contiguous(), node_out,
                              edge_out, xo, so, do, eo, flag)
    return xo, so, do, eo, int(flag)


def hand_case(seed=0):
    """Four ragged graphs.  Graph 0 (7 nodes): shuffled edges with a multi-edge (2->3 twice and 3->2), a self-loop on 4,
    an isolated residue 6 and an absent (all-zero, edgeless) row 5.  Graph 1: 3 nodes.  Graph 2: 40 nodes and 600 random
    edges, more than one 256-edge CTA round, with self-loops and repeats.  Graph 3: one node, no edge."""
    gen = torch.Generator().manual_seed(seed)
    e0 = torch.tensor([[0, 1], [1, 0], [2, 3], [2, 3], [3, 2], [4, 4], [1, 2], [3, 4], [4, 0], [0, 3], [2, 0]])
    e0 = e0[torch.randperm(e0.shape[0], generator=gen)]
    e1 = torch.tensor([[0, 1], [2, 1], [1, 2]])
    e2 = torch.randint(0, 40, (600, 2), generator=gen)
    counts, edges = [7, 3, 40, 1], [e0, e1, e2, torch.zeros(0, 2, dtype=torch.int64)]
    x = torch.randn(sum(counts), 23, generator=gen)
    x[5] = 0.0
    return {"x": x, "src": torch.cat([e[:, 0] for e in edges]), "dst": torch.cat([e[:, 1] for e in edges]),
            "edge_attr": torch.rand(sum(e.shape[0] for e in edges), 1, generator=gen),
            "node_counts": torch.tensor(counts), "edge_counts": torch.tensor([e.shape[0] for e in edges])}


def _contacts_of(arr):
    """Every (sample, u, v) contact of the batch, u < v, in order."""
    eoff = _offsets(arr["edge_counts"])
    out = []
    for s in range(arr["node_counts"].numel()):
        pairs = {(min(a, b), max(a, b)) for a, b in zip(arr["src"][eoff[s]:eoff[s + 1]].tolist(),
                                                        arr["dst"][eoff[s]:eoff[s + 1]].tolist()) if a != b}
        out += [(s, u, v) for u, v in sorted(pairs)]
    return out


def _residues_of(arr):
    return [(s, a, -1) for s, n in enumerate(arr["node_counts"].tolist()) for a in range(n)]


@pytest.mark.parametrize("which", ["residues", "contacts", "mixed", "reversed"])
def test_contract_equals_explicit_edits(which):
    arr = hand_case()
    res, con = _residues_of(arr), _contacts_of(arr)
    assert (0, 2, 3) in con and (0, 0, 4) in con and len(res) == 51
    variants = {"residues": res, "contacts": con, "mixed": res[::3] + con[::5], "reversed": (res + con)[::-1]}[which]
    got = run_contract(arr, variants)
    ref = _explicit(arr, variants)
    assert got[4] == 0
    for a, k in zip(got[:4], ("x", "src", "dst", "edge_attr")):
        assert torch.equal(a, ref[k]), k


def test_contract_drops_exactly_the_touching_edges():
    arr = hand_case()
    x, src, dst, ea, flag = run_contract(arr, [(0, 2, 3), (0, 4, -1), (0, 3, -1), (0, 6, -1), (0, 5, -1)])
    assert flag == 0
    counts = [11 - 3, 11 - 3, 11 - 5, 11, 11]                # {2,3}: three edges; row 4: 4->4, 3->4, 4->0; row 3: five
    assert torch.equal(_offsets(counts)[-1], torch.tensor(src.numel()))
    assert torch.equal(x[7 + 4], torch.zeros(23)) and torch.equal(x[3 * 7 + 6], torch.zeros(23))
    assert torch.equal(x[:7], arr["x"][:7])                   # a contact leaves the rows alone


def test_contract_flags():
    arr = hand_case(1)
    good = [(0, 1, -1), (2, 3, 9)]
    cases = {"sample": (4, 0, -1), "below": (-1, 0, -1), "a_past": (1, 3, -1), "a_below": (1, -1, -1),
             "b_past": (1, 0, 3), "b_below": (1, 0, -2), "b_equal": (2, 5, 5)}
    ref = run_contract(arr, good + good)
    for name, bad in cases.items():
        got = run_contract(arr, good + [bad] + good)
        assert got[4] == 1, name
        nodes = int(arr["node_counts"][0] + arr["node_counts"][2])
        skipped = got[0].shape[0] - ref[0].shape[0]                  # the rejected variant's block stays NaN-filled
        assert torch.isnan(got[0][nodes:nodes + skipped]).all(), name
        assert torch.equal(torch.cat([got[0][:nodes], got[0][nodes + skipped:]]), ref[0]), name
    # offsets that disagree with variant 1: a node block one row too long, an edge block one edge longer than its kept
    # count; variants 0 and 2 are still written, variant 1 is not
    lib = [(0, 1, -1), (2, 3, 9), (1, 0, -1)]
    ref = _explicit(arr, lib)
    no, eo = _offsets(ref["node_counts"]), _offsets(ref["edge_counts"])
    one = torch.tensor([0, 0, 1, 1])
    for name, (n_, e_) in {"nodes": (no + one, eo), "kept": (no, eo + one)}.items():
        got = run_contract(arr, lib, node_out=n_, edge_out=e_)
        assert got[4] == 1, name
        assert torch.equal(got[0][:7], ref["x"][:7]) and torch.equal(got[0][int(n_[2]):], ref["x"][int(no[2]):]), name
        assert torch.isnan(got[0][7:int(n_[2])]).all() and (got[1][int(e_[1]):int(e_[2])] == -7).all(), name
        assert torch.equal(got[1][int(e_[2]):], ref["src"][int(eo[2]):]), name
    xo = torch.full((int(no[-1]), 23), float("nan"))               # outputs shorter than the offsets claim
    so, do = torch.full((int(eo[-1]) - 1,), -7), torch.full((int(eo[-1]) - 1,), -7)
    ea_o, flag = torch.full((int(eo[-1]) - 1, 1), float("nan")), torch.zeros(1, dtype=torch.int32)
    t = torch.tensor(lib)
    occlusion_expand_contract(arr["x"], _offsets(arr["node_counts"]), _offsets(arr["edge_counts"]), arr["src"], arr["dst"],
                              arr["edge_attr"], t[:, 0], t[:, 1], t[:, 2], no, eo, xo, so, do, ea_o, flag)
    assert int(flag) == 1 and torch.isnan(xo[int(no[2]):]).all() and not torch.isnan(xo[:int(no[2])]).any()


# ---- tables and the pass split ----------------------------------------------------------------------------------------
@pytest.fixture
def cpu_backend(monkeypatch):
    for name in KC.ALL:
        monkeypatch.setattr(_C, name, getattr(KC, name))
    monkeypatch.setattr(_C, "head_mc_infer", head_mc_infer_contract)
    monkeypatch.setattr(_C, "occlusion_expand", occlusion_expand_contract)
    monkeypatch.setattr(trunk, "_require_device_batch", lambda g: None)
    yield


def _run_passes(arr, tables):
    """The contract run pass by pass with the tables' offsets and totals, concatenated -> (x, src, dst, edge_attr, flag)."""
    smp, na, nb, nv, kept, ncs, ecs, passes, node_tot, edge_tot, c = tables
    g = graph_batch(arr)
    outs, flag = [], 0
    for (j, r), n_p, e_p in zip(passes, node_tot, edge_tot):
        xo, eo = torch.full((n_p, 23), float("nan")), torch.full((e_p, 1), float("nan"))
        so, do = torch.full((e_p,), -7), torch.full((e_p,), -7)
        f = torch.zeros(1, dtype=torch.int32)
        occlusion_expand_contract(arr["x"], g.node_off, g.edge_off, arr["src"], arr["dst"], arr["edge_attr"], smp[j:j + r],
                                  na[j:j + r], nb[j:j + r], ncs[j:j + r + 1] - ncs[j], ecs[j:j + r + 1] - ecs[j], xo, so,
                                  do, eo, f)
        outs.append((xo, so, do, eo))
        flag |= int(f)
    return [torch.cat(t) for t in zip(*outs)] + [flag]


@pytest.mark.parametrize("max_graphs", [1, 5, 7, 4096])
def test_tables_and_pass_split(cpu_backend, max_graphs):
    arr = hand_case(2)
    g = graph_batch(arr)
    res, con = _residues_of(arr), _contacts_of(arr)
    present = [v for v in res if v[:2] != (0, 5)]                     # row 5 of graph 0 is absent
    for tables, variants in ((_residue_tables(g, None, max_graphs)[0], present),
                             (_contact_tables(g, None, max_graphs)[0], con)):
        smp, na, nb, nv, kept, ncs, ecs, passes, node_tot, edge_tot, c = tables
        assert c == len(variants)
        assert [tuple(t) for t in torch.stack([smp, na, nb], 1).tolist()] == variants
        assert passes == variant_passes(c, max_graphs)
        if max_graphs in (5, 7):                                      # a pass boundary falls inside a sample
            assert any(int(smp[j - 1]) == int(smp[j]) for j, _ in passes[1:])
        ref = _explicit(arr, variants)
        assert torch.equal(kept, ref["edge_counts"]) and torch.equal(nv, ref["node_counts"])
        got = _run_passes(arr, tables)
        assert got[4] == 0
        for a, k in zip(got[:4], ("x", "src", "dst", "edge_attr")):
            assert torch.equal(a, ref[k]), k


def test_selection(cpu_backend):
    arr = hand_case(3)
    g = graph_batch(arr)
    n = int(arr["node_counts"].sum())
    sel = torch.zeros(n, dtype=torch.bool)
    sel[[5, 2, 10 + 7]] = True                                         # the absent row is scored when selected
    tables, rows = _residue_tables(g, sel, 4096)
    assert rows.tolist() == [2, 5, 17] and tables[-1] == 3
    assert [int(t) for t in tables[1]] == [2, 5, 7]
    tables, ec = _contact_tables(g, sel, 4096)                        # contacts with an endpoint at row 2 or graph-2 row 7
    con = [v for v in _contacts_of(arr) if (v[0] == 0 and 2 in v[1:]) or (v[0] == 2 and 7 in v[1:])]
    assert [tuple(t) for t in torch.stack(tables[:3], 1).tolist()] == con
    eoff = _offsets(arr["edge_counts"])
    for e in range(int(eoff[-1])):
        s = int(torch.searchsorted(eoff, e, right=True)) - 1
        a, b = int(arr["src"][e]), int(arr["dst"][e])
        key = (s, min(a, b), max(a, b))
        assert int(ec[e]) == (con.index(key) if a != b and key in con else -1)


# ---- errors before any kernel call --------------------------------------------------------------------------------------
def test_errors_before_any_kernel_call(cpu_backend, monkeypatch):
    gd = load_golden("hybrid_v2")
    model = build_model("HybridModelv2", gd)
    d = gd["dense"]
    g = graph_batch(gd["graph"])
    launched = []
    for name in ("occlusion_expand", "head_mc_infer", "collate_csr", "linear_tc", "vae_mid_infer"):
        monkeypatch.setattr(_C, name, lambda *a, **k: launched.append(1))
    n = g.n_nodes
    for fn in (occlude_residues, occlude_contacts):
        def bad(exc, match, m=model, **kw):
            with pytest.raises(exc, match=match):
                fn(m, g, d["seq"], d["prop"], **kw)

        bad(ValueError, "bool tensor", nodes=torch.ones(n, dtype=torch.int64))
        bad(ValueError, "bool tensor", nodes=torch.ones(n + 1, dtype=torch.bool))
        bad(ValueError, "bool tensor", nodes=[True] * n)
        bad(ValueError, "nothing to occlude", nodes=torch.zeros(n, dtype=torch.bool))
        bad(ValueError, "max_graphs", max_graphs=0)
        bad(ValueError, "samples", samples=0)
        bad(ValueError, "eps", eps=torch.zeros(2, 2, 32))
        for name in ("StructureModel", "StructureModelv2", "SequenceModel", "DualModel"):
            bad(NotImplementedError, "HybridModelv2_SSL", m=I.model_map[name](vae_input_dim=231, device="cpu").eval())
        model.train()
        bad(RuntimeError, "eval")
        model.eval()
    absent = torch.zeros(n, dtype=torch.bool)
    absent[[10, 11]] = True                                           # padded rows: no contact
    with pytest.raises(ValueError, match="no contact"):
        occlude_contacts(model, g, d["seq"], d["prop"], nodes=absent)
    for fn in (occlude_residues_pair, occlude_contacts_pair):
        with pytest.raises(NotImplementedError, match="HybridModel_Comparative"):
            fn(model, (g, g), (d["seq"], d["seq"]), (d["prop"], d["prop"]))
    assert not launched


# ---- whole runs through the kernel contracts ------------------------------------------------------------------------
def _og64(arrays):
    g = oracle_graph(arrays)
    return dict(g, x=g["x"].double(), edge_attr=g["edge_attr"].double())


def _peptide_rows(arr, rows=3):
    """The first ``rows`` rows of every graph."""
    off = _offsets(arr["node_counts"])
    sel = torch.zeros(int(off[-1]), dtype=torch.bool)
    for s in range(arr["node_counts"].numel()):
        sel[off[s]:off[s] + rows] = True
    return sel


@pytest.mark.parametrize("mode,max_graphs", [("residues", 4096), ("residues", 7), ("contacts", 4096), ("contacts", 5)])
def test_occlusion_matches_fp64_oracle_per_variant(cpu_backend, mode, max_graphs):
    gd = load_golden("hybrid_v2")
    model = build_model("HybridModelv2", gd)
    d = gd["dense"]
    arr = gd["graph"]
    g = graph_batch(arr)
    eps = torch.randn(2, 3, 32, generator=torch.Generator().manual_seed(3))
    n = g.n_nodes
    if mode == "residues":
        nodes = _peptide_rows(arr, 4)
        nodes[10] = True                                              # an absent row, selected explicitly
        res = occlude_residues(model, g, d["seq"], d["prop"], nodes=nodes, eps=eps, max_graphs=max_graphs)
        rows = nodes.nonzero().flatten()
        variants = [(int(r) // 12, int(r) % 12, -1) for r in rows]
        logits = res.logits[rows]
        assert res.logits.shape == (n, 2) and torch.isnan(res.logits[~nodes]).all()
        assert torch.isnan(res.prob_mean[~nodes]).all() and not torch.isnan(res.prob_mean[nodes]).any()
        assert torch.allclose(res.logits[10], res.base.logits[0], rtol=0, atol=1e-6)
    else:
        res = occlude_contacts(model, g, d["seq"], d["prop"], nodes=_peptide_rows(arr, 2), eps=eps, max_graphs=max_graphs)
        variants = [v for v in _contacts_of(arr) if v[1] < 2]
        assert [tuple(t) for t in torch.stack([res.sample, res.u, res.v], 1).tolist()] == variants
        logits = res.logits
        assert res.edge_contact.shape == (g.n_edges,)
    occ = _explicit(arr, variants)
    samples = torch.tensor([v[0] for v in variants])
    p64 = {k: v.detach().double() for k, v in model.state_dict().items()}
    for k in range(2):
        ref = R.hybrid_forward(p64, _og64(occ), d["seq"][samples].double(), d["prop"][samples].double(),
                               eps[k][samples].double(), version="v2", n_layers=int(gd["meta"]["gcn_layers"]))[3].reshape(-1)
        assert rel_err(logits[:, k], ref) < TOL, k
    pr = torch.sigmoid(logits.double())
    mean = res.prob_mean[rows] if mode == "residues" else res.prob_mean
    std = res.prob_std[rows] if mode == "residues" else res.prob_std
    assert float((mean.double() - pr.mean(-1)).abs().max()) < 1e-7
    assert float((std.double() - pr.std(-1, unbiased=False)).abs().max()) < 1e-7
    assert all(q.grad is None for q in model.parameters())


@pytest.mark.parametrize("mode", ["residues", "contacts"])
@pytest.mark.parametrize("use_wt", [True, False])
def test_pair_matches_fp64_oracle_and_draws_once_per_item(cpu_backend, use_wt, mode):
    gd = load_golden("comparative_v2")
    model = _comparative(use_wt, gd)
    d = gd["dense"]
    calls = []

    def sample_eps(like):
        calls.append(torch.randn(like.shape, generator=torch.Generator().manual_seed(20 + len(calls))))
        return calls[-1]

    model.sample_eps = sample_eps
    arr_c, arr_w = gd["graph_c"], gd["graph_w"]
    gc, gw = graph_batch(arr_c), graph_batch(arr_w)
    args = ((gc, gw), (d["seq_c"], d["seq_w"]), (d["prop_c"], d["prop_w"]))
    nodes = _peptide_rows(arr_c, 2)
    if mode == "residues":
        res = occlude_residues_pair(model, *args, nodes=nodes, samples=2, max_graphs=3)
        rows = nodes.nonzero().flatten()
        variants = [(int(r) // 10, int(r) % 10, -1) for r in rows]
        logits = res.logits[rows]
    else:
        res = occlude_contacts_pair(model, *args, nodes=nodes, samples=2, max_graphs=3)
        variants = [v for v in _contacts_of(arr_c) if v[1] < 2]
        logits = res.logits
    b = arr_c["node_counts"].numel()
    assert [tuple(c.shape) for c in calls] == [(2 * b, 32)] * (2 if use_wt else 1)
    eps_c = calls[0].reshape(2, b, 32)
    eps_w = calls[1].reshape(2, b, 32) if use_wt else torch.zeros(2, b, 32)
    samples = torch.tensor([v[0] for v in variants])
    occ = _explicit(arr_c, variants)
    wt = _explicit(arr_w, [(int(s), 0, 9) for s in samples])         # {0, 9} is no contact: the wild type unchanged
    assert torch.equal(wt["edge_counts"], arr_w["edge_counts"][samples])
    p64 = {k: v.detach().double() for k, v in model.state_dict().items()}
    for k in range(2):
        ref = R.comparative_forward(p64, (_og64(occ), _og64(wt)), (d["seq_c"][samples].double(), d["seq_w"][samples].double()),
                                    (d["prop_c"][samples].double(), d["prop_w"][samples].double()),
                                    (eps_c[k][samples].double(), eps_w[k][samples].double()),
                                    n_layers=int(gd["meta"]["gcn_layers"]), use_wt=use_wt)[4].reshape(-1)
        assert rel_err(logits[:, k], ref) < TOL, k


def test_flag_raises_after_the_passes(cpu_backend, monkeypatch):
    gd = load_golden("hybrid_v2")
    model = build_model("HybridModelv2", gd)
    d = gd["dense"]
    g = graph_batch(gd["graph"])

    def wrong(*a):                                                    # a kernel that reports a rejected variant
        occlusion_expand_contract(*a)
        a[-1].fill_(1)

    monkeypatch.setattr(_C, "occlusion_expand", wrong)
    with pytest.raises(RuntimeError, match="rejected"):
        occlude_residues(model, g, d["seq"], d["prop"], max_graphs=4)
