"""Shapley values of contacts (immunostruct_b200/shapley.py, ``contact_shapley``), host logic on CPU: the contracts of the
two edge kernels (is_shapley_edge_plan: numpy uint32 Philox4x32-10 keys on counter word 3 = 3 and a rank histogram;
is_shapley_edge_expand: per-variant boolean edge-mask edits) against brute force and the definitions, the estimator on
synthetic set functions over edges, every error raised before a kernel call, the bool form's contact numbering against
occlusion's, and whole runs through the per-kernel contracts against the fp64 oracle's forward on each host-built
coalition graph, single and pair.  The device kernels are checked in tests/test_contact_shapley_gpu.py, which shares the
contracts; the reduction's contract is the residue game's (tests/test_shapley_host.py)."""
import numpy as np
import pytest
import torch

import immunostruct_b200 as I
from immunostruct_b200 import _C, occlusion, shapley, trunk
from immunostruct_b200.shapley import _edge_sizes, _plan, contact_shapley, contact_shapley_pair
from oracle import kernel_contracts as KC
from oracle import reference_ops as R

from conftest import load_golden
from helpers import build_model, graph_batch
from test_coordnoise_host import philox4x32_10
from test_occlusion_host import _contacts_of, _offsets, hand_case
from test_predictive_host import _comparative, head_mc_infer_contract
from test_shapley_host import (_exact, _og64, _oracle_phi, _redundant, plan_ranks, run_reduce,
                               shapley_reduce_contract)


# ---- the kernels' contracts ---------------------------------------------------------------------------------------------
def edge_plan_ranks(seed, b, u, p):
    """Rank of each of the P players of sample b in permutation 2u: order by (Philox key v0 of counter (p, b, u, 3), p)."""
    key = philox4x32_10((np.arange(p), b, u, 3), (seed & 0xFFFFFFFF, seed >> 32))[0]
    rank = np.empty(p, dtype=np.int64)
    rank[np.lexsort((np.arange(p), key))] = np.arange(p)
    return rank


def shapley_edge_plan_contract(edge_off, edge_players, player_off, var_off, seed, ranks, kept, flag):
    """Contract of is_shapley_edge_plan (signature of ``_C.shapley_edge_plan``): rank rows 2u / 2u+1 of every sample
    (-1 past P_b) and the kept-edge count of every variant, an edge of player q being kept in coalition j of permutation
    t iff j <= rank_t(q), an edge with an id outside [0, P_b) always.  flag |= 1 for P_b > min(256, Pmax) or a variant
    count that is not 1 + T (P_b - 1); that sample is not written."""
    b, t, pmax = ranks.shape
    eo, po, vo = (x.cpu().numpy() for x in (edge_off, player_off, var_off))
    ids = edge_players.cpu().numpy().astype(np.int64)
    rk, kp = ranks.cpu().numpy(), kept.cpu().numpy()
    bad = False
    for s in range(b):
        p, v0, nvar = int(po[s + 1] - po[s]), int(vo[s]), int(vo[s + 1] - vo[s])
        if not (0 <= p <= min(256, pmax) and nvar == (1 + t * (p - 1) if p else 0)):
            bad = True
            continue
        rk[s] = -1
        if p == 0:
            continue
        w = ids[int(eo[s]):int(eo[s + 1])]
        for u in range(t // 2):
            r0 = edge_plan_ranks(seed, s, u, p)
            for tt, r in ((2 * u, r0), (2 * u + 1, p - 1 - r0)):
                rk[s, tt, :p] = r
                m = np.where((w >= 0) & (w < p), r[np.clip(w, 0, p - 1)], p)
                suffix = np.cumsum(np.bincount(m, minlength=p + 1)[::-1])[::-1]    # suffix[j] = #{m >= j}
                kp[v0 + 1 + tt * (p - 1):v0 + 1 + (tt + 1) * (p - 1)] = suffix[1:p]
                kp[v0] = suffix[p]
    ranks.copy_(torch.from_numpy(rk))
    kept.copy_(torch.from_numpy(kp))
    if bad:
        flag.fill_(1)


def shapley_edge_expand_contract(x23, node_off, edge_off, src_local, dst_local, edge_attr, edge_players, ranks, sample,
                                 rank_row, threshold, node_out, edge_out, x23_out, src_out, dst_out, edge_attr_out,
                                 flag):
    """Contract of is_shapley_edge_expand (signature of ``_C.shapley_edge_expand``): variant v is base graph s =
    sample[v] with its rows copied and every edge e with edge_players[e] >= 0 and ranks[rank_row[v], edge_players[e]] <
    threshold[v] dropped; rows to node_out[v]..., the kept edges in base order to edge_out[v]....  flag |= 1, and the
    variant is not written, for an index out of range, an edge player id >= Pmax, or offsets that disagree with the
    counts."""
    b = node_off.numel() - 1
    rk = ranks.reshape(-1, ranks.shape[-1])
    n_rows, pmax = rk.shape
    n_out, e_out = x23_out.shape[0], src_out.shape[0]
    bad = False
    for v in range(sample.numel()):
        s, row, j = int(sample[v]), int(rank_row[v]), int(threshold[v])
        if not (0 <= s < b and 0 <= row < n_rows and 0 <= j <= pmax):
            bad = True
            continue
        n0, nb = int(node_off[s]), int(node_off[s + 1] - node_off[s])
        e0, eb = int(edge_off[s]), int(edge_off[s + 1] - edge_off[s])
        no, n1, eo, e1 = int(node_out[v]), int(node_out[v + 1]), int(edge_out[v]), int(edge_out[v + 1])
        ids = edge_players[e0:e0 + eb].long()
        if not (no >= 0 and n1 - no == nb and n1 <= n_out and eo >= 0 and e1 >= eo and e1 <= e_out) \
                or bool((ids >= pmax).any()):
            bad = True
            continue
        gone = (ids >= 0) & (rk[row][ids.clamp(0, pmax - 1)].long() < j)
        keep = (~gone).nonzero().flatten()
        if keep.numel() != e1 - eo:
            bad = True
            continue
        x23_out[no:n1] = x23[n0:n0 + nb]
        src_out[eo:e1], dst_out[eo:e1] = src_local[e0 + keep], dst_local[e0 + keep]
        edge_attr_out.reshape(-1)[eo:e1] = edge_attr.reshape(-1)[e0 + keep]
    if bad:
        flag.fill_(1)


# ---- helpers ----------------------------------------------------------------------------------------------------------
def edge_group_case(seed=0):
    """hand_case's four graphs with edge players: graph 0's 11 edges in 5 groups (one holds the self-loop's position,
    one edge never removed); graph 1 has no players; graph 2's 600 edges in 9 groups, every seventh edge a non-player;
    graph 3 has no edge."""
    arr = hand_case(seed)
    ids = torch.full((614,), -1, dtype=torch.int64)
    ids[:11] = torch.tensor([0, 1, 0, 2, -1, 3, 1, 2, 4, 0, 3])
    g2 = torch.arange(600) % 9
    g2[::7] = -1
    ids[14:] = g2
    return arr, ids


def _tables(arr, ids, t):
    """Counts, offsets and variant tables of the contract plan -> (P [B], player_off, var_off)."""
    eo = _offsets(arr["edge_counts"])
    p = torch.tensor([int(ids[eo[s]:eo[s + 1]].max()) + 1 if eo[s + 1] > eo[s] else 0
                      for s in range(len(eo) - 1)]).clamp_min(0)
    nvar = torch.where(p > 0, 1 + t * (p - 1), 0)
    return p, _offsets(p), _offsets(nvar)


def run_plan(arr, ids, t, seed):
    p, po, vo = _tables(arr, ids, t)
    ranks = torch.zeros(len(p), t, max(int(p.max()), 1), dtype=torch.int32)
    kept = torch.full((int(vo[-1]),), -7, dtype=torch.int64)
    flag = torch.zeros(1, dtype=torch.int32)
    shapley_edge_plan_contract(_offsets(arr["edge_counts"]), ids.to(torch.int32), po, vo, seed, ranks, kept, flag)
    return p, po, vo, ranks, kept, int(flag)


def chain(p, ranks, vo):
    """(sample, rank row, threshold) of every variant, in the call's order."""
    out = []
    t = ranks.shape[1]
    for s, ps in enumerate(p.tolist()):
        if ps:
            out.append((s, s * t, ps))
            out += [(s, s * t + tt, j) for tt in range(t) for j in range(1, ps)]
    assert len(out) == int(vo[-1])
    return out


def edge_coalitions(arr, ids, ranks, variants):
    """The variants built one by one with boolean edge masks: graph arrays of the coalition graphs in order."""
    off, eoff = _offsets(arr["node_counts"]), _offsets(arr["edge_counts"])
    rk = ranks.reshape(-1, ranks.shape[-1]).long()
    xs, srcs, dsts, eas, nc, ec = [], [], [], [], [], []
    for s, row, j in variants:
        local = ids[eoff[s]:eoff[s + 1]]
        gone = torch.tensor([bool(i >= 0 and rk[row, i] < j) for i in local.tolist()], dtype=torch.bool)
        src, dst, ea = (arr[k][eoff[s]:eoff[s + 1]] for k in ("src", "dst", "edge_attr"))
        xs.append(arr["x"][off[s]:off[s + 1]])
        srcs.append(src[~gone])
        dsts.append(dst[~gone])
        eas.append(ea[~gone])
        nc.append(int(off[s + 1] - off[s]))
        ec.append(int((~gone).sum()))
    return {"x": torch.cat(xs), "src": torch.cat(srcs), "dst": torch.cat(dsts), "edge_attr": torch.cat(eas),
            "node_counts": torch.tensor(nc), "edge_counts": torch.tensor(ec)}


def run_expand(arr, ids, ranks, variants, node_out=None, edge_out=None):
    """The expansion contract on (sample, row, threshold) variants, outputs NaN / -7 prefilled; offsets those of the
    explicit edits unless given.  -> (x, src, dst, edge_attr, flag)."""
    nc = arr["node_counts"]
    node_out = _offsets(nc[[min(max(v[0], 0), len(nc) - 1) for v in variants]]) if node_out is None else node_out
    if edge_out is None:
        fine = [v if 0 <= v[0] < len(nc) and 0 <= v[1] < ranks.numel() // ranks.shape[-1] and 0 <= v[2] <= ranks.shape[-1]
                else (0, 0, 0) for v in variants]
        edge_out = _offsets(edge_coalitions(arr, ids, ranks, fine)["edge_counts"])
    n, e = int(node_out[-1]), int(edge_out[-1])
    xo, eo = torch.full((n, 23), float("nan")), torch.full((e, 1), float("nan"))
    so, do = torch.full((e,), -7, dtype=torch.int64), torch.full((e,), -7, dtype=torch.int64)
    flag = torch.zeros(1, dtype=torch.int32)
    t = torch.tensor(variants, dtype=torch.int64).reshape(-1, 3).T.contiguous()
    shapley_edge_expand_contract(arr["x"], _offsets(nc), _offsets(arr["edge_counts"]), arr["src"], arr["dst"],
                                 arr["edge_attr"], ids.to(torch.int32), ranks, t[0], t[1], t[2], node_out, edge_out, xo,
                                 so, do, eo, flag)
    return xo, so, do, eo, int(flag)


# ---- plan -------------------------------------------------------------------------------------------------------------
def test_plan_ranks_follow_the_keys_pair_up_and_differ_from_residue_games():
    arr, ids = edge_group_case()
    seed = 0x1234_5678_9ABC_DEF0
    p, po, vo, ranks, kept, flag = run_plan(arr, ids, 6, seed)
    assert flag == 0 and p.tolist() == [5, 0, 9, 0]
    differ = 0
    for s, ps in enumerate(p.tolist()):
        assert (ranks[s, :, ps:] == -1).all()
        for u in range(3):
            key = [int(philox4x32_10((q, s, u, 3), (seed & 0xFFFFFFFF, seed >> 32))[0]) for q in range(ps)]
            want = [sum((key[o], o) < (key[q], q) for o in range(ps)) for q in range(ps)]
            assert ranks[s, 2 * u, :ps].tolist() == want
            assert ranks[s, 2 * u + 1, :ps].tolist() == [ps - 1 - w for w in want]
            assert sorted(want) == list(range(ps))
            if ps:
                differ += want != plan_ranks(seed, s, u, ps).tolist()       # the residue game's stream 2
    assert differ == 6
    assert not torch.equal(run_plan(arr, ids, 6, seed + 1)[3], ranks)
    assert torch.equal(run_plan(arr, ids, 10, seed)[3][:, :6], ranks)      # a pair's rows do not depend on T


def test_plan_kept_counts_against_brute_force():
    arr, ids = edge_group_case(1)
    p, po, vo, ranks, kept, flag = run_plan(arr, ids, 4, 11)
    assert flag == 0
    variants = chain(p, ranks, vo)
    assert torch.equal(kept, edge_coalitions(arr, ids, ranks, variants)["edge_counts"])
    assert int(kept[0]) == 1                                               # graph 0 keeps only its non-player edge
    # ids outside [0, P_b) count as never removed, as the kernel reads them
    wide = ids.clone()
    wide[4] = 7
    k2, r2, flag = torch.zeros_like(kept), torch.zeros_like(ranks), torch.zeros(1, dtype=torch.int32)
    shapley_edge_plan_contract(_offsets(arr["edge_counts"]), wide.to(torch.int32), po, vo, 11, r2, k2, flag)
    assert torch.equal(k2, kept) and int(flag) == 0


def test_plan_flags_counts_that_disagree():
    arr, ids = edge_group_case()
    p, po, vo = _tables(arr, ids, 4)
    for po_, vo_ in ((po, vo + torch.tensor([0, 1, 1, 1, 1])), (po + torch.tensor([0, 0, 0, 0, 1]), vo)):
        ranks = torch.zeros(4, 4, 9, dtype=torch.int32)
        kept = torch.zeros(int(vo_[-1]) + 8, dtype=torch.int64)
        flag = torch.zeros(1, dtype=torch.int32)
        shapley_edge_plan_contract(_offsets(arr["edge_counts"]), ids.to(torch.int32), po_, vo_, 1, ranks, kept, flag)
        assert int(flag) == 1


# ---- expand -----------------------------------------------------------------------------------------------------------
def test_expand_contract_equals_edge_mask_edits():
    arr, ids = edge_group_case(2)
    p, po, vo, ranks, kept, _ = run_plan(arr, ids, 4, 3)
    variants = chain(p, ranks, vo)
    got = run_expand(arr, ids, ranks, variants[::-1])
    ref = edge_coalitions(arr, ids, ranks, variants[::-1])
    assert got[4] == 0
    for a, k in zip(got[:4], ("x", "src", "dst", "edge_attr")):
        assert torch.equal(a, ref[k]), k
    # rows are never touched, and any coalition: S as the rank row "0 for S, 1 otherwise" with threshold 1
    sub = torch.ones(2, 9, dtype=torch.int32)
    sub[0, [1, 3]] = 0
    sub[1, [0]] = 0
    got = run_expand(arr, ids, sub, [(0, 0, 1), (2, 0, 1), (2, 1, 1), (0, 1, 0)])
    assert torch.equal(got[0][:7], arr["x"][:7]) and got[4] == 0
    keep0 = ~torch.isin(ids[:11], torch.tensor([1, 3]))
    assert torch.equal(got[1][:int(keep0.sum())], arr["src"][:11][keep0])
    e_last = int(arr["edge_counts"][0])
    assert torch.equal(got[1][-e_last:], arr["src"][:11])                  # threshold 0 removes nothing


def test_expand_flags():
    arr, ids = edge_group_case(3)
    p, po, vo, ranks, kept, _ = run_plan(arr, ids, 2, 5)
    good = [(0, 0, 2), (2, 4, 3)]
    ref = run_expand(arr, ids, ranks, good + good)
    rows = ranks.numel() // ranks.shape[-1]
    for name, bad in {"sample": (4, 0, 1), "below": (-1, 0, 1), "row": (0, rows, 1), "row_below": (0, -1, 1),
                      "threshold": (0, 0, ranks.shape[-1] + 1), "threshold_below": (0, 0, -1)}.items():
        got = run_expand(arr, ids, ranks, good + [bad] + good)
        assert got[4] == 1, name
        nodes = 7 + 40
        skipped = got[0].shape[0] - ref[0].shape[0]
        assert torch.isnan(got[0][nodes:nodes + skipped]).all(), name
        assert torch.equal(torch.cat([got[0][:nodes], got[0][nodes + skipped:]]), ref[0]), name
    wide = ids.clone()
    wide[3] = ranks.shape[-1]                                             # an edge player id past the rank row
    no = _offsets(arr["node_counts"][[0, 2]])
    eo = _offsets(edge_coalitions(arr, ids, ranks, good)["edge_counts"])
    got = run_expand(arr, wide, ranks, good, edge_out=eo)
    assert got[4] == 1 and torch.isnan(got[0][:7]).all() and torch.equal(got[0][7:], ref[0][7:47])
    got = run_expand(arr, ids, ranks, good, edge_out=eo + torch.tensor([0, 0, 1]))
    assert got[4] == 1 and torch.equal(got[0][:7], ref[0][:7]) and torch.isnan(got[0][7:]).all()
    got = run_expand(arr, ids, ranks, good, node_out=no + torch.tensor([0, 1, 1]))
    assert got[4] == 1 and torch.isnan(got[0][:8]).all() and not torch.isnan(got[0][8:]).any()


# ---- the estimator on synthetic set functions over edges ---------------------------------------------------------------
def _game(fn, p, t, seed, k=1):
    """φ, se, gap of ``fn(removed frozenset of players) -> value`` as every draw's logit of one sample whose P players
    are the P edges of a two-row graph."""
    arr = {"node_counts": torch.tensor([2]), "edge_counts": torch.tensor([p]), "src": torch.zeros(p, dtype=torch.int64),
           "dst": torch.ones(p, dtype=torch.int64)}
    ids = torch.arange(p)
    pp, po, vo, ranks, kept, _ = run_plan(arr, ids, t, seed)
    rk = ranks[0].long()
    variants = chain(pp, ranks, vo)
    assert kept.tolist() == [p - j for _, _, j in variants]
    values = [fn(frozenset(q for q in range(p) if rk[row, q] < j)) for _, row, j in variants]
    logits = torch.tensor(values, dtype=torch.float64).float()[:, None].repeat(1, k)
    base = torch.tensor([[fn(frozenset())]], dtype=torch.float64).float().repeat(1, k)
    return run_reduce(logits, base, ranks, po, vo)


def test_two_players_are_exact():
    fn = lambda s: {frozenset(): 2.0, frozenset({0}): 1.5, frozenset({1}): 0.25, frozenset({0, 1}): -1.0}[s]
    phi, se, gap, _ = _game(fn, 2, 2, 1)
    np.testing.assert_allclose(phi[0].numpy(), _exact(fn, 2), rtol=1e-6)
    assert torch.isnan(se).all()


def test_mean_converges_to_the_enumerated_values():
    phi, se, gap, _ = _game(_redundant, 5, 2 * 400, 3)
    exact = _exact(_redundant, 5)
    assert exact[0] == pytest.approx(exact[1]) and exact[0] > 0.3         # single-contact occlusion gives 0 to both
    assert (np.abs(phi[0].numpy() - exact) <= 4 * se[0].numpy() + 1e-6).all()
    assert float(phi[0, 4]) == 0.0 and float(se[0, 4]) == 0.0            # the dummy: exactly 0
    assert abs(float(gap[0, 0])) < 1e-12 and abs(float(gap[1, 0])) < 1e-12
    assert float(phi[0].sum()) == pytest.approx(_redundant(frozenset()) - _redundant(frozenset(range(5))), abs=1e-6)


# ---- arguments and the bool form -----------------------------------------------------------------------------------------
@pytest.fixture
def cpu_backend(monkeypatch):
    for name in KC.ALL:
        monkeypatch.setattr(_C, name, getattr(KC, name))
    monkeypatch.setattr(_C, "head_mc_infer", head_mc_infer_contract)
    monkeypatch.setattr(_C, "shapley_edge_plan", shapley_edge_plan_contract)
    monkeypatch.setattr(_C, "shapley_edge_expand", shapley_edge_expand_contract)
    monkeypatch.setattr(_C, "shapley_reduce", shapley_reduce_contract)
    monkeypatch.setattr(trunk, "_require_device_batch", lambda g: None)
    yield


def test_errors_before_any_kernel_call(cpu_backend, monkeypatch):
    gd = load_golden("hybrid_v2")
    model = build_model("HybridModelv2", gd)
    d = gd["dense"]
    g = graph_batch(gd["graph"])
    pair_model = _comparative(True, load_golden("comparative_v2"))
    gc = graph_batch(load_golden("comparative_v2")["graph_c"])
    launched = []
    for name in ("shapley_edge_plan", "shapley_edge_expand", "shapley_reduce", "head_mc_infer", "collate_csr",
                 "linear_tc", "vae_mid_infer"):
        monkeypatch.setattr(_C, name, lambda *a, _n=name, **k: launched.append(_n))
    n, e = g.n_nodes, g.n_edges
    assert n != e
    every = torch.arange(e) % 3

    def bad(exc, match, m=model, fn=contact_shapley, players=every, **kw):
        with pytest.raises(exc, match=match):
            fn(m, g, d["seq"], d["prop"], players, **kw)

    for wrong in (torch.ones(e, dtype=torch.int32), torch.ones(e, dtype=torch.bool), torch.ones(n), torch.zeros(n + 1,
                  dtype=torch.bool), torch.zeros(e + 1, dtype=torch.int64), [0] * e, None):
        bad(ValueError, "int64 tensor", players=wrong)
    with pytest.raises(TypeError):
        contact_shapley(model, g, d["seq"], d["prop"])                    # players is required
    bad(ValueError, "nothing to attribute", players=torch.zeros(n, dtype=torch.bool))
    bad(ValueError, "nothing to attribute", players=torch.full((e,), -1))
    for wrong in ([0, 2], [1, 1], [-2, 0]):                               # a gap in the ids, no id 0, an id below -1
        ids = torch.full((e,), -1)
        ids[:2] = torch.tensor(wrong)
        bad(ValueError, "exactly 0 .. P_b - 1", players=ids)
    ids = torch.full((e,), -1)
    first = int(gd["graph"]["edge_counts"][0])
    ids[:first] = torch.arange(first)
    ids[0] = 300
    bad(ValueError, "301 players, more than 256", players=ids)
    for t in (0, 1, 3, 2 ** 16 + 2, 4.0, True):
        bad(ValueError, "permutations", permutations=t)
    bad(ValueError, "seed", seed=-1)
    bad(ValueError, "seed", seed=2 ** 64)
    bad(ValueError, "max_graphs", max_graphs=0)
    bad(ValueError, "samples", samples=0)
    # the checks that need no device data raise before the players are read
    touched = []
    players = shapley._edge_players
    monkeypatch.setattr(shapley, "_edge_players", lambda *a: touched.append(1) or players(*a))
    for kw in (dict(eps=torch.zeros(2, 2, 32)), dict(eps=torch.zeros(2, 3, 31)), dict(permutations=3),
               dict(seed=-1), dict(max_graphs=0)):
        bad(ValueError, "eps|permutations|seed|max_graphs", **kw)
    ec = torch.arange(gc.n_edges) % 2
    for eps in (torch.zeros(2, 3, 32), (torch.zeros(2, gc.n_graphs, 32), torch.zeros(2, gc.n_graphs + 1, 32)),
                (torch.zeros(2, gc.n_graphs, 32), None)):
        with pytest.raises(ValueError, match="eps"):
            contact_shapley_pair(pair_model, (gc, gc), (d["seq"], d["seq"]), (d["prop"], d["prop"]), ec, eps=eps)
    assert not touched
    monkeypatch.setattr(shapley, "_edge_players", players)
    for name in ("StructureModel", "StructureModelv2", "SequenceModel", "DualModel"):
        bad(NotImplementedError, "HybridModelv2_SSL", m=I.model_map[name](vae_input_dim=231, device="cpu").eval())
    model.train()
    bad(RuntimeError, "eval")
    model.eval()
    with pytest.raises(NotImplementedError, match="HybridModel_Comparative"):
        contact_shapley_pair(model, (g, g), (d["seq"], d["seq"]), (d["prop"], d["prop"]), every)
    assert not launched


def test_bool_form_numbers_contacts_as_occlusion(cpu_backend):
    arr = hand_case(4)
    g = graph_batch(arr)
    with pytest.raises(ValueError, match=r"\d+ players, more than 256"):                 # graph 2 has ~400 contacts
        _edge_sizes(g, torch.ones(51, dtype=torch.bool), 4)
    mixed = torch.arange(51) < 11                                           # graphs 0 and 1, and row 0 of graph 2
    for sel in (mixed, torch.arange(51) % 10 == 0):
        (ids, count, nvar, pmax, v, q), (u, w) = _edge_sizes(g, sel, 4)
        (smp, na, nb, *_), edge_contact = occlusion._contact_tables(g, sel, 4096)
        eo = _offsets(arr["edge_counts"])
        sample = torch.repeat_interleave(torch.arange(4), arr["edge_counts"])
        po = _offsets(count)
        assert torch.equal(torch.where(edge_contact >= 0, edge_contact - po[sample], -1), ids)
        assert q == smp.numel() and torch.equal(u, na) and torch.equal(w, nb)
        assert torch.equal(count, torch.bincount(smp, minlength=4))
        selected = [c for c in _contacts_of(arr) if bool(sel[_offsets(arr["node_counts"])[c[0]] + c[1]]) or
                    bool(sel[_offsets(arr["node_counts"])[c[0]] + c[2]])]
        assert list(zip(smp.tolist(), u.tolist(), w.tolist())) == selected
        loops = arr["src"] == arr["dst"]
        assert loops.any() and (ids[loops] == -1).all()                  # a self-loop is never a player
        assert (ids[:int(eo[1])] >= 0).sum() > 0
    # explicit groups carry no endpoints
    arr2, eids = edge_group_case()
    (_, count, *_), (u, w) = _edge_sizes(graph_batch(arr2), eids, 2)
    assert count.tolist() == [5, 0, 9, 0] and (u == -1).all() and (w == -1).all() and u.numel() == 14
    with pytest.raises(ValueError, match="nothing to attribute"):
        _edge_sizes(graph_batch(arr2), torch.zeros(51, dtype=torch.bool), 2)


# ---- whole runs through the kernel contracts ------------------------------------------------------------------------
def _peptide(arr, rows=9):
    """bool [ΣN]: rows 0 .. rows-1 of every graph."""
    sel = torch.zeros(int(arr["node_counts"].sum()), dtype=torch.bool)
    off = _offsets(arr["node_counts"])
    for s in range(len(off) - 1):
        sel[off[s]:off[s] + rows] = True
    return sel


def _groups(arr):
    """Per graph: every edge touching row 0 one group, every other edge touching row 1 or 2 another, the rest kept."""
    eo = _offsets(arr["edge_counts"])
    ids = torch.full((int(eo[-1]),), -1)
    for s in range(len(eo) - 1):
        src, dst = arr["src"][eo[s]:eo[s + 1]], arr["dst"][eo[s]:eo[s + 1]]
        a = (src == 0) | (dst == 0)
        b = ~a & ((src <= 2) | (dst <= 2))
        ids[eo[s]:eo[s + 1]] = torch.where(a, 0, torch.where(b, 1, -1))
    return ids


@pytest.mark.parametrize("max_graphs,form", [(4096, "groups"), (7, "bool"), (1, "bool")])
def test_single_matches_fp64_oracle(cpu_backend, max_graphs, form):
    gd = load_golden("hybrid_v2")
    model = build_model("HybridModelv2", gd)
    d = gd["dense"]
    arr = gd["graph"]
    g = graph_batch(arr)
    eps = torch.randn(2, 3, 32, generator=torch.Generator().manual_seed(3))
    players = _groups(arr) if form == "groups" else _peptide(arr, 2)
    res = contact_shapley(model, g, d["seq"], d["prop"], players, permutations=4, seed=77, eps=eps,
                          max_graphs=max_graphs)
    ids = res.edge_player
    if form == "groups":
        assert torch.equal(ids, players) and (res.u == -1).all()
    p, po, vo, ranks, _, _ = run_plan(arr, ids, 4, 77)
    assert torch.equal(res.offsets, po) and res.seed == 77 and res.permutations == 4 and int(p.min()) >= 2
    variants = chain(p, ranks, vo)
    co = edge_coalitions(arr, ids, ranks, variants)
    samples = torch.tensor([v[0] for v in variants])
    p64 = {k: v.detach().double() for k, v in model.state_dict().items()}
    n_layers = int(gd["meta"]["gcn_layers"])
    ref = torch.stack([R.hybrid_forward(p64, _og64(co), d["seq"][samples].double(), d["prop"][samples].double(),
                                        eps[k][samples].double(), version="v2", n_layers=n_layers)[3].reshape(-1)
                       for k in range(2)], 1)
    base = torch.stack([R.hybrid_forward(p64, _og64(arr), d["seq"].double(), d["prop"].double(), eps[k].double(),
                                         version="v2", n_layers=n_layers)[3].reshape(-1) for k in range(2)], 1)
    phi, se = _oracle_phi(ref, base, ranks, po, vo)
    scale = float(ref.abs().max())
    for i, (f, s) in enumerate(((res.logit, res.logit_se), (res.prob, res.prob_se))):
        assert float((f.double() - phi[i]).abs().max()) <= 1e-4 * scale, i
        assert float((s.double() - se[i]).abs().max()) <= 1e-4 * scale, i
    assert float(res.gap_logit.abs().max()) <= 1e-9 * scale and float(res.gap_prob.abs().max()) <= 1e-9
    empty = torch.tensor([int(vo[s]) for s in range(3)])
    assert float((res.empty.logits.double() - ref[empty]).abs().max()) <= 1e-4 * scale
    assert all(q.grad is None for q in model.parameters())


@pytest.mark.parametrize("use_wt", [True, False])
def test_pair_matches_fp64_oracle_and_draws_once_per_item(cpu_backend, use_wt):
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
    res = contact_shapley_pair(model, (gc, gw), (d["seq_c"], d["seq_w"]), (d["prop_c"], d["prop_w"]),
                               _peptide(arr_c, 2), permutations=2, seed=5, samples=2, max_graphs=3)
    b = arr_c["node_counts"].numel()
    assert [tuple(c.shape) for c in calls] == [(2 * b, 32)] * (2 if use_wt else 1)
    eps_c = calls[0].reshape(2, b, 32)
    eps_w = calls[1].reshape(2, b, 32) if use_wt else torch.zeros(2, b, 32)
    ids = res.edge_player
    p, po, vo, ranks, _, _ = run_plan(arr_c, ids, 2, 5)
    variants = chain(p, ranks, vo)
    samples = torch.tensor([v[0] for v in variants])
    co = edge_coalitions(arr_c, ids, ranks, variants)
    wt = edge_coalitions(arr_w, torch.full((int(arr_w["edge_counts"].sum()),), -1), ranks, variants)   # unchanged
    p64 = {k: v.detach().double() for k, v in model.state_dict().items()}
    n_layers = int(gd["meta"]["gcn_layers"])

    def fwd(gc_, gw_, idx):
        return torch.stack([R.comparative_forward(p64, (_og64(gc_), _og64(gw_)),
                                                  (d["seq_c"][idx].double(), d["seq_w"][idx].double()),
                                                  (d["prop_c"][idx].double(), d["prop_w"][idx].double()),
                                                  (eps_c[k][idx].double(), eps_w[k][idx].double()), n_layers=n_layers,
                                                  use_wt=use_wt)[4].reshape(-1) for k in range(2)], 1)

    ref = fwd(co, wt, samples)
    base = fwd(arr_c, arr_w, torch.arange(b))
    phi, _ = _oracle_phi(ref, base, ranks, po, vo)
    scale = float(ref.abs().max())
    assert float((res.logit.double() - phi[0]).abs().max()) <= 1e-4 * scale
    assert float((res.prob.double() - phi[1]).abs().max()) <= 1e-4 * scale
    assert torch.isnan(res.logit_se).all()


def test_flag_raises_after_the_reduction(cpu_backend, monkeypatch):
    gd = load_golden("hybrid_v2")
    model = build_model("HybridModelv2", gd)
    d = gd["dense"]
    g = graph_batch(gd["graph"])

    def wrong(*a):                                                    # an expansion that reports a rejected variant
        shapley_edge_expand_contract(*a)
        a[-1].fill_(1)

    monkeypatch.setattr(_C, "shapley_edge_expand", wrong)
    with pytest.raises(RuntimeError, match="rejected"):
        contact_shapley(model, g, d["seq"], d["prop"], _peptide(gd["graph"], 2), permutations=2, max_graphs=5)


def test_plan_helper_sizes_contact_games(cpu_backend):
    """``_plan`` with the edge launch sizes the passes from the kept-edge counts of the edge plan."""
    arr, ids = edge_group_case(5)
    g = graph_batch(arr)
    plan = _plan(g, _edge_sizes(g, ids, 4)[0], 4, 9, 100, launch=lambda *a: shapley_edge_plan_contract(
        a[0].edge_off, *a[1:]))
    p, po, vo, ranks, kept, _ = run_plan(arr, ids, 4, 9)
    assert torch.equal(plan["ranks"], ranks) and torch.equal(plan["kept"], kept)
    assert plan["edge_tot"] == [int(kept[j:j + r].sum()) for j, r in plan["passes"]]


# ---- the existing Shapley kernels keep their SASS -----------------------------------------------------------------------
def test_existing_shapley_kernels_keep_their_sass(tmp_path):
    """SHA-1 of the cuobjdump -sass text of the three residue-game kernels of csrc/shapley.cu, recorded from the source
    before the contact kernels were added, with the nvcc release named in the file."""
    import json
    import os
    import shutil
    import subprocess

    from immunostruct_b200 import build
    from test_neighbors_host import ROOT, _kernel_sass, _nvcc_release
    if not os.path.exists(build.NVCC) or shutil.which(os.path.join(os.path.dirname(build.NVCC), "cuobjdump")) is None:
        pytest.skip("the CUDA toolkit is not installed")
    ref = json.load(open(os.path.join(ROOT, "tests", "golden", "shapley_sass.json")))
    if _nvcc_release() != ref["nvcc_release"]:
        pytest.skip(f"the SASS was recorded with nvcc {ref['nvcc_release']}")
    obj = str(tmp_path / "shapley.o")
    subprocess.run([build.NVCC, *build.FLAGS, "-I", build.CSRC, "-I", os.path.join(ROOT, "include"), "-c",
                    os.path.join(build.CSRC, "shapley.cu"), "-o", obj], check=True, stdout=subprocess.DEVNULL,
                   stderr=subprocess.DEVNULL)
    assert _kernel_sass(obj, ref["kernels"]) == ref["kernels"]
