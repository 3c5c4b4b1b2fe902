"""Shapley values of residues (immunostruct_b200/shapley.py), host logic on CPU: the contracts of the three kernels
(is_shapley_plan: numpy uint32 Philox4x32-10 keys and a min-rank histogram; is_shapley_expand: per-variant boolean-mask
edits; is_shapley_reduce: an fp64 restatement) against brute force and the definitions, the estimator on synthetic set
functions, every error raised before a kernel call, and whole runs through the per-kernel contracts against the fp64
oracle's forward on each host-built coalition graph, single and pair.  The device kernels are checked in
tests/test_shapley_gpu.py, which shares the contracts."""
import itertools
import math

import numpy as np
import pytest
import torch
from scipy import stats

import immunostruct_b200 as I
from immunostruct_b200 import _C, shapley, trunk
from immunostruct_b200.shapley import _plan, _sizes, residue_shapley, residue_shapley_pair
from oracle import kernel_contracts as KC
from oracle import reference_ops as R

from conftest import load_golden, oracle_graph
from helpers import build_model, graph_batch
from test_coordnoise_host import philox4x32_10
from test_occlusion_host import _offsets, hand_case
from test_predictive_host import _comparative, head_mc_infer_contract


# ---- the kernels' contracts ---------------------------------------------------------------------------------------------
def plan_ranks(seed, b, u, p):
    """Rank of each of the P players of sample b in permutation 2u: order by (Philox key v0 of counter (p, b, u, 2), p)."""
    key = philox4x32_10((np.arange(p), b, u, 2), (seed & 0xFFFFFFFF, seed >> 32))[0]
    rank = np.empty(p, dtype=np.int64)
    rank[np.lexsort((np.arange(p), key))] = np.arange(p)
    return rank


def shapley_plan_contract(node_off, edge_off, src_local, dst_local, players, player_off, var_off, seed, ranks, kept,
                          flag):
    """Contract of is_shapley_plan (signature of ``_C.shapley_plan``): rank rows 2u / 2u+1 of every sample (-1 past P_b)
    and the kept-edge count of every variant, an edge being kept in coalition j of permutation t iff j <= the smaller
    rank_t of its player endpoints (P_b for a non-player endpoint).  flag |= 1 for P_b > min(256, Pmax) or a variant
    count that is not 1 + T (P_b - 1); that sample is not written."""
    b, t, pmax = ranks.shape
    no, eo, po, vo = (x.cpu().numpy() for x in (node_off, edge_off, player_off, var_off))
    src, dst, ids = src_local.cpu().numpy(), dst_local.cpu().numpy(), players.cpu().numpy().astype(np.int64)
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
        e = slice(int(eo[s]), int(eo[s + 1]))
        who = [ids[int(no[s]) + x] for x in (src[e], dst[e])]
        for u in range(t // 2):
            r0 = plan_ranks(seed, s, u, p)
            for tt, r in ((2 * u, r0), (2 * u + 1, p - 1 - r0)):
                rk[s, tt, :p] = r
                m = np.minimum(*[np.where(w >= 0, r[np.clip(w, 0, p - 1)], p) for w in who])
                suffix = np.cumsum(np.bincount(m, minlength=p + 1)[::-1])[::-1]    # suffix[j] = #{m >= j}
                kp[v0 + 1 + tt * (p - 1):v0 + 1 + (tt + 1) * (p - 1)] = suffix[1:p]
                kp[v0] = suffix[p]
    ranks.copy_(torch.from_numpy(rk))
    kept.copy_(torch.from_numpy(kp))
    if bad:
        flag.fill_(1)


def shapley_expand_contract(x23, node_off, edge_off, src_local, dst_local, edge_attr, players, ranks, sample, rank_row,
                            threshold, node_out, edge_out, x23_out, src_out, dst_out, edge_attr_out, flag):
    """Contract of is_shapley_expand (signature of ``_C.shapley_expand``): variant v is base graph s = sample[v] with every
    row i with players[i] >= 0 and ranks[rank_row[v], players[i]] < threshold[v] zeroed and every edge touching such a row
    dropped; rows to node_out[v]..., the kept edges in base order to edge_out[v]....  flag |= 1, and the variant is not
    written, for an index out of range, n_s > 256, a player id >= Pmax, or offsets that disagree with the counts."""
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
        ids = players[n0:n0 + nb].long()
        if not (nb <= 256 and no >= 0 and n1 - no == nb and n1 <= n_out and eo >= 0 and e1 >= eo and e1 <= e_out) \
                or bool((ids >= pmax).any()):
            bad = True
            continue
        gone = (ids >= 0) & (rk[row][ids.clamp(0, pmax - 1)].long() < j)
        src, dst = src_local[e0:e0 + eb], dst_local[e0:e0 + eb]
        keep = (~(gone[src] | gone[dst])).nonzero().flatten()
        if keep.numel() != e1 - eo:
            bad = True
            continue
        x23_out[no:n1] = torch.where(gone[:, None], 0.0, x23[n0:n0 + nb])
        src_out[eo:e1], dst_out[eo:e1] = src[keep], dst[keep]
        edge_attr_out.reshape(-1)[eo:e1] = edge_attr.reshape(-1)[e0 + keep]
    if bad:
        flag.fill_(1)


def _values(lg):
    """(v_logit, v_prob) in fp64 of logits [.., K]: the means over the draws, summed in k order."""
    x = lg.astype(np.float64)
    return x.sum(-1) / x.shape[-1], (1.0 / (1.0 + np.exp(-x))).sum(-1) / x.shape[-1]


def shapley_reduce_contract(logits, base_logits, ranks, player_off, var_off, phi, se, gap, flag):
    """Contract of is_shapley_reduce (signature of ``_C.shapley_reduce``), in fp64 rounded to fp32."""
    b, t, pmax = ranks.shape
    lg, bl, rk = (x.cpu().numpy() for x in (logits, base_logits, ranks))
    po, vo = player_off.cpu().numpy(), var_off.cpu().numpy()
    ph, sd, gp = phi.cpu().numpy(), se.cpu().numpy(), gap.cpu().numpy()
    vl, vp = _values(lg) if lg.shape[0] else (np.zeros(0), np.zeros(0))
    bvl, bvp = _values(bl)
    u_n = t // 2
    bad = False
    for s in range(b):
        p, q0, v0, nvar = int(po[s + 1] - po[s]), int(po[s]), int(vo[s]), int(vo[s + 1] - vo[s])
        if not (0 <= p <= min(256, pmax) and nvar == (1 + t * (p - 1) if p else 0) and v0 + nvar <= lg.shape[0]):
            bad = True
            continue
        if p == 0:
            gp[:, s] = 0.0
            continue
        r = rk[s, :, :p].astype(np.int64)
        if ((r < 0) | (r >= p)).any():
            bad = True
            continue
        d = np.zeros((2, u_n, p))
        for tt in range(t):
            chain = [np.concatenate([[bv[s]], v[v0 + 1 + tt * (p - 1):v0 + 1 + (tt + 1) * (p - 1)], [v[v0]]])
                     for bv, v in ((bvl, vl), (bvp, vp))]
            for i in range(2):
                d[i, tt // 2] += chain[i][r[tt]] - chain[i][r[tt] + 1]
        d *= 0.5
        f = d.sum(1) / u_n
        ph[:, q0:q0 + p] = f
        sd[:, q0:q0 + p] = np.sqrt(((d - f[:, None]) ** 2).sum(1) / (u_n * (u_n - 1))) if u_n > 1 else np.nan
        gp[:, s] = (np.array([bvl[s] - vl[v0], bvp[s] - vp[v0]])) - f.sum(1)
    phi.copy_(torch.from_numpy(ph))
    se.copy_(torch.from_numpy(sd))
    gap.copy_(torch.from_numpy(gp))
    if bad:
        flag.fill_(1)


# ---- helpers ----------------------------------------------------------------------------------------------------------
def group_case(seed=0):
    """hand_case's four graphs with players: graph 0 groups rows {0, 1} -> 0, 2 -> 1, 4 -> 2, 6 -> 3 (rows 3 and the
    absent 5 never removed); graph 1 has no players; graph 2 puts its 40 rows into 7 groups, every fifth row a
    non-player; graph 3 has one player."""
    arr = hand_case(seed)
    ids = torch.full((51,), -1, dtype=torch.int64)
    ids[:7] = torch.tensor([0, 0, 1, -1, 2, -1, 3])
    g2 = torch.arange(40) % 7
    g2[::5] = -1
    ids[10:50] = g2
    ids[50] = 0
    return arr, ids


def _tables(arr, ids, t):
    """Counts, offsets and variant tables of the contract plan -> (P [B], player_off, var_off)."""
    no = _offsets(arr["node_counts"])
    p = torch.tensor([int(ids[no[s]:no[s + 1]].max()) + 1 for s in range(len(no) - 1)]).clamp_min(0)
    nvar = torch.where(p > 0, 1 + t * (p - 1), 0)
    return p, _offsets(p), _offsets(nvar)


def run_plan(arr, ids, t, seed):
    p, po, vo = _tables(arr, ids, t)
    ranks = torch.zeros(len(p), t, max(int(p.max()), 1), dtype=torch.int32)
    kept = torch.full((int(vo[-1]),), -7, dtype=torch.int64)
    flag = torch.zeros(1, dtype=torch.int32)
    shapley_plan_contract(_offsets(arr["node_counts"]), _offsets(arr["edge_counts"]), arr["src"], arr["dst"],
                          ids.to(torch.int32), po, vo, seed, ranks, kept, flag)
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


def coalitions(arr, ids, ranks, variants):
    """The variants built one by one with boolean masks: graph arrays of the coalition graphs in order."""
    off, eoff = _offsets(arr["node_counts"]), _offsets(arr["edge_counts"])
    rk = ranks.reshape(-1, ranks.shape[-1]).long()
    xs, srcs, dsts, eas, nc, ec = [], [], [], [], [], []
    for s, row, j in variants:
        local = ids[off[s]:off[s + 1]]
        gone = torch.tensor([bool(i >= 0 and rk[row, i] < j) for i in local.tolist()], dtype=torch.bool)
        x = arr["x"][off[s]:off[s + 1]].clone()
        x[gone] = 0.0
        src, dst, ea = (arr[k][eoff[s]:eoff[s + 1]] for k in ("src", "dst", "edge_attr"))
        mask = ~(gone[src] | gone[dst])
        xs.append(x)
        srcs.append(src[mask])
        dsts.append(dst[mask])
        eas.append(ea[mask])
        nc.append(x.shape[0])
        ec.append(int(mask.sum()))
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
        edge_out = _offsets(coalitions(arr, ids, ranks, fine)["edge_counts"])
    n, e = int(node_out[-1]), int(edge_out[-1])
    xo, eo = torch.full((n, 23), float("nan")), torch.full((e, 1), float("nan"))
    so, do = torch.full((e,), -7, dtype=torch.int64), torch.full((e,), -7, dtype=torch.int64)
    flag = torch.zeros(1, dtype=torch.int32)
    t = torch.tensor(variants, dtype=torch.int64).reshape(-1, 3).T.contiguous()
    shapley_expand_contract(arr["x"], _offsets(nc), _offsets(arr["edge_counts"]), arr["src"], arr["dst"], arr["edge_attr"],
                            ids.to(torch.int32), ranks, t[0], t[1], t[2], node_out, edge_out, xo, so, do, eo, flag)
    return xo, so, do, eo, int(flag)


def run_reduce(logits, base_logits, ranks, po, vo):
    q, b = int(po[-1]), base_logits.shape[0]
    phi, se, gap = torch.full((2, q), float("nan")), torch.full((2, q), float("nan")), torch.full((2, b), float("nan"))
    flag = torch.zeros(1, dtype=torch.int32)
    shapley_reduce_contract(logits, base_logits, ranks, po, vo, phi, se, gap, flag)
    return phi, se, gap, int(flag)


# ---- plan -------------------------------------------------------------------------------------------------------------
def test_plan_ranks_follow_the_keys_and_pair_up():
    arr, ids = group_case()
    seed = 0x1234_5678_9ABC_DEF0
    p, po, vo, ranks, kept, flag = run_plan(arr, ids, 6, seed)
    assert flag == 0 and p.tolist() == [4, 0, 7, 1]
    for s, ps in enumerate(p.tolist()):
        assert (ranks[s, :, ps:] == -1).all()
        for u in range(3):
            key = [int(philox4x32_10((q, s, u, 2), (seed & 0xFFFFFFFF, seed >> 32))[0]) for q in range(ps)]
            want = [sum((key[o], o) < (key[q], q) for o in range(ps)) for q in range(ps)]
            assert ranks[s, 2 * u, :ps].tolist() == want
            assert ranks[s, 2 * u + 1, :ps].tolist() == [ps - 1 - w for w in want]
            assert sorted(want) == list(range(ps))
    other = run_plan(arr, ids, 6, seed + 1)[3]
    assert not torch.equal(other, ranks)
    assert torch.equal(run_plan(arr, ids, 10, seed)[3][:, :6], ranks)      # a pair's rows do not depend on T


def test_plan_rank_distribution_is_uniform():
    arr = {"node_counts": torch.tensor([5, 5]), "edge_counts": torch.tensor([0, 0]), "src": torch.zeros(0, dtype=torch.int64),
           "dst": torch.zeros(0, dtype=torch.int64)}
    ids = torch.arange(10) % 5
    ranks = run_plan(arr, ids, 2 * 3000, 7)[3]
    perms = ranks[:, 0::2].reshape(-1, 5).tolist()
    index = {q: i for i, q in enumerate(itertools.permutations(range(5)))}
    counts = np.bincount([index[tuple(r)] for r in perms], minlength=120)
    assert stats.chisquare(counts).pvalue > 1e-4
    for q in range(5):                                                     # and the rank of each player alone
        assert stats.chisquare(np.bincount(ranks[:, 0::2, q].reshape(-1).numpy(), minlength=5)).pvalue > 1e-4


def test_plan_kept_counts_against_brute_force():
    arr, ids = group_case(1)
    e0 = torch.randperm(11, generator=torch.Generator().manual_seed(9))
    assert int(arr["edge_counts"][0]) == 11
    arr["src"][:11], arr["dst"][:11] = arr["src"][:11][e0], arr["dst"][:11][e0]
    p, po, vo, ranks, kept, flag = run_plan(arr, ids, 4, 11)
    assert flag == 0
    variants = chain(p, ranks, vo)
    assert torch.equal(kept, coalitions(arr, ids, ranks, variants)["edge_counts"])
    # the empty variant of graph 0 removes rows 0, 1, 2, 4 and 6, and every edge of graph 0 touches one of them
    assert int(kept[0]) == 0


def test_plan_flags_counts_that_disagree():
    arr, ids = group_case()
    p, po, vo = _tables(arr, ids, 4)
    for po_, vo_ in ((po, vo + torch.tensor([0, 1, 1, 1, 1])), (po + torch.tensor([0, 0, 0, 0, 1]), vo)):
        ranks = torch.zeros(4, 4, 8, dtype=torch.int32)
        kept = torch.zeros(int(vo_[-1]) + 8, dtype=torch.int64)
        flag = torch.zeros(1, dtype=torch.int32)
        shapley_plan_contract(_offsets(arr["node_counts"]), _offsets(arr["edge_counts"]), arr["src"], arr["dst"],
                              ids.to(torch.int32), po_, vo_, 1, ranks, kept, flag)
        assert int(flag) == 1


# ---- expand -----------------------------------------------------------------------------------------------------------
def test_expand_contract_equals_mask_edits():
    arr, ids = group_case(2)
    p, po, vo, ranks, kept, _ = run_plan(arr, ids, 4, 3)
    variants = chain(p, ranks, vo)
    got = run_expand(arr, ids, ranks, variants[::-1])
    ref = coalitions(arr, ids, ranks, variants[::-1])
    assert got[4] == 0
    for a, k in zip(got[:4], ("x", "src", "dst", "edge_attr")):
        assert torch.equal(a, ref[k]), k
    # any coalition: S as the rank row "0 for S, 1 otherwise" with threshold 1
    sub = torch.ones(2, 7, dtype=torch.int32)
    sub[0, [1, 3]] = 0
    sub[1, [0]] = 0
    got = run_expand(arr, ids, sub, [(0, 0, 1), (2, 0, 1), (2, 1, 1), (0, 1, 0)])
    x0 = arr["x"][:7].clone()
    x0[[2, 6]] = 0.0
    assert torch.equal(got[0][:7], x0) and got[4] == 0
    assert torch.equal(got[0][-7:], arr["x"][:7])                          # threshold 0 removes nothing


def test_expand_flags():
    arr, ids = group_case(3)
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
    wide[3] = ranks.shape[-1]                                             # a player id past the rank row
    no = _offsets(arr["node_counts"][[0, 2]])
    eo = _offsets(coalitions(arr, ids, ranks, good)["edge_counts"])
    got = run_expand(arr, wide, ranks, good, edge_out=eo)
    assert got[4] == 1 and torch.isnan(got[0][:7]).all() and torch.equal(got[0][7:], ref[0][7:47])
    got = run_expand(arr, ids, ranks, good, edge_out=eo + torch.tensor([0, 0, 1]))
    assert got[4] == 1 and torch.equal(got[0][:7], ref[0][:7]) and torch.isnan(got[0][7:]).all()
    got = run_expand(arr, ids, ranks, good, node_out=no + torch.tensor([0, 1, 1]))
    assert got[4] == 1 and torch.isnan(got[0][:8]).all() and not torch.isnan(got[0][8:]).any()


# ---- reduce -----------------------------------------------------------------------------------------------------------
def _direct(values, ranks, p, t):
    """φ and se of one sample from v(t, j) [2, T, P+1] by the definition, averaging per player over its positions."""
    u_n = t // 2
    d = np.zeros((2, u_n, p))
    for tt in range(t):
        order = np.argsort(ranks[tt, :p])                                 # order[pos] = the player at position pos
        for pos, q in enumerate(order):
            d[:, tt // 2, q] += 0.5 * (values[:, tt, pos] - values[:, tt, pos + 1])
    f = d.mean(1)
    return f, d.std(1, ddof=1) / math.sqrt(u_n) if u_n > 1 else np.full_like(f, np.nan)


def test_reduce_against_direct_restatement():
    arr, ids = group_case(4)
    t, k = 6, 3
    p, po, vo, ranks, kept, _ = run_plan(arr, ids, t, 8)
    gen = torch.Generator().manual_seed(4)
    logits = torch.randn(int(vo[-1]), k, generator=gen) * 2
    base = torch.randn(4, k, generator=gen)
    phi, se, gap, flag = run_reduce(logits, base, ranks, po, vo)
    assert flag == 0
    lv = np.stack(_values(logits.numpy()))
    bv = np.stack(_values(base.numpy()))
    for s, ps in enumerate(p.tolist()):
        if not ps:
            assert gap[:, s].tolist() == [0.0, 0.0]
            continue
        v0 = int(vo[s])
        values = np.zeros((2, t, ps + 1))
        values[:, :, 0] = bv[:, s, None]
        values[:, :, ps] = lv[:, v0, None]
        for tt in range(t):
            values[:, tt, 1:ps] = lv[:, v0 + 1 + tt * (ps - 1):v0 + 1 + (tt + 1) * (ps - 1)]
        f, e = _direct(values, ranks[s].numpy(), ps, t)
        q = slice(int(po[s]), int(po[s + 1]))
        np.testing.assert_allclose(phi[:, q].numpy(), f, rtol=1e-6, atol=1e-7)
        np.testing.assert_allclose(se[:, q].numpy(), e, rtol=1e-6, atol=1e-7)
        assert float(np.abs(gap[:, s].numpy()).max()) < 1e-12
    bad = ranks.clone()
    bad[0, 1, 0] = 9
    assert run_reduce(logits, base, bad, po, vo)[3] == 1


# ---- the estimator on synthetic set functions --------------------------------------------------------------------------
def _game(fn, p, t, seed, k=1):
    """φ, se, gap of the set function ``fn(removed frozenset) -> value`` used as every draw's logit of one sample."""
    arr = {"node_counts": torch.tensor([p]), "edge_counts": torch.tensor([0]), "src": torch.zeros(0, dtype=torch.int64),
           "dst": torch.zeros(0, dtype=torch.int64)}
    ids = torch.arange(p)
    pp, po, vo, ranks, _, _ = run_plan(arr, ids, t, seed)
    rk = ranks[0].long()
    values = [fn(frozenset(q for q in range(p) if rk[row, q] < j)) for _, row, j in chain(pp, ranks, vo)]
    logits = torch.tensor(values, dtype=torch.float64).float()[:, None].repeat(1, k)
    base = torch.tensor([[fn(frozenset())]], dtype=torch.float64).float().repeat(1, k)
    return run_reduce(logits, base, ranks, po, vo)


def _exact(fn, p):
    """Enumerated Shapley values of the value loss of removal, v(∅ removed) - v(all removed) split over the players."""
    out = np.zeros(p)
    for i in range(p):
        rest = [q for q in range(p) if q != i]
        for size in range(p):
            w = math.factorial(size) * math.factorial(p - size - 1) / math.factorial(p)
            for s in itertools.combinations(rest, size):
                out[i] += w * (fn(frozenset(s)) - fn(frozenset(s) | {i}))
    return out


def _redundant(removed):
    """Five players: 0 and 1 back each other up (a contact both make), 2 adds, 3 interacts with 2, 4 is a dummy."""
    v = 0.0 if {0, 1} <= removed else 1.5
    v += 0.0 if 2 in removed else 0.7
    v += -0.4 if {2, 3} <= removed else 0.0
    return v


def test_two_players_are_exact():
    fn = lambda s: {frozenset(): 2.0, frozenset({0}): 1.5, frozenset({1}): 0.25, frozenset({0, 1}): -1.0}[s]
    phi, se, gap, _ = _game(fn, 2, 2, 1)
    np.testing.assert_allclose(phi[0].numpy(), _exact(fn, 2), rtol=1e-6)
    assert torch.isnan(se).all()


def test_mean_converges_to_the_enumerated_values():
    phi, se, gap, _ = _game(_redundant, 5, 2 * 400, 3)
    exact = _exact(_redundant, 5)
    assert exact[0] == pytest.approx(exact[1]) and exact[0] > 0.3         # occlusion would give 0 to both
    assert (np.abs(phi[0].numpy() - exact) <= 4 * se[0].numpy() + 1e-6).all()
    assert float(phi[0, 4]) == 0.0 and float(se[0, 4]) == 0.0            # the dummy: exactly 0
    assert abs(float(phi[0, 0] - phi[0, 1])) <= 4 * math.hypot(float(se[0, 0]), float(se[0, 1]))
    assert abs(float(gap[0, 0])) < 1e-12 and abs(float(gap[1, 0])) < 1e-12
    assert float(phi[0].sum()) == pytest.approx(_redundant(frozenset()) - _redundant(frozenset(range(5))), abs=1e-6)


# ---- arguments --------------------------------------------------------------------------------------------------------
@pytest.fixture
def cpu_backend(monkeypatch):
    for name in KC.ALL:
        monkeypatch.setattr(_C, name, getattr(KC, name))
    monkeypatch.setattr(_C, "head_mc_infer", head_mc_infer_contract)
    monkeypatch.setattr(_C, "shapley_plan", shapley_plan_contract)
    monkeypatch.setattr(_C, "shapley_expand", shapley_expand_contract)
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
    for name in ("shapley_plan", "shapley_expand", "shapley_reduce", "head_mc_infer", "collate_csr", "linear_tc",
                 "vae_mid_infer"):
        monkeypatch.setattr(_C, name, lambda *a, _n=name, **k: launched.append(_n))
    n = g.n_nodes

    def bad(exc, match, m=model, fn=residue_shapley, **kw):
        with pytest.raises(exc, match=match):
            fn(m, g, d["seq"], d["prop"], **kw)

    bad(ValueError, "bool or int64", players=torch.ones(n, dtype=torch.int32))
    bad(ValueError, "bool or int64", players=torch.ones(n + 1, dtype=torch.bool))
    bad(ValueError, "bool or int64", players=[True] * n)
    bad(ValueError, "nothing to attribute", players=torch.zeros(n, dtype=torch.bool))
    bad(ValueError, "nothing to attribute", players=torch.full((n,), -1))
    for wrong in ([0, 2], [1, 1], [-2, 0]):                               # a gap in the ids, no id 0, an id below -1
        ids = torch.full((n,), -1)
        ids[:2] = torch.tensor(wrong)
        bad(ValueError, "exactly 0 .. P_b - 1", players=ids)
    ids = torch.full((n,), -1)
    ids[0] = 256
    bad(ValueError, "more than 256 players", players=ids)
    for t in (0, 1, 3, 2 ** 16 + 2, 4.0, True):
        bad(ValueError, "permutations", permutations=t)
    bad(ValueError, "seed", seed=-1)
    bad(ValueError, "seed", seed=2 ** 64)
    bad(ValueError, "max_graphs", max_graphs=0)
    bad(ValueError, "samples", samples=0)
    bad(ValueError, "eps", eps=torch.zeros(2, 2, 32))
    # the checks that need no device data raise before the players are read (no device work, no host read)
    touched = []
    players = shapley._players
    monkeypatch.setattr(shapley, "_players", lambda *a: touched.append(1) or players(*a))
    for kw in (dict(eps=torch.zeros(2, 2, 32)), dict(eps=torch.zeros(2, 3, 31)), dict(permutations=3),
               dict(seed=-1), dict(max_graphs=0)):
        bad(ValueError, "eps|permutations|seed|max_graphs", **kw)
    for eps in (torch.zeros(2, 3, 32), (torch.zeros(2, gc.n_graphs, 32), torch.zeros(2, gc.n_graphs + 1, 32)),
                (torch.zeros(2, gc.n_graphs, 32), None)):
        with pytest.raises(ValueError, match="eps"):
            residue_shapley_pair(pair_model, (gc, gc), (d["seq"], d["seq"]), (d["prop"], d["prop"]), eps=eps)
    assert not touched
    monkeypatch.setattr(shapley, "_players", players)
    for name in ("StructureModel", "StructureModelv2", "SequenceModel", "DualModel"):
        bad(NotImplementedError, "HybridModelv2_SSL", m=I.model_map[name](vae_input_dim=231, device="cpu").eval())
    model.train()
    bad(RuntimeError, "eval")
    model.eval()
    with pytest.raises(NotImplementedError, match="HybridModel_Comparative"):
        residue_shapley_pair(model, (g, g), (d["seq"], d["seq"]), (d["prop"], d["prop"]))
    assert not launched


def test_players_default_and_bool(cpu_backend):
    gd = load_golden("hybrid_v2")
    g = graph_batch(gd["graph"])
    plan = _plan(g, _sizes(g, None, 2), 2, 1, 4096)
    nc = gd["graph"]["node_counts"].tolist()
    assert nc == [12, 12, 12]
    assert plan["ids"].tolist() == sum(([*range(10), -1, -1] for _ in nc), [])     # rows 10, 11 are padded
    sel = torch.zeros(36, dtype=torch.bool)
    sel[[1, 4, 30]] = True
    plan = _plan(g, _sizes(g, sel, 4), 4, 1, 4096)
    assert plan["ids"][[1, 4, 30]].tolist() == [0, 1, 0] and plan["count"].tolist() == [2, 0, 1]
    assert plan["voff"].tolist() == [0, 5, 5, 6] and plan["q"] == 3


# ---- whole runs through the kernel contracts ------------------------------------------------------------------------
def _og64(arrays):
    g = oracle_graph(arrays)
    return dict(g, x=g["x"].double(), edge_attr=g["edge_attr"].double())


def _oracle_phi(ref_logits, base_logits, ranks, po, vo):
    """φ, gap of fp64 oracle logits through the reduce's definition, in fp64."""
    phi, se, gap = (torch.zeros(2, int(po[-1]), dtype=torch.float64), torch.zeros(2, int(po[-1]), dtype=torch.float64),
                    torch.zeros(2, base_logits.shape[0], dtype=torch.float64))
    shapley_reduce_contract(ref_logits, base_logits, ranks, po, vo, phi, se, gap, torch.zeros(1, dtype=torch.int32))
    return phi, se


def _groups(arr):
    """Per graph: rows 0..2 one group (the peptide's N-terminus), 3..5 another, rows 6 and 8 single players."""
    ids = torch.full((int(arr["node_counts"].sum()),), -1)
    off = _offsets(arr["node_counts"])
    for s in range(len(off) - 1):
        ids[off[s]:off[s] + 9] = torch.tensor([0, 0, 0, 1, 1, 1, 2, -1, 3])
    return ids


@pytest.mark.parametrize("max_graphs", [4096, 7, 1])
def test_single_matches_fp64_oracle(cpu_backend, max_graphs):
    gd = load_golden("hybrid_v2")
    model = build_model("HybridModelv2", gd)
    d = gd["dense"]
    arr = gd["graph"]
    g = graph_batch(arr)
    eps = torch.randn(2, 3, 32, generator=torch.Generator().manual_seed(3))
    ids = _groups(arr)
    res = residue_shapley(model, g, d["seq"], d["prop"], players=ids, permutations=4, seed=77, eps=eps,
                          max_graphs=max_graphs)
    p, po, vo, ranks, _, _ = run_plan(arr, ids, 4, 77)
    assert torch.equal(res.players, ids) and torch.equal(res.offsets, po) and res.seed == 77 and res.permutations == 4
    variants = chain(p, ranks, vo)
    co = coalitions(arr, ids, ranks, variants)
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
    sel = torch.zeros(int(arr_c["node_counts"].sum()), dtype=torch.bool)
    off = _offsets(arr_c["node_counts"])
    for s in range(len(off) - 1):
        sel[off[s]:off[s] + 3] = True
    res = residue_shapley_pair(model, (gc, gw), (d["seq_c"], d["seq_w"]), (d["prop_c"], d["prop_w"]), players=sel,
                               permutations=2, seed=5, samples=2, max_graphs=3)
    b = arr_c["node_counts"].numel()
    assert [tuple(c.shape) for c in calls] == [(2 * b, 32)] * (2 if use_wt else 1)
    eps_c = calls[0].reshape(2, b, 32)
    eps_w = calls[1].reshape(2, b, 32) if use_wt else torch.zeros(2, b, 32)
    ids = res.players
    p, po, vo, ranks, _, _ = run_plan(arr_c, ids, 2, 5)
    variants = chain(p, ranks, vo)
    samples = torch.tensor([v[0] for v in variants])
    co = coalitions(arr_c, ids, ranks, variants)
    wt = coalitions(arr_w, torch.full((int(arr_w["node_counts"].sum()),), -1), ranks, variants)   # unchanged
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
        shapley_expand_contract(*a)
        a[-1].fill_(1)

    monkeypatch.setattr(_C, "shapley_expand", wrong)
    with pytest.raises(RuntimeError, match="rejected"):
        residue_shapley(model, g, d["seq"], d["prop"], permutations=2, max_graphs=5)
