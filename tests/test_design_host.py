"""Beam search over residue substitutions (immunostruct_b200/design.py), host logic on CPU: the contracts of the two
round kernels (is_design_expand, is_design_select) -- key packing, the slot rule against a brute-force enumeration of
each sample's neighbours, the tie and NaN rules, ``allowed`` and ``max_mutations`` -- every error raised before a kernel
call, the round sizes and pass split, and whole searches through the per-kernel contracts against the fp64 oracle and
against exhaustive enumeration.  The device kernels are checked in tests/test_design_gpu.py, which shares the contracts."""
import itertools

import pytest
import torch
import torch.nn.functional as F

import immunostruct_b200 as I
from immunostruct_b200 import _C, trunk
from immunostruct_b200.design import beam_search, beam_search_pair, round_slots
from immunostruct_b200.resident import scan_passes
from oracle import kernel_contracts as KC
from oracle import reference_ops as R

from conftest import load_golden, oracle_graph, rel_err
from helpers import build_model, graph_batch
from test_predictive_host import _comparative, head_mc_infer_contract

TOL = 1e-4


def pack_keys(states):
    """Keys of states [..., P]: sum_p digit_p 20^p, digit 0 at absent sites (-1)."""
    pw = 20 ** torch.arange(states.shape[-1], dtype=torch.int64, device=states.device)
    return (states.clamp_min(0) * pw).sum(-1)


def objective(mean, std, kappa):
    """fmaf(kappa, std, mean) in fp32 (kappa rounded to fp32 first): the product is exact in fp64, the sum rounds once to
    fp64 and once to fp32."""
    kappa = float(torch.tensor(float(kappa), dtype=torch.float32))
    return (kappa * std.double() + mean.double()).float()


def slots_of(n_states, n_sites, device=None):
    """(w, p, c) of the slots k = (w P + p) 20 + c of a round, int64 [n_states P 20] each."""
    k = torch.arange(n_states * n_sites * 20, device=device)
    return k // (n_sites * 20), k // 20 % n_sites, k % 20


def slot_valid(beam, native, allowed, node_index, n_states, max_mutations):
    """The slot rule, bool [Wt P 20, B]: parent valid, site present, residue allowed and new, within max_mutations of the
    native state, and canonical: no valid state l < Wt equals the new state, and none with l < w differs from it at one
    site only (slot (l, p', c') yields it first)."""
    states, _, n_mut, valid = beam[:4]
    P = states.shape[2]
    w, p, c = slots_of(n_states, P, states.device)
    st = states[:, :n_states]
    sp, nat = st[:, w, p], native[:, p]                                        # [B, S]
    ok = valid[:, w] & (node_index[:, p] >= 0) & allowed[:, p, c] & (sp != c)
    ok &= n_mut[:, w] - (sp != nat).long() + (c != nat).long() <= max_mutations
    new = st[:, w].clone()                                                     # [B, S, P]
    new[:, torch.arange(w.numel()), p] = c
    h = (new[:, :, None] != st[:, None]).sum(-1)                               # [B, S, Wt]: sites where state l differs
    lw = torch.arange(n_states, device=states.device)
    dup = valid[:, None, :n_states] & ((h == 0) | ((h == 1) & (lw[None, None] < w[None, :, None])))
    return (ok & ~dup.any(-1)).t()


def design_expand_contract(x23, node_off, node_index, seq, seq_index, seq_columns, beam, native, allowed, n_states,
                           max_mutations, slot0, x23_out, seq_out, flag):
    """Contract of is_design_expand (signature of ``_C.design_expand``): copy k of the base batch holds slot slot0 + k =
    (w, p, c); every present site q of graph b gets residue d = c if q == p and the slot is valid for b, else
    states[b, w, q]: one_hot_20(d) in the residue columns of node row node_off[b] + node_index[b, q], one_hot_V(
    seq_columns[d]) in sequence row seq_index[b, q].  flag |= 1 when the base rows of site p are not exactly one-hot or
    contradict seq_columns, or a present site's index or residue is out of range (that site is not written)."""
    states = beam[0]
    b, P = node_index.shape
    n, (L, V) = x23.shape[0], seq.shape[1:]
    r = seq_out.shape[0] // b
    ok = slot_valid(beam, native, allowed, node_index, n_states, max_mutations)[slot0:slot0 + r]      # [r, B]
    w, p, c = (t[slot0:slot0 + r] for t in slots_of(n_states, P))
    d = states[:, w].permute(1, 0, 2).clone()                                                          # [r, B, P]
    q = torch.arange(P)
    hit = (q[None, None] == p[:, None, None]) & ok[..., None]
    d = torch.where(hit, c[:, None, None].expand(r, b, P), d)
    counts = (node_off[1:] - node_off[:-1])[None, :, None]
    ni, si = node_index[None].expand(r, b, P), seq_index[None].expand(r, b, P)
    present = ni >= 0
    dc = d.clamp(0, 19)
    sc = torch.where((d >= 0) & (d < 20), seq_columns.long()[dc], -1)
    good = present & (ni < counts) & (si >= 0) & (si < L) & (sc >= 0) & (sc < V)
    xo, so = x23.repeat(r, 1).reshape(r, n, 23), seq.repeat(r, 1, 1).reshape(r, b, L, V)
    kk, bb, qq = good.nonzero(as_tuple=True)
    xo[kk, node_off[bb] + ni[kk, bb, qq], :20] = F.one_hot(d[kk, bb, qq], 20).to(xo.dtype)
    so[kk, bb, si[kk, bb, qq]] = F.one_hot(sc[kk, bb, qq], V).to(so.dtype)
    x23_out.copy_(xo.reshape(r * n, 23))
    seq_out.copy_(so.reshape(r * b, L, V))
    # the base rows of each copy's site p
    np_, sp_ = node_index[:, p].t(), seq_index[:, p].t()                                               # [r, B]
    chk = (np_ >= 0) & (np_ < counts[0, :, 0][None]) & (sp_ >= 0) & (sp_ < L)
    xr = x23[(node_off[:-1][None] + np_.clamp_min(0)).clamp_max(max(n - 1, 0)), :20]
    sr = seq[torch.arange(b)[None].expand(r, b), sp_.clamp(0, L - 1)]
    one_hot = lambda t: ((t == 1).sum(-1) == 1) & ((t != 0).sum(-1) == 1)
    rows_ok = one_hot(xr) & one_hot(sr) & (seq_columns.long()[xr.argmax(-1)] == sr.argmax(-1))
    if bool((chk & ~rows_ok).any() | (present & ~good).any()):
        flag.fill_(1)


def design_select_contract(beam, round_logits, round_mean, round_std, native, allowed, node_index, n_states,
                           max_mutations, kappa, maximize, beam_out, best):
    """Contract of is_design_select (signature of ``_C.design_select``): the pool is the first ``n_states`` beam entries
    and the round's slots; an entry is eligible when valid and its objective fmaf(kappa, std, mean) is not NaN; the next
    beam is the first W eligible entries by objective (descending with ``maximize``), ties to the smaller key, then
    invalid entries holding the native state with NaN scores.  best = the objective of entry 0."""
    states, keys, n_mut, valid, logits, mean, std, _ = beam
    b, W, P = states.shape
    w, p, c = slots_of(n_states, P)
    ok = slot_valid(beam, native, allowed, node_index, n_states, max_mutations).t()                  # [B, S]
    st = states[:, :n_states]
    new = st[:, w].clone()                                                                             # [B, S, P]
    new[:, torch.arange(w.numel()), p] = c
    sp, nat = st[:, w, p], native[:, p]
    pool_states = torch.cat([st, new], 1)
    pool_keys = torch.cat([keys[:, :n_states], keys[:, w] + (c - sp.clamp_min(0)) * 20 ** p], 1)
    pool_nmut = torch.cat([n_mut[:, :n_states], n_mut[:, w] - (sp != nat).long() + (c != nat).long()], 1)
    pool_logits = torch.cat([logits[:, :n_states], round_logits.transpose(0, 1)], 1)
    pool_mean = torch.cat([mean[:, :n_states], round_mean.t()], 1)
    pool_std = torch.cat([std[:, :n_states], round_std.t()], 1)
    pool_obj = objective(pool_mean, pool_std, kappa)
    pool_ok = torch.cat([valid[:, :n_states], ok], 1) & ~torch.isnan(pool_obj)
    nan = float("nan")
    out = [torch.empty_like(t) for t in beam_out]
    for i in range(b):
        idx = pool_ok[i].nonzero().flatten()
        idx = idx[pool_keys[i, idx].argsort(stable=True)]
        idx = idx[pool_obj[i, idx].argsort(stable=True, descending=bool(maximize))][:W]
        n = idx.numel()
        out[0][i] = native[i]
        out[0][i, :n] = pool_states[i, idx]
        out[1][i] = pack_keys(native[i])
        out[1][i, :n] = pool_keys[i, idx]
        out[2][i] = 0
        out[2][i, :n] = pool_nmut[i, idx]
        out[3][i] = False
        out[3][i, :n] = True
        for f, src in ((4, pool_logits), (5, pool_mean), (6, pool_std), (7, pool_obj)):
            out[f][i] = nan
            out[f][i, :n] = src[i, idx]
        best[i] = pool_obj[i, idx[0]] if n else nan
    for dst, src in zip(beam_out, out):
        dst.copy_(src)


def make_beam(states, valid, native, logits, mean, std):
    """A beam tuple from its states [B, W, P], valid [B, W] and scores."""
    n_mut = ((states != native[:, None]) & (native[:, None] >= 0)).sum(-1)
    obj = torch.full_like(mean, float("nan"))
    return (states, pack_keys(states), n_mut, valid, logits, mean, std, obj)


def _random_beam(seed, b=5, W=6, P=4, K=2):
    """A beam whose states differ in one or two sites (so that slots collide), the last site absent in sample 1."""
    gen = torch.Generator().manual_seed(seed)
    native = torch.randint(0, 20, (b, P), generator=gen)
    native[1, P - 1] = -1
    states = native[:, None].repeat(1, W, 1)
    for i in range(b):
        for w in range(1, W):
            q = torch.randperm(min(3, P - 1), generator=gen)[:int(torch.randint(1, 3, (1,), generator=gen))]
            states[i, w, q] = torch.randint(0, 4, (q.numel(),), generator=gen)
    for i in range(b):                                                          # distinct states: drop repeats
        seen = set()
        for w in range(W):
            t = tuple(states[i, w].tolist())
            if t in seen:
                states[i, w] = native[i]
                states[i, w, 0] = (native[i, 0] + 5 + w) % 20
            seen.add(tuple(states[i, w].tolist()))
    valid = torch.rand(b, W, generator=gen) < 0.8
    valid[:, 0] = True
    logits = torch.randn(b, W, K, generator=gen)
    mean, std = torch.rand(b, W, generator=gen), torch.rand(b, W, generator=gen) / 4
    return make_beam(states, valid, native, logits, mean, std), native


def test_key_packing():
    states = torch.tensor([[0, 0, 0], [1, 0, 0], [0, 1, 0], [19, 19, 19], [3, -1, 2]])
    assert pack_keys(states).tolist() == [0, 1, 20, 19 + 19 * 20 + 19 * 400, 3 + 2 * 400]
    top = torch.full((14,), 19)
    assert int(pack_keys(top)) == 20 ** 14 - 1 < 2 ** 63                     # P = 14 fits int64


@pytest.mark.parametrize("seed", [0, 1, 2])
@pytest.mark.parametrize("max_mutations", [1, 2, 4])
def test_slot_rule_against_enumeration(seed, max_mutations):
    """The valid slots of each sample are exactly one slot (the first in slot order) per distinct neighbour of the valid
    beam that is allowed, within max_mutations and not in the beam.  (A beam state holds native or allowed residues only,
    as every state a search reaches does: the rule relies on it.)"""
    beam, native = _random_beam(seed)
    states, _, n_mut, valid = beam[:4]
    b, W, P = states.shape
    gen = torch.Generator().manual_seed(seed + 10)
    allowed = torch.rand(b, P, 20, generator=gen) < 0.7
    allowed.scatter_(2, states.clamp_min(0).transpose(1, 2), True)          # a search's states only hold allowed residues
    ni = torch.where(native >= 0, 0, -1)
    for n_states in (1, 3, W):
        ok = slot_valid(beam, native, allowed, ni, n_states, max_mutations)
        w, p, c = slots_of(n_states, P)
        for i in range(b):
            members = {tuple(states[i, l].tolist()) for l in range(n_states) if valid[i, l]}
            expect = {}
            for l in range(n_states):
                if not valid[i, l]:
                    continue
                for q in range(P):
                    if native[i, q] < 0:
                        continue
                    for col in range(20):
                        s = list(states[i, l].tolist())
                        if s[q] == col or not allowed[i, q, col]:
                            continue
                        s[q] = col
                        dist = sum(a != n_ for a, n_ in zip(s, native[i].tolist()) if n_ >= 0)
                        if dist <= max_mutations and tuple(s) not in members:
                            expect.setdefault(tuple(s), (l * P + q) * 20 + col)
            got = ok[:, i].nonzero().flatten().tolist()
            assert sorted(got) == sorted(expect.values()), (i, n_states)
            for k in got:
                s = list(states[i, w[k]].tolist())
                s[p[k]] = int(c[k])
                assert int(n_mut[i, w[k]] - (states[i, w[k], p[k]] != native[i, p[k]]).long()
                           + (c[k] != native[i, p[k]]).long()) == sum(a != n_ for a, n_ in zip(s, native[i].tolist())
                                                                      if n_ >= 0)


def _select(beam, native, round_mean, round_std, n_states, kappa=0.0, maximize=True, allowed=None, max_mutations=None,
            round_logits=None):
    b, W, P = beam[0].shape
    K = beam[4].shape[2]
    n = n_states * P * 20
    allowed = torch.ones(b, P, 20, dtype=torch.bool) if allowed is None else allowed
    ni = torch.where(native >= 0, 0, -1)
    rl = torch.randn(n, b, K) if round_logits is None else round_logits
    out = tuple(torch.empty_like(t) for t in beam)
    best = torch.empty(b)
    design_select_contract(beam, rl, round_mean, round_std, native, allowed, ni, n_states,
                           P if max_mutations is None else max_mutations, kappa, maximize, out, best)
    return out, best, rl


def test_select_order_ties_nan_and_empty_entries():
    beam, native = _random_beam(3, b=2, W=4, P=2)
    n = 4 * 2 * 20
    mean = torch.rand(n, 2, generator=torch.Generator().manual_seed(4))
    std = torch.zeros(n, 2)
    mean[:, 0] = 0.5                                                             # sample 0: every entry tied
    mean[::3, 1] = float("nan")                                                  # sample 1: NaN slots are never taken
    beam = beam[:5] + (torch.where(torch.arange(2)[:, None] == 0, 0.5, beam[5]), torch.zeros(2, 4)) + beam[7:]
    for maximize in (True, False):
        out, best, _ = _select(beam, native, mean, std, 4, maximize=maximize)
        assert torch.equal(out[1], pack_keys(out[0])) and out[3].all()
        assert (out[1][0].diff() > 0).all()                                     # ties: ascending keys
        o1 = out[7][1]
        assert not torch.isnan(o1).any() and ((o1.diff() <= 0) if maximize else (o1.diff() >= 0)).all()
        assert torch.equal(best, out[7][:, 0])
    # a pool smaller than W: the native state and at most one slot; the rest is invalid and holds the native state
    allowed = torch.zeros(2, 2, 20, dtype=torch.bool)
    allowed[:, 0, 7] = True
    start = make_beam(native[:, None].repeat(1, 4, 1), torch.arange(4).expand(2, 4) == 0, native, beam[4], beam[5], beam[6])
    out, best, _ = _select(start, native, torch.rand(40, 2), torch.zeros(40, 2), 1, allowed=allowed)
    for i in range(2):
        n_valid = 1 + int(native[i, 0] != 7)
        assert int(out[3][i].sum()) == n_valid and out[3][i, :n_valid].all()
        assert torch.equal(out[0][i, n_valid:], native[i].expand(4 - n_valid, 2))
        assert torch.isnan(out[5][i, n_valid:]).all() and torch.isnan(out[4][i, n_valid:]).all()


def test_select_kappa_objective():
    beam, native = _random_beam(5, b=3, W=4, P=3)
    n = 4 * 3 * 20
    gen = torch.Generator().manual_seed(6)
    mean, std = torch.rand(n, 3, generator=gen), torch.rand(n, 3, generator=gen) / 4
    for kappa in (-1.5, 0.1, 2.0):
        out, _, _ = _select(beam, native, mean, std, 4, kappa=kappa)
        v = out[3]
        o = objective(out[5], out[6], kappa)
        assert torch.equal(out[7][v], o[v])
        for i in range(3):
            assert (o[i][v[i]].diff() <= 0).all()


@pytest.mark.parametrize("max_graphs", [3, 60, 61, 4096])
def test_round_sizes_and_pass_split(max_graphs):
    assert round_slots(9, 8, 9) == [180] + [1440] * 8
    assert round_slots(3, 1, 3) == [60] * 3
    assert sum(round_slots(9, 8, 9)) * 8 == 93_600                            # DESIGN 4.4e: 8 templates, P = W = T = 9 / 8 / 9
    b = 3
    for n in (60, 240):
        passes = scan_passes(n, b, max_graphs)
        per = max_graphs // b
        assert [j for j, _ in passes] == list(range(0, n, per)) and sum(r for _, r in passes) == n
        assert all(1 <= r <= per for _, r in passes)


# ---- whole searches through the kernel contracts ----------------------------------------------------------------------
@pytest.fixture
def cpu_backend(monkeypatch):
    for name in KC.ALL:
        monkeypatch.setattr(_C, name, getattr(KC, name))
    monkeypatch.setattr(_C, "head_mc_infer", head_mc_infer_contract)
    monkeypatch.setattr(_C, "design_expand", design_expand_contract)
    monkeypatch.setattr(_C, "design_select", design_select_contract)
    monkeypatch.setattr(trunk, "_require_device_batch", lambda g: None)
    yield


def _sites(graph_arrays, seq, n_sites=2):
    """Sites on node rows 0, 3 (and 5) of each graph, at sequence rows 2, 6 (and 8), the second absent for sample 1; the
    sequence rows at the sites carry the residue's column under the reversed alphabet map."""
    cols = torch.arange(20).flip(0)
    counts = graph_arrays["node_counts"]
    off = torch.cat([torch.zeros(1, dtype=torch.int64), counts.cumsum(0)])
    b = counts.numel()
    ni = torch.tensor([[0, 3, 5][:n_sites]] * b)
    si = torch.tensor([[2, 6, 8][:n_sites]] * b)
    ni[1, 1] = si[1, 1] = -1
    seq = seq.clone()
    for i in range(b):
        for p in range(n_sites):
            if ni[i, p] >= 0:
                seq[i, si[i, p]] = F.one_hot(cols[graph_arrays["x"][off[i] + ni[i, p], :20].argmax()], seq.shape[2]).float()
    return ni, si, cols, seq, off


def _apply(arrays, seq, off, ni, si, cols, states):
    """The host-built batch of one state per sample (states [B, P], -1 at absent sites)."""
    x, s = arrays["x"].clone(), seq.clone()
    for i in range(ni.shape[0]):
        for p in range(ni.shape[1]):
            if ni[i, p] >= 0:
                x[off[i] + ni[i, p], :20] = F.one_hot(states[i, p], 20).float()
                s[i, si[i, p]] = F.one_hot(cols[states[i, p]], s.shape[2]).float()
    return dict(arrays, x=x), s


def _og64(arrays):
    g = oracle_graph(arrays)
    return dict(g, x=g["x"].double(), edge_attr=g["edge_attr"].double())


def _native(arrays, off, ni):
    return torch.where(ni < 0, -1, arrays["x"][off[:-1, None] + ni.clamp_min(0), :20].argmax(-1))


@pytest.mark.parametrize("max_graphs", [45, 4096])
def test_search_matches_fp64_oracle_and_invariants(cpu_backend, max_graphs):
    gd = load_golden("hybrid_v2")
    model = build_model("HybridModelv2", gd)
    d = gd["dense"]
    ni, si, cols, seq, off = _sites(gd["graph"], d["seq"])
    native = _native(gd["graph"], off, ni)
    allowed = torch.zeros(2, 20, dtype=torch.bool)
    allowed[:, [1, 4, 9, 13]] = True
    eps = torch.randn(2, 3, 32, generator=torch.Generator().manual_seed(3))
    res = beam_search(model, graph_batch(gd["graph"]), seq, d["prop"], ni, si, seq_columns=cols, allowed=allowed, beam=3,
                      max_mutations=2, eps=eps, max_graphs=max_graphs)
    assert res.states.shape == (3, 3, 2) and res.logits.shape == (3, 3, 2) and res.history.shape == (3, 3)
    assert torch.equal(res.history[:, 0], objective(res.base.prob_mean, res.base.prob_std, 0.0))
    assert (res.history.diff(dim=1) >= 0).all()
    assert torch.equal(res.history[:, -1], res.objective[:, 0])
    p64 = {k: v.detach().double() for k, v in model.state_dict().items()}
    for w in range(3):
        assert res.valid[:, w].all()
        st = res.states[:, w]
        assert (st[1, 1] == -1) and (st[ni < 0] == -1).all()                   # absent sites never change
        changed = (st != native) & (ni >= 0)
        assert torch.equal(res.n_mutations[:, w], changed.sum(1)) and (res.n_mutations[:, w] <= 2).all()
        assert (allowed[torch.arange(2).expand(3, 2), st.clamp_min(0)] | ~changed).all()
        arr, s = _apply(gd["graph"], seq, off, ni, si, cols, st.clamp_min(0))
        for k in range(2):
            ref = R.hybrid_forward(p64, _og64(arr), s.double(), d["prop"].double(), eps[k].double(), version="v2",
                                   n_layers=int(gd["meta"]["gcn_layers"]))[3].reshape(-1)
            assert rel_err(res.logits[:, w, k], ref) < TOL, (w, k)
    assert torch.equal(res.objective, res.prob_mean)
    for i in range(3):                                                          # distinct states, best first
        assert len({tuple(t) for t in res.states[i].tolist()}) == 3
        assert (res.objective[i].diff() <= 0).all()
    assert all(q.grad is None for q in model.parameters())


def test_exhaustive_search_is_the_full_enumeration(cpu_backend):
    """Two sites with three allowed residues each: 9 states, fewer than W = 12, so after two rounds the beam is every
    state, ordered by objective."""
    gd = load_golden("hybrid_v2")
    model = build_model("HybridModelv2", gd)
    d = gd["dense"]
    ni, si, cols, seq, off = _sites(gd["graph"], d["seq"])
    ni[1, 1], si[1, 1] = 3, 6                                                    # every site present
    seq = _sites(gd["graph"], d["seq"])[3]
    seq[1, 6] = F.one_hot(cols[gd["graph"]["x"][off[1] + 3, :20].argmax()], 21).float()
    native = _native(gd["graph"], off, ni)
    allowed = torch.zeros(3, 2, 20, dtype=torch.bool)
    for i in range(3):
        for p in range(2):
            allowed[i, p, [int(native[i, p]), (int(native[i, p]) + 3) % 20, (int(native[i, p]) + 8) % 20]] = True
    eps = torch.randn(1, 3, 32, generator=torch.Generator().manual_seed(5))
    for maximize in (True, False):
        res = beam_search(model, graph_batch(gd["graph"]), seq, d["prop"], ni, si, seq_columns=cols, allowed=allowed,
                          beam=12, eps=eps, maximize=maximize)
        assert res.valid[:, :9].all() and not res.valid[:, 9:].any()
        for i in range(3):
            got = {tuple(t) for t in res.states[i, :9].tolist()}
            want = set(itertools.product(*(allowed[i, p].nonzero().flatten().tolist() for p in range(2))))
            assert got == want
            o = res.objective[i, :9]
            assert ((o.diff() <= 0) if maximize else (o.diff() >= 0)).all()
        assert torch.equal(res.history[:, -1], res.objective[:, 0])


@pytest.mark.parametrize("use_wt", [True, False])
def test_pair_search_matches_fp64_oracle_and_draws_once_per_item(cpu_backend, use_wt):
    gd = load_golden("comparative_v2")
    model = _comparative(use_wt, gd)
    d = gd["dense"]
    ni, si, cols, seq_c, off = _sites(gd["graph_c"], d["seq_c"])
    calls = []

    def sample_eps(like):
        calls.append(torch.randn(like.shape, generator=torch.Generator().manual_seed(20 + len(calls))))
        return calls[-1]

    model.sample_eps = sample_eps
    gc, gw = graph_batch(gd["graph_c"]), graph_batch(gd["graph_w"])
    res = beam_search_pair(model, (gc, gw), (seq_c, d["seq_w"]), (d["prop_c"], d["prop_w"]), ni, si, seq_columns=cols,
                           beam=2, rounds=2, samples=2, max_graphs=40)
    b = gd["graph_c"]["node_counts"].numel()
    assert [tuple(c.shape) for c in calls] == [(2 * b, 32)] * (2 if use_wt else 1)
    eps_c = calls[0].reshape(2, b, 32)
    eps_w = calls[1].reshape(2, b, 32) if use_wt else torch.zeros(2, b, 32)
    p64 = {k: v.detach().double() for k, v in model.state_dict().items()}
    for w in range(2):
        arr, s = _apply(gd["graph_c"], seq_c, off, ni, si, cols, res.states[:, w].clamp_min(0))
        for k in range(2):
            ref = R.comparative_forward(p64, (_og64(arr), _og64(gd["graph_w"])), (s.double(), d["seq_w"].double()),
                                        (d["prop_c"].double(), d["prop_w"].double()), (eps_c[k].double(), eps_w[k].double()),
                                        n_layers=int(gd["meta"]["gcn_layers"]), use_wt=use_wt)[4].reshape(-1)
            assert rel_err(res.logits[:, w, k], ref) < TOL, (w, k)


def test_errors_before_any_kernel_call(cpu_backend, monkeypatch):
    gd = load_golden("hybrid_v2")
    model = build_model("HybridModelv2", gd)
    d = gd["dense"]
    ni, si, cols, seq, _ = _sites(gd["graph"], d["seq"])
    g, prop = graph_batch(gd["graph"]), d["prop"]
    launched = []
    for name in ("design_expand", "design_select", "head_mc_infer", "collate_csr"):
        monkeypatch.setattr(_C, name, lambda *a, **k: launched.append(1))

    def bad(exc, match, m=model, **kw):
        args = dict(node_index=ni, seq_index=si, seq_columns=cols)
        args.update(kw)
        with pytest.raises(exc, match=match):
            beam_search(m, g, seq, prop, args.pop("node_index"), args.pop("seq_index"), **args)

    bad(ValueError, "int64", node_index=ni.int())
    bad(ValueError, "same shape", seq_index=si[:, :1])
    one_sided = si.clone()
    one_sided[0, 0] = -1
    bad(ValueError, "absent", seq_index=one_sided)
    past = ni.clone()
    past[2, 0] = 12
    bad(ValueError, "node count", node_index=past)
    bad(ValueError, "sequence length", seq_index=torch.where(si >= 0, si + 9, si))
    bad(ValueError, "seq_columns", seq_columns=cols[:19])
    bad(ValueError, "seq_columns", seq_columns=torch.zeros(20, dtype=torch.int64))
    wide = torch.zeros(3, 15, dtype=torch.int64)
    bad(ValueError, "at most 14 sites", node_index=wide, seq_index=wide)
    for beam in (0, 33, 2.0):
        bad(ValueError, "beam", beam=beam)
    for m in (0, 3, 1.5):
        bad(ValueError, "max_mutations", max_mutations=m)
    for r in (0, -1, 1.0):
        bad(ValueError, "rounds", rounds=r)
    for kappa in (float("nan"), float("inf"), "1"):
        bad(ValueError, "kappa", kappa=kappa)
    for allowed in (torch.ones(2, 20), torch.ones(2, 19, dtype=torch.bool), torch.ones(4, 2, 20, dtype=torch.bool),
                    torch.ones(20, dtype=torch.bool)):
        bad(ValueError, "allowed", allowed=allowed)
    bad(ValueError, "max_graphs", max_graphs=2)
    bad(ValueError, "samples", samples=0)
    for name in ("StructureModel", "StructureModelv2", "SequenceModel", "DualModel"):
        bad(NotImplementedError, "HybridModelv2_SSL", m=I.model_map[name](vae_input_dim=231, device="cpu").eval())
    with pytest.raises(NotImplementedError, match="HybridModel_Comparative"):
        beam_search_pair(model, (g, g), (seq, seq), (prop, prop), ni, si, seq_columns=cols)
    model.train()
    bad(RuntimeError, "eval")
    assert not launched


def test_flag_raises_after_the_rounds(cpu_backend):
    gd = load_golden("hybrid_v2")
    model = build_model("HybridModelv2", gd)
    d = gd["dense"]
    ni, si, cols, seq, _ = _sites(gd["graph"], d["seq"])
    g = graph_batch(gd["graph"])
    padded = ni.clone()
    padded[0, 1] = 11                                                           # rows 10 and 11 of each graph are padding
    with pytest.raises(ValueError, match="one-hot"):
        beam_search(model, g, seq, d["prop"], padded, si, seq_columns=cols, beam=1, rounds=1)
    with pytest.raises(ValueError, match="seq_columns"):
        beam_search(model, g, seq, d["prop"], ni, si, seq_columns=cols.roll(3), beam=1, rounds=1)
