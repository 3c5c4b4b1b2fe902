"""Beam search over residue substitutions on the B200: both round kernels (is_design_expand, is_design_select) against
their contracts bit for bit, the exhaustive search against ``score_variants`` on the full enumeration, max_mutations = 1
against ``mutational_scan``, the greedy search against a host loop over ``score_variants``, every beam member against
``score_variants`` and the fused eval forward of the host-built batch, the invariants, the launch count per round, no
host read between rounds, the draws, parameter gradients, the pair and the pass size.

A candidate's score is held to 1e-6 relative against the same state run in another batch: where a graph sits in a batch
changes two summation orders of the eval path (tests/test_mutscan_gpu.py, DESIGN 4.4c).  Where two objectives lie closer
than that, their order may differ between two such runs, and the comparisons of states allow for it."""
import itertools

import pytest
import torch

import immunostruct_b200 as I
from immunostruct_b200 import _C
from immunostruct_b200.design import beam_search, beam_search_pair, round_slots
from immunostruct_b200.mutagenesis import mutational_scan, score_variants
from immunostruct_b200.predictive import predictive, predictive_pair
from immunostruct_b200.resident import scan_passes
from immunostruct_b200.synthetic import synthetic_dense

from helpers import graph_batch, inject_eps, log_error
from test_design_host import design_expand_contract, design_select_contract, make_beam, objective, pack_keys
from test_variants_gpu import _arrays, _case, _close, _eps, _mutants
from test_variants_host import library_tables

pytestmark = pytest.mark.gpu
DEV = "cuda"
TOL = 1e-5
BATCH_TOL = 1e-6
ROWS = [0, 3, 7, 10, 1, 5, 9, 11]          # site rows (node row = sequence row) among the 12 peptide rows of _case


def _sites(b, n_sites, absent=True):
    ni = torch.tensor([ROWS[:n_sites]] * b)
    if absent:
        ni[2::5, -1] = -1
    return ni, ni.clone()


def _native(c, ni):
    off = torch.cat([torch.zeros(1, dtype=torch.int64), c["arr"]["node_counts"].cumsum(0)])
    return torch.where(ni < 0, -1, c["arr"]["x"][off[:-1, None] + ni.clamp_min(0), :20].argmax(-1))


def _search(c, ni, si, **kw):
    return beam_search(c["model"], c["g"], c["seq"], c["prop"], ni, si, seq_columns=c["cols"], **kw)


def _library(ni, si, states):
    """score_variants library of states [B, W, P] (-1 at absent sites), sample-major."""
    b, w, _ = states.shape
    return [(i, [(int(ni[i, p]), int(si[i, p]), int(states[i, j, p])) for p in range(ni.shape[1]) if ni[i, p] >= 0])
            for i in range(b) for j in range(w)]


def _gap_tol(logits):
    """The probability difference the batch position can make: 1e-6 relative of the logit (sigmoid' <= 1/4), and at
    least 1e-6 of the probability scale (an fp32 ulp of a probability near 0.5 is 3e-8)."""
    return BATCH_TOL * max(float(logits.abs().max()) / 4, 1.0)


def _sensitive(c, scale=100.0):
    """At its random initialisation the model moves the probability by less than the 1e-6 near-tie window when one
    residue changes, and a comparison of selected states would compare nothing.  Scaling the vae_fc1 columns of the
    12 peptide sequence rows (before any call) makes substitutions move it by far more."""
    with torch.no_grad():
        c["model"].vae_fc1.weight[:, :12 * c["seq"].shape[2]] *= scale
    return c


def _same(a, b):
    a, b = a.cpu(), b.cpu()
    if a.dtype.is_floating_point:
        return torch.equal(torch.isnan(a), torch.isnan(b)) and torch.equal(a.nan_to_num(0.0), b.nan_to_num(0.0))
    return torch.equal(a, b)


# ---- the kernels against their contracts ------------------------------------------------------------------------------
def _random_beam(c, ni, W, seed):
    """Distinct states near the native one (site 0 differs by w), valid at random, with ``allowed`` holding every digit."""
    gen = torch.Generator().manual_seed(seed)
    native = _native(c, ni)
    b, P = ni.shape
    states = native[:, None].repeat(1, W, 1)
    states[:, :, 0] = (native[:, :1] + torch.arange(W)) % 20
    extra = torch.randint(0, 20, (b, W, P), generator=gen)
    flip = (torch.rand(b, W, P, generator=gen) < 0.3) & (ni[:, None] >= 0)
    flip[:, :, 0] = False
    states = torch.where(flip, extra, states)
    valid = torch.rand(b, W, generator=gen) < 0.8
    valid[:, 0] = True
    allowed = torch.rand(b, P, 20, generator=gen) < 0.6
    allowed.scatter_(2, states.clamp_min(0).transpose(1, 2), True)
    K = 3
    beam = make_beam(states, valid, native, torch.randn(b, W, K, generator=gen), torch.rand(b, W, generator=gen),
                     torch.rand(b, W, generator=gen) / 4)
    return beam, native, allowed


@pytest.mark.parametrize("b", [7, 512])
def test_expand_kernel_against_contract(b):
    c = _case(b, 5, big=True)
    assert int(c["arr"]["node_counts"][0]) == 256
    ni, si = _sites(b, 4)
    W, n_states, max_mut = 8, 6, 3
    beam, native, allowed = _random_beam(c, ni, W, 6)
    dev = lambda t: t.to(DEV).contiguous()
    n_slots = n_states * 4 * 20
    r = 4096 // b if b > 7 else 37
    assert 2 * r * b > 4 * 4 * _C.num_sms() or b == 7                # many units per CTA at B = 512
    n, (L, V) = c["g"].n_nodes, c["seq"].shape[1:]
    for slot0 in sorted({0, 2 * r, n_slots - r}):                    # passes at the start, inside and at the end of a round
        xo = torch.full((r * n, 23), float("nan"), device=DEV)
        so = torch.full((r * b, L, V), float("nan"), device=DEV)
        flag = torch.zeros(1, dtype=torch.int32, device=DEV)
        _C.design_expand(c["g"].ndata["x"], c["g"].node_off, dev(ni), c["seq"], dev(si), dev(c["cols"]),
                         tuple(dev(t) for t in beam), dev(native), dev(allowed), n_states, max_mut, slot0, xo, so, flag)
        rx, rs = torch.empty(r * n, 23), torch.empty(r * b, L, V)
        rf = torch.zeros(1, dtype=torch.int32)
        off = c["g"].node_off.cpu()
        design_expand_contract(c["arr"]["x"], off, ni, c["seq_cpu"], si, c["cols"], beam, native, allowed, n_states,
                               max_mut, slot0, rx, rs, rf)
        assert int(flag) == int(rf) == 0
        assert torch.equal(xo.cpu(), rx) and torch.equal(so.cpu(), rs)
    # a site on a padded row (sample 1's graph of 200 nodes ends in 10 padded rows) raises the flag
    bad_ni = ni.clone()
    bad_ni[1, 1] = 195
    xo = torch.empty(r * n, 23, device=DEV)
    so = torch.empty(r * b, L, V, device=DEV)
    flag = torch.zeros(1, dtype=torch.int32, device=DEV)
    _C.design_expand(c["g"].ndata["x"], c["g"].node_off, dev(bad_ni), c["seq"], dev(si), dev(c["cols"]),
                     tuple(dev(t) for t in beam), dev(native), dev(allowed), n_states, max_mut, 20, xo, so, flag)
    rx, rs, rf = torch.empty(r * n, 23), torch.empty(r * b, L, V), torch.zeros(1, dtype=torch.int32)
    design_expand_contract(c["arr"]["x"], c["g"].node_off.cpu(), bad_ni, c["seq_cpu"], si, c["cols"], beam, native,
                           allowed, n_states, max_mut, 20, rx, rs, rf)
    assert int(flag) == int(rf) == 1
    assert torch.equal(xo.cpu(), rx) and torch.equal(so.cpu(), rs)


@pytest.mark.parametrize("b", [7, 512])
@pytest.mark.parametrize("maximize,kappa", [(True, 0.0), (False, 0.75)])
def test_select_kernel_against_contract(b, maximize, kappa):
    c = _case(b, 7)
    ni, si = _sites(b, 4)
    W, n_states, max_mut = 8, 8, 2
    beam, native, allowed = _random_beam(c, ni, W, 8)
    gen = torch.Generator().manual_seed(9)
    n = n_states * 4 * 20
    K = beam[4].shape[2]
    mean = (torch.rand(n, b, generator=gen) * 64).round() / 64                 # many exact ties: the key decides
    mean[torch.rand(n, b, generator=gen) < 0.05] = float("nan")
    std = torch.where(torch.rand(n, b, generator=gen) < 0.5, 0.0, torch.rand(n, b, generator=gen) / 4)
    logits = torch.randn(n, b, K, generator=gen)
    outs = []
    for device in (DEV, "cpu"):
        d = lambda t: t.to(device).contiguous()
        out = tuple(torch.empty_like(d(t)) for t in beam)
        hist = torch.full((b, 3), -1.0, device=device)
        fn = _C.design_select if device == DEV else design_select_contract
        fn(tuple(d(t) for t in beam), d(logits), d(mean), d(std), d(native), d(allowed), d(ni), n_states, max_mut, kappa,
           maximize, out, hist[:, 1])
        outs.append((out, hist))
    (got, gh), (ref, rh) = outs
    for i, (a, r_) in enumerate(zip(got, ref)):
        assert _same(a, r_), i
    assert _same(gh, rh) and (gh[:, 0] == -1).all()
    assert torch.equal(got[1].cpu(), pack_keys(got[0].cpu()))
    again = tuple(torch.empty_like(t) for t in got)
    _C.design_select(tuple(t.to(DEV) for t in beam), logits.to(DEV), mean.to(DEV), std.to(DEV), native.to(DEV),
                     allowed.to(DEV), ni.to(DEV), n_states, max_mut, kappa, maximize, again, torch.empty(b, device=DEV))
    assert all(_same(a, r_) for a, r_ in zip(again, got))                     # bit-reproducible


# ---- searches against enumeration ---------------------------------------------------------------------------------------
def _three_allowed(native):
    b, P = native.shape
    allowed = torch.zeros(b, P, 20, dtype=torch.bool)
    for off in (0, 3, 11):
        allowed.scatter_(2, ((native.clamp_min(0) + off) % 20).unsqueeze(2), True)
    return allowed


def test_exhaustive_search_is_the_enumeration():
    b = 6
    c = _case(b, 21)
    ni, si = _sites(b, 3, absent=False)
    native = _native(c, ni)
    allowed = _three_allowed(native)
    eps = _eps(2, b, 22)
    res = _search(c, ni, si, allowed=allowed, beam=32, eps=eps)                 # rounds = max_mutations = P = 3
    assert res.valid[:, :27].all() and not res.valid[:, 27:].any()
    states = res.states[:, :27].cpu()
    for i in range(b):
        want = set(itertools.product(*(allowed[i, p].nonzero().flatten().tolist() for p in range(3))))
        assert {tuple(t) for t in states[i].tolist()} == want
    ref = score_variants(c["model"], c["g"], c["seq"], c["prop"], *library_tables(_library(ni, si, states)),
                         seq_columns=c["cols"], eps=eps)
    _close(res.logits[:, :27].reshape(-1, 2), ref.logits, BATCH_TOL, "design")
    tol = _gap_tol(ref.logits)
    ro = ref.prob_mean.reshape(b, 27).cpu()
    assert float((res.prob_mean[:, :27].cpu() - ro).abs().max()) <= tol
    gap = ro[:, :-1] - ro[:, 1:]
    assert ((gap >= 0) | (gap.abs() <= 2 * tol)).all()                        # the same order but for near-ties
    assert torch.equal(res.history[:, -1], res.objective[:, 0])


def test_single_mutation_is_the_top_of_the_scan():
    b, P, W = 8, 4, 8
    c = _sensitive(_case(b, 23))
    ni, si = _sites(b, P)
    native = _native(c, ni)
    gen = torch.Generator().manual_seed(24)
    allowed = torch.rand(P, 20, generator=gen) < 0.5
    eps = _eps(2, b, 25)
    res = _search(c, ni, si, allowed=allowed, max_mutations=1, beam=W, eps=eps)
    assert res.history.shape == (b, 2)
    scan = mutational_scan(c["model"], c["g"], c["seq"], c["prop"], ni, si, seq_columns=c["cols"], eps=eps)
    tol = _gap_tol(scan.logits.nan_to_num(0.0))
    compared = 0
    for i in range(b):
        cand = {tuple(native[i].tolist()): float(scan.base.prob_mean[i])}
        for p in range(P):
            for col in range(20):
                if ni[i, p] >= 0 and allowed[p, col] and col != native[i, p]:
                    s = native[i].clone()
                    s[p] = col
                    cand[tuple(s.tolist())] = float(scan.prob_mean[i, p, col])
        order = sorted(cand, key=lambda s: -cand[s])
        got = [tuple(t) for t in res.states[i].cpu().tolist()]
        n = min(W, len(order))
        assert res.valid[i, :n].all() and not res.valid[i, n:].any()
        for j, s in enumerate(got[:n]):
            assert abs(float(res.prob_mean[i, j]) - cand[s]) <= tol
        # the selected set is the scan's top W unless the W-th and (W+1)-th lie within the tolerance
        if len(order) <= W or cand[order[W - 1]] - cand[order[W]] > 2 * tol:
            assert set(got[:n]) == set(order[:n])
            compared += 1
    log_error(f"design max_mutations=1: {compared} of {b} samples without a near-tie at the beam's edge")
    assert compared >= b // 2


def test_greedy_search_matches_a_host_loop():
    b, P = 8, 4
    c = _sensitive(_case(b, 26))
    ni, si = _sites(b, P)
    native = _native(c, ni)
    allowed = _three_allowed(native)
    eps = _eps(1, b, 27)
    res = _search(c, ni, si, allowed=allowed, beam=1, eps=eps)
    tol = 2 * _gap_tol(res.logits)                        # a top-two gap below this is a near-tie (module docstring)
    cur, tied = native.clone(), torch.zeros(b, dtype=torch.bool)
    for t in range(P):
        lib, owner = [], []
        for i in range(b):
            nb = [cur[i].clone()]
            for p in range(P):
                for col in allowed[i, p].nonzero().flatten().tolist():
                    if ni[i, p] >= 0 and col != cur[i, p]:
                        s = cur[i].clone()
                        s[p] = col
                        nb.append(s)
            lib += [(i, [(int(ni[i, p]), int(si[i, p]), int(s[p])) for p in range(P) if ni[i, p] >= 0]) for s in nb]
            owner.append(torch.stack(nb))
        sc = score_variants(c["model"], c["g"], c["seq"], c["prop"], *library_tables(lib), seq_columns=c["cols"],
                            eps=eps).prob_mean.cpu()
        at = 0
        for i in range(b):
            m = sc[at:at + owner[i].shape[0]]
            at += owner[i].shape[0]
            top = m.topk(2).values
            tied[i] |= bool(top[0] - top[1] <= tol)
            best = int(torch.argmax(m))
            if not tied[i]:
                assert abs(float(res.history[i, t + 1]) - float(m[best])) <= tol
            cur[i] = owner[i][best]
    log_error(f"design greedy: {int((~tied).sum())} of {b} samples without a near-tie")
    assert int((~tied).sum()) >= b // 2
    assert torch.equal(res.states[~tied, 0].cpu(), cur[~tied])


@pytest.fixture
def precision(request):
    prev = I.get_precision()
    I.set_precision(request.param)
    yield request.param
    I.set_precision(prev)


@pytest.mark.parametrize("precision", ["fp16x2", "bf16x3", "bf16"], indirect=True)
@pytest.mark.parametrize("name", ["HybridModel", "HybridModelv2", "HybridModel_SSL", "HybridModelv2_SSL"])
def test_members_match_score_variants_and_the_fused_forward(precision, name):
    b, W = 12, 4
    c = _case(b, 28, name)
    ni, si = _sites(b, 3)
    eps = _eps(3, b, 29)
    res = _search(c, ni, si, beam=W, rounds=2, eps=eps, max_graphs=b * 37)
    assert res.valid.all()
    lib = _library(ni, si, res.states.cpu())
    ref = score_variants(c["model"], c["g"], c["seq"], c["prop"], *library_tables(lib), seq_columns=c["cols"], eps=eps)
    _close(res.logits.reshape(-1, 3), ref.logits, BATCH_TOL, "design")
    for w in range(W):
        _, g, seq, _ = _mutants(c, _library(ni, si, res.states[:, w:w + 1].cpu()))
        for k in (0, 2):
            inject_eps(c["model"], eps[k])
            with torch.no_grad():
                fwd = c["model"](g, seq, c["prop"])[3].reshape(-1)
            _close(res.logits[:, w, k], fwd, TOL if name.endswith("_SSL") else BATCH_TOL, "design")
        del c["model"].sample_eps


@pytest.mark.parametrize("maximize,kappa", [(True, 0.0), (False, 0.0), (True, -1.25), (False, 0.6)])
def test_invariants(maximize, kappa):
    b, P, W = 16, 4, 6
    c = _case(b, 30)
    ni, si = _sites(b, P)
    native = _native(c, ni)
    allowed = torch.rand(P, 20, generator=torch.Generator().manual_seed(31)) < 0.4
    res = _search(c, ni, si, allowed=allowed, max_mutations=2, rounds=3, beam=W, maximize=maximize, kappa=kappa,
                  eps=_eps(4, b, 32))
    h = res.history.cpu()
    assert ((h.diff(dim=1) >= 0) if maximize else (h.diff(dim=1) <= 0)).all()
    assert torch.equal(res.history[:, -1], res.objective[:, 0])
    v = res.valid.cpu()
    st = res.states.cpu()
    assert v[:, 0].all()
    assert (st[ni[:, None].expand_as(st) < 0] == -1).all()                    # absent sites never change
    changed = (st != native[:, None]) & (ni[:, None] >= 0)
    assert torch.equal(res.n_mutations.cpu()[v], changed.sum(-1)[v]) and (res.n_mutations.cpu()[v] <= 2).all()
    assert (allowed[torch.arange(P).expand_as(st), st.clamp_min(0)] | ~changed)[v].all()
    obj = objective(res.prob_mean, res.prob_std, kappa)
    assert _same(res.objective, obj)                                           # fmaf(kappa, std, mean)
    o = res.objective.cpu()
    for i in range(b):
        oi = o[i][v[i]]
        assert ((oi.diff() <= 0) if maximize else (oi.diff() >= 0)).all()
        assert len({tuple(t) for t in st[i][v[i]].tolist()}) == int(v[i].sum())
    pr = torch.sigmoid(res.logits.double())
    assert float((res.prob_mean.double()[res.valid] - pr.mean(-1)[res.valid]).abs().max()) <= 1e-7
    assert float((res.prob_std.double()[res.valid] - pr.std(-1, unbiased=False)[res.valid]).abs().max()) <= 1e-7


# ---- launches, host reads, draws, gradients ------------------------------------------------------------------------------
def _launches(fn):
    before = _C.LAUNCHES
    out = fn()
    return _C.LAUNCHES - before, out


def test_launches_host_reads_draws_and_grads(monkeypatch):
    b, P, W, T, k = 16, 3, 4, 3, 2
    max_graphs = b * 25
    c = _case(b, 33)
    model = c["model"]
    ni, si = _sites(b, P)
    params = list(model.parameters())
    for i, q in enumerate(params[::3]):
        q.grad = torch.full_like(q, float(i + 1))
    before = [None if q.grad is None else q.grad.clone() for q in params]
    eps = _eps(k, b, 34)
    run = lambda **kw: _search(c, ni, si, beam=W, rounds=T, max_graphs=max_graphs, **kw)
    run(eps=eps)                                                                 # warm-up
    trunk_head, _ = _launches(lambda: predictive(model, c["g"], c["seq"], c["prop"], eps=eps))
    sizes = round_slots(P, W, T)
    plans = [scan_passes(s, b, max_graphs) for s in sizes]
    per_pass = {}
    for r in {r for plan in plans for _, r in plan}:
        g_r = c["g"].replicate(r)
        per_pass[r] = _launches(lambda: predictive(model, g_r, c["seq"].repeat(r, 1, 1), c["prop"].repeat(r, 1),
                                                   eps=eps.repeat(1, r, 1)))[0]
    assert len(per_pass) == 3 and len(plans[1]) > 1                              # several passes of three sizes
    n, res = _launches(lambda: run(eps=eps))
    rounds = sum(sum(per_pass[r] + 1 for _, r in plan) + 1 for plan in plans)   # passes x (expand + trunk + head) + select
    assert n == trunk_head + len(per_pass) + rounds, (n, trunk_head, rounds)
    # no host read from the first expansion to the last selection
    state = {"selects": 0}
    expand, select = _C.design_expand, _C.design_select

    def expand_(*a):
        torch.cuda.set_sync_debug_mode("error")
        expand(*a)

    def select_(*a):
        select(*a)
        state["selects"] += 1
        if state["selects"] == T:
            torch.cuda.set_sync_debug_mode("default")

    monkeypatch.setattr(_C, "design_expand", expand_)
    monkeypatch.setattr(_C, "design_select", select_)
    try:
        again = run(eps=eps)
    finally:
        torch.cuda.set_sync_debug_mode("default")
    assert state["selects"] == T
    monkeypatch.setattr(_C, "design_expand", expand)
    monkeypatch.setattr(_C, "design_select", select)
    assert _same(again.logits, res.logits) and torch.equal(again.states, res.states)
    calls = []
    model.sample_eps = lambda like: calls.append(tuple(like.shape)) or torch.randn_like(like)
    drawn = run(samples=k)
    assert calls == [(k * b, 32)] and drawn.logits.shape == (b, W, k)
    del model.sample_eps
    for q, b_ in zip(params, before):
        assert (q.grad is None) == (b_ is None) and (b_ is None or torch.equal(q.grad, b_))
    assert not res.logits.requires_grad


@pytest.mark.parametrize("use_wt", [True, False])
def test_pair(use_wt):
    b, W = 12, 3
    c = _case(b, 35, "HybridModelv2_Comparative", use_wt_for_downstream=use_wt)
    ni, si = _sites(b, 3)
    aw = _arrays(b, 36)
    dw = synthetic_dense(b, seed=36)
    gw, seq_w, prop_w = graph_batch(aw, DEV), dw["seq"].to(DEV), dw["prop"].to(DEV)
    args = ((c["g"], gw), (c["seq"], seq_w), (c["prop"], prop_w))
    calls = []
    c["model"].sample_eps = lambda like: calls.append(tuple(like.shape)) or torch.randn_like(like)
    res = beam_search_pair(c["model"], *args, ni, si, seq_columns=c["cols"], beam=W, rounds=2, samples=3,
                           max_graphs=b * 40)
    assert calls == [(3 * b, 32)] * (2 if use_wt else 1)                       # no wild-type draw without use_wt
    del c["model"].sample_eps
    eps = (_eps(3, b, 37), _eps(3, b, 38))
    res = beam_search_pair(c["model"], *args, ni, si, seq_columns=c["cols"], beam=W, rounds=2, eps=eps, max_graphs=b * 40)
    base = predictive_pair(c["model"], *args, eps=eps)
    assert torch.equal(res.base.logits, base.logits)
    for w in range(W):
        _, g, seq, _ = _mutants(c, _library(ni, si, res.states[:, w:w + 1].cpu()))
        ref = predictive_pair(c["model"], (g, gw), (seq, seq_w), (c["prop"], prop_w), eps=eps)
        _close(res.logits[:, w], ref.logits, BATCH_TOL, "design pair")


def test_pass_size():
    b, P, W = 32, 3, 6
    c = _case(b, 39)
    ni, si = _sites(b, P)
    eps = _eps(2, b, 40)
    runs = [_search(c, ni, si, beam=W, eps=eps, max_graphs=m) for m in (4096, b * 7, b * 13)]
    assert [len(scan_passes(s, b, m)) for s, m in ((W * P * 20, 4096), (W * P * 20, b * 7))] == [3, 52]
    tol = _gap_tol(runs[0].logits)
    for other in runs[1:]:
        assert torch.equal(other.valid, runs[0].valid)
        same = (other.states == runs[0].states).all(-1)
        # entries whose states differ were near-ties: their objectives agree to the tolerance
        assert float((other.objective - runs[0].objective)[runs[0].valid].abs().max()) <= 2 * tol
        log_error(f"design pass size: {int((~same).sum())} of {int(same.numel())} entries differ (near-ties)")
        if same.any():
            _close(other.logits[same], runs[0].logits[same], BATCH_TOL, "design")
