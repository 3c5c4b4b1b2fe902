"""Shapley values of contacts on the B200: the edge plan and edge expansion kernels against their contracts bit for bit
(self-loops, multi-edges, isolated rows, graphs without edges, P = 1 and P = 256), chain entries against the fused eval
forward of the host-built edge-masked batch and the fp64 oracle, the j = 1 entries against contact occlusion, ``base``
against ``predictive``, determinism and pass-size independence, the launches and the absence of host reads between
passes, gradients, and the pair form.

An entry is held to 1e-6 relative against the same graph run in another batch: where a graph sits in a batch changes two
summation orders of the eval path (tests/test_mutscan_gpu.py, DESIGN 4.4c)."""
import pytest
import torch

import immunostruct_b200 as I
from immunostruct_b200 import _C, shapley
from immunostruct_b200.occlusion import occlude_contacts
from immunostruct_b200.predictive import predictive, predictive_pair
from immunostruct_b200.shapley import _edge_plan, _edge_sizes, _plan, contact_shapley, contact_shapley_pair
from immunostruct_b200.synthetic import synthetic_dense, synthetic_graph_arrays
from oracle import reference_ops as R

from helpers import concat_graphs, graph_batch, inject_eps, log_error
from test_contact_shapley_host import (chain, edge_coalitions, edge_group_case, shapley_edge_expand_contract,
                                       shapley_edge_plan_contract)
from test_occlusion_host import _offsets
from test_shapley_host import shapley_reduce_contract
from test_variants_gpu import _arrays, _case, _og64

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


def _close(got, ref, tol=TOL, what="contact shapley"):
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
    return t.view(torch.int32) if t.dtype == torch.float32 else t


class _Capture:
    """Records what the kernels were handed: the edge plan's ranks and the variants' logits."""

    def __init__(self, monkeypatch):
        self.ranks, self.logits = [], []
        plan, reduce = _C.shapley_edge_plan, _C.shapley_reduce

        def plan_(*a):
            plan(*a)
            self.ranks.append(a[5])

        def reduce_(*a):
            self.logits.append(a[0].clone())
            reduce(*a)

        monkeypatch.setattr(_C, "shapley_edge_plan", plan_)
        monkeypatch.setattr(_C, "shapley_reduce", reduce_)


# ---- the kernels against their contracts ------------------------------------------------------------------------------
def _grid_case(which):
    """(graph arrays, edge players int64 [ΣE]) of the kernel grid."""
    if which == "hand":                                       # self-loops, multi-edges, an isolated row, no-edge graph
        return edge_group_case(7)
    if which == "p1_p256":                                    # graph 0: 256 players, graph 1: one, graph 2: none
        arr = concat_graphs(synthetic_graph_arrays(1, 200, 10, seed=3, n_pad=10),
                            synthetic_graph_arrays(2, 60, 10, seed=4, n_pad=5))
        e = arr["edge_counts"].tolist()
        ids = torch.full((sum(e),), -1, dtype=torch.int64)
        ids[:e[0]] = torch.arange(e[0]) % 256
        ids[e[0]:e[0] + e[1]:3] = 0
        return arr, ids
    arr = synthetic_graph_arrays(512, 200, 10, seed=5, n_pad=10)  # the peptide interface of 512 samples
    g = graph_batch(arr, DEV)
    return arr, _edge_sizes(g, _rows(arr, range(9)), 2)[0][0].cpu()


def _device_plan(arr, ids, t, seed, max_graphs=4096):
    g = graph_batch(arr, DEV)
    return g, _plan(g, _edge_sizes(g, ids, t)[0], t, seed, max_graphs, _edge_plan)


@pytest.mark.parametrize("which,t", [("hand", 2), ("hand", 64), ("p1_p256", 4), ("p1_p256", 64), ("interface", 16)])
def test_plan_against_contract(which, t):
    arr, ids = _grid_case(which)
    seed = 0xDEAD_BEEF_0123_4567
    g, plan = _device_plan(arr, ids, t, seed)
    if which == "p1_p256":
        assert plan["count"].tolist() == [256, 1, 0]
    ranks = torch.full(tuple(plan["ranks"].shape), -9, dtype=torch.int32)
    kept = torch.full((plan["kept"].numel(),), -9, dtype=torch.int64)
    flag = torch.zeros(1, dtype=torch.int32)
    shapley_edge_plan_contract(_offsets(arr["edge_counts"]), plan["ids32"].cpu(), plan["poff"].cpu(),
                               plan["voff"].cpu(), seed, ranks, kept, flag)
    assert int(flag) == 0 and int(plan["flag"]) == 0
    assert torch.equal(plan["ranks"].cpu(), ranks)
    assert torch.equal(plan["kept"].cpu(), kept)


def _expand_both(arr, plan, lo, hi, max_graphs):
    """The expansion of variants lo .. hi-1 in passes of ``max_graphs``, device against contract, bit for bit."""
    smp, row, thr, nv, kept = (plan[k][lo:hi] for k in ("smp", "row", "thr", "nv", "kept"))
    off, eoff = _offsets(arr["node_counts"]), _offsets(arr["edge_counts"])
    for j in range(0, hi - lo, max_graphs):
        r = min(max_graphs, hi - lo - j)
        no = torch.cat([torch.zeros(1, dtype=torch.int64, device=DEV), nv[j:j + r].cumsum(0)])
        eo = torch.cat([torch.zeros(1, dtype=torch.int64, device=DEV), kept[j:j + r].cumsum(0)])
        n_p, e_p = int(no[-1]), int(eo[-1])
        outs = []
        for dev in (DEV, "cpu"):
            t_ = lambda x: x.to(dev)
            xo, ea = torch.full((n_p, 23), float("nan"), device=dev), torch.full((e_p, 1), float("nan"), device=dev)
            so, do = (torch.full((e_p,), -7, dtype=torch.int64, device=dev) for _ in range(2))
            flag = torch.zeros(1, dtype=torch.int32, device=dev)
            fn = _C.shapley_edge_expand if dev == DEV else shapley_edge_expand_contract
            fn(t_(arr["x"]), t_(off), t_(eoff), t_(arr["src"]), t_(arr["dst"]), t_(arr["edge_attr"]), t_(plan["ids32"]),
               t_(plan["ranks"]), t_(smp[j:j + r]), t_(row[j:j + r]), t_(thr[j:j + r]), t_(no), t_(eo), xo, so, do, ea,
               flag)
            outs.append([x.cpu() for x in (xo, so, do, ea, flag)])
        for a, b_ in zip(*outs):
            assert torch.equal(_bits(a), _bits(b_))
        assert int(outs[0][4]) == 0


@pytest.mark.parametrize("which,t", [("hand", 4), ("p1_p256", 2), ("interface", 16)])
def test_expand_against_contract(which, t):
    arr, ids = _grid_case(which)
    _, plan = _device_plan(arr, ids, t, 17)
    v = plan["smp"].numel()
    lo, hi = (0, v) if which != "interface" else (v // 2, v // 2 + 3000)      # a run of 3 000 variants mid-batch
    assert 2 * 1024 > 4 * _C.num_sms()                                        # every CTA loops over several units
    _expand_both(arr, plan, lo, hi, 1024)


def test_expand_any_coalition_and_flags():
    arr, ids = edge_group_case(8)
    g = graph_batch(arr, DEV)
    ranks = torch.ones(3, 9, dtype=torch.int32)
    ranks[0, [0, 2]] = 0
    ranks[1, 3] = 0
    lib = [(0, 0, 1), (2, 1, 1), (2, 2, 1), (9, 0, 1), (1, 3, 1), (2, 0, 10), (0, 2, 0), (3, 0, 1)]   # 3, 4, 5 bad
    t = torch.tensor(lib).T.contiguous()
    nc = arr["node_counts"]
    fine = [v if v[0] < 4 and v[1] < 3 and v[2] <= 9 else (0, 0, 0) for v in lib]
    no = _offsets(nc[[v[0] for v in fine]])
    eo = _offsets(edge_coalitions(arr, ids, ranks, fine)["edge_counts"])
    outs = []
    for dev in (DEV, "cpu"):
        xo = torch.full((int(no[-1]), 23), float("nan"), device=dev)
        so, do = (torch.full((int(eo[-1]),), -7, dtype=torch.int64, device=dev) for _ in range(2))
        ea = torch.full((int(eo[-1]), 1), float("nan"), device=dev)
        flag = torch.zeros(1, dtype=torch.int32, device=dev)
        fn = _C.shapley_edge_expand if dev == DEV else shapley_edge_expand_contract
        fn(*(x.to(dev) for x in (arr["x"], g.node_off, g.edge_off, arr["src"], arr["dst"], arr["edge_attr"],
                                 ids.to(torch.int32), ranks, t[0], t[1], t[2], no, eo)), xo, so, do, ea, flag)
        outs.append([x.cpu() for x in (xo, so, do, ea, flag)])
    assert int(outs[0][4]) == int(outs[1][4]) == 1
    assert all(torch.equal(_bits(a), _bits(b_)) for a, b_ in zip(*outs))
    keep0 = ~torch.isin(ids[:11], torch.tensor([0, 2]))
    assert torch.equal(outs[0][1][:int(keep0.sum())], arr["src"][:11][keep0])
    # an edge player id past the rank row: that variant is not written
    wide = ids.to(torch.int32).clone()
    wide[1] = 9
    flag = torch.zeros(1, dtype=torch.int32, device=DEV)
    xo = torch.full((int(no[-1]), 23), float("nan"), device=DEV)
    _C.shapley_edge_expand(*(x.to(DEV) for x in (arr["x"], g.node_off, g.edge_off, arr["src"], arr["dst"],
                                                  arr["edge_attr"], wide, ranks, t[0], t[1], t[2], no, eo)), xo,
                           *(torch.full((int(eo[-1]),), -7, dtype=torch.int64, device=DEV) for _ in range(2)),
                           torch.zeros(int(eo[-1]), 1, device=DEV), flag)
    assert int(flag) == 1 and torch.isnan(xo[:7]).all() and not torch.isnan(xo[7:47]).any()


# ---- entries against the fused eval forward and the fp64 oracle ---------------------------------------------------------
def _coalition_batch(c, plan, lo, hi, pad_to=None):
    """The host-built edge-masked graphs of variants lo .. hi-1: (device batch, sequences, properties, device samples,
    arrays)."""
    ranks = plan["ranks"].cpu()
    variants = list(zip(plan["smp"][lo:hi].tolist(), plan["row"][lo:hi].tolist(), plan["thr"][lo:hi].tolist()))
    if pad_to:
        variants += variants[-1:] * (pad_to - len(variants))
    arr = edge_coalitions(c["arr"], plan["ids"].cpu(), ranks, variants)
    samples = torch.tensor([v[0] for v in variants], device=DEV)
    return graph_batch(arr, DEV), c["seq"][samples], c["prop"][samples], samples, arr


def _fused_forward(c, plan, eps_k):
    """Logits of the fused eval forward of every coalition graph on draw ``eps_k``, B at a time."""
    b, v, out = c["b"], plan["smp"].numel(), []
    for lo in range(0, v, b):
        hi = min(v, lo + b)
        g, seq, prop, samples, _ = _coalition_batch(c, plan, lo, hi, pad_to=b)
        inject_eps(c["model"], eps_k[samples])
        with torch.no_grad():
            out.append(c["model"](g, seq, prop)[3].reshape(-1)[:hi - lo])
    del c["model"].sample_eps
    return torch.cat(out)


@pytest.mark.parametrize("precision", ["fp16x2", "bf16x3"], indirect=True)
def test_chain_entries_match_the_fused_forward(precision, monkeypatch):
    c = _case(12, 12)
    eps = _eps(3, 12, 14)
    players = _rows(c["arr"], (3,))
    cap = _Capture(monkeypatch)
    res = contact_shapley(c["model"], c["g"], c["seq"], c["prop"], players, permutations=4, seed=3, eps=eps,
                          max_graphs=c["b"])
    g = c["g"]
    plan = _plan(g, _edge_sizes(g, players, 4)[0], 4, 3, c["b"], _edge_plan)
    assert torch.equal(cap.ranks[0], plan["ranks"]) and torch.equal(res.edge_player, plan["ids"])
    logits = cap.logits[0]
    for k in (0, 2):
        _close(logits[:, k], _fused_forward(c, plan, eps[k]), BATCH_TOL)
    assert torch.equal(res.empty.logits, logits[plan["voff"][:-1]])


@pytest.mark.parametrize("precision", ["fp16x2", "bf16x3"], indirect=True)
def test_entries_match_fp64_oracle(precision, monkeypatch):
    c = _case(3, 31, ragged=False)
    eps = _eps(2, 3, 33)
    eo = _offsets(c["arr"]["edge_counts"])
    ids = torch.full((int(eo[-1]),), -1, dtype=torch.int64)
    for s in range(3):                                            # three groups of edges per graph, some kept
        ids[eo[s]:eo[s + 1]] = torch.arange(int(eo[s + 1] - eo[s])) % 4 - 1
    cap = _Capture(monkeypatch)
    res = contact_shapley(c["model"], c["g"], c["seq"], c["prop"], ids, permutations=2, seed=8, eps=eps, max_graphs=4)
    plan = _plan(c["g"], _edge_sizes(c["g"], ids, 2)[0], 2, 8, 4, _edge_plan)
    _, seq, _, samples, arr = _coalition_batch(c, plan, 0, plan["smp"].numel())
    p64 = {k: v.detach().double().cpu() for k, v in c["model"].state_dict().items()}
    ref = torch.stack([R.hybrid_forward(p64, _og64(arr), seq.double().cpu(), c["prop"][samples].double().cpu(),
                                        eps[k][samples].double().cpu(), version="v2")[3].reshape(-1) for k in range(2)], 1)
    _close(cap.logits[0].cpu(), ref)
    base = torch.stack([R.hybrid_forward(p64, _og64(c["arr"]), c["seq"].double().cpu(), c["prop"].double().cpu(),
                                         eps[k].double().cpu(), version="v2")[3].reshape(-1) for k in range(2)], 1)
    phi, se, gap = (torch.zeros(2, 9, dtype=torch.float64), torch.zeros(2, 9, dtype=torch.float64),
                    torch.zeros(2, 3, dtype=torch.float64))
    shapley_reduce_contract(ref, base, plan["ranks"].cpu(), plan["poff"].cpu(), plan["voff"].cpu(), phi, se, gap,
                            torch.zeros(1, dtype=torch.int32))
    scale = float(ref.abs().max())
    assert float((res.logit.double().cpu() - phi[0]).abs().max()) <= 2 * TOL * scale
    assert float(res.gap_logit.abs().max()) <= 1e-9 * scale and float(res.gap_prob.abs().max()) <= 1e-9


def test_first_entries_match_contact_occlusion(monkeypatch):
    c = _case(9, 15)
    eps = _eps(2, 9, 16)
    players = _rows(c["arr"], (0, 5))
    cap = _Capture(monkeypatch)
    res = contact_shapley(c["model"], c["g"], c["seq"], c["prop"], players, permutations=6, seed=4, eps=eps)
    plan = _plan(c["g"], _edge_sizes(c["g"], players, 6)[0], 6, 4, 4096, _edge_plan)
    occ = occlude_contacts(c["model"], c["g"], c["seq"], c["prop"], nodes=players, eps=eps)
    assert torch.equal(res.u, occ.u) and torch.equal(res.v, occ.v)            # one player per contact, same order
    first = (plan["thr"] == 1).nonzero().flatten()                            # j = 1: the first-ranked contact alone
    smp, row = plan["smp"][first], plan["row"][first]
    ranks = plan["ranks"].reshape(-1, plan["ranks"].shape[-1])
    who = (ranks[row] == 0).int().argmax(1)                                   # the player of rank 0
    _close(cap.logits[0][first], occ.logits[plan["poff"][smp] + who], BATCH_TOL)


# ---- base, determinism, pass size ---------------------------------------------------------------------------------------
def test_base_seed_and_pass_size(monkeypatch):
    b = 16
    c = _case(b, 41)
    eps = _eps(2, b, 43)
    players = _rows(c["arr"], range(0, 9, 4))
    cap = _Capture(monkeypatch)
    run = lambda m, seed=11: contact_shapley(c["model"], c["g"], c["seq"], c["prop"], players, permutations=8,
                                             seed=seed, eps=eps, max_graphs=m)
    a, a2, other = run(4096), run(4096), run(97)
    for f in ("logit", "prob", "logit_se", "prob_se", "gap_logit", "gap_prob"):
        assert torch.equal(_bits(getattr(a, f)), _bits(getattr(a2, f))), f
    assert torch.equal(cap.ranks[0], cap.ranks[1]) and torch.equal(cap.ranks[0], cap.ranks[2])
    assert torch.equal(cap.logits[0], cap.logits[1])
    _close(cap.logits[2], cap.logits[0], BATCH_TOL)
    scale = float(cap.logits[0].abs().max())
    for f in ("logit", "logit_se"):
        assert float((getattr(other, f) - getattr(a, f)).abs().max()) <= 2 * BATCH_TOL * scale, f
    ref = predictive(c["model"], c["g"], c["seq"], c["prop"], eps=eps)
    for f in ("logits", "prob_mean", "prob_std"):
        assert torch.equal(getattr(a.base, f), getattr(ref, f)), f
    assert float(a.gap_logit.abs().max()) <= 1e-9 * scale and float(a.gap_prob.abs().max()) <= 1e-9
    third = run(4096, seed=12)
    assert not torch.equal(cap.ranks[-1], cap.ranks[0]) and a.seed == 11 and third.seed == 12


# ---- launches, host reads, gradients -----------------------------------------------------------------------------------
def _names(fn, monkeypatch):
    names = []
    call = _C._call
    monkeypatch.setattr(_C, "_call", lambda name, *a: names.append(name) or call(name, *a))
    out = fn()
    monkeypatch.setattr(_C, "_call", call)
    return names, out


def test_launches_no_host_read_between_passes_and_gradients(monkeypatch):
    b, max_graphs = 12, 200
    c = _case(b, 51)
    model = c["model"]
    params = list(model.parameters())
    for i, q in enumerate(params[::3]):
        q.grad = torch.full_like(q, float(i + 1))
    before = [None if q.grad is None else q.grad.clone() for q in params]
    eps = _eps(4, b, 53)
    players = _rows(c["arr"], (2, 6))
    run = lambda: contact_shapley(model, c["g"], c["seq"], c["prop"], players, permutations=4, seed=1, eps=eps,
                                  max_graphs=max_graphs)
    run()                                                                              # warm-up
    base, _ = _names(lambda: predictive(model, c["g"], c["seq"], c["prop"], eps=eps), monkeypatch)
    plan = _plan(c["g"], _edge_sizes(c["g"], players, 4)[0], 4, 1, max_graphs, _edge_plan)
    expected = list(base) + ["is_shapley_edge_plan"]
    for j, r in plan["passes"]:
        g_r = _coalition_batch(c, plan, j, j + r)[0]
        with torch.no_grad():
            trunk, _ = _names(lambda: model.structure_embedding(g_r, project=False), monkeypatch)
        expected += ["is_shapley_edge_expand", "is_collate_csr"] + trunk + ["is_head_mc_infer"]
    expected.append("is_shapley_reduce")
    assert len(plan["passes"]) >= 2
    names, res = _names(run, monkeypatch)
    assert names == expected
    assert names.count("is_vae_mid_infer") == 1                                        # the encoder ran once
    gathered = shapley.score_gathered

    def strict(*a, **k):                                                               # no host read inside the loop
        torch.cuda.synchronize()
        torch.cuda.set_sync_debug_mode("error")
        try:
            return gathered(*a, **k)
        finally:
            torch.cuda.set_sync_debug_mode("default")

    monkeypatch.setattr(shapley, "score_gathered", strict)
    strict_res = run()
    assert torch.equal(strict_res.logit, res.logit)
    for q, b_ in zip(params, before):
        assert (q.grad is None) == (b_ is None) and (b_ is None or torch.equal(q.grad, b_))
    assert not res.logit.requires_grad


@pytest.mark.parametrize("use_wt", [True, False])
def test_pair_against_forward_comparative(use_wt, monkeypatch):
    b = 8
    c = _case(b, 61, "HybridModelv2_Comparative", use_wt_for_downstream=use_wt)
    aw = _arrays(b, 62)
    dw = synthetic_dense(b, seed=62)
    gw, seq_w, prop_w = graph_batch(aw, DEV), dw["seq"].to(DEV), dw["prop"].to(DEV)
    args = ((c["g"], gw), (c["seq"], seq_w), (c["prop"], prop_w))
    calls = []
    c["model"].sample_eps = lambda like: calls.append(like.shape[0]) or torch.randn(
        like.shape, generator=torch.Generator().manual_seed(70 + len(calls))).to(like.device)
    players = _rows(c["arr"], (4,))
    cap = _Capture(monkeypatch)
    res = contact_shapley_pair(c["model"], *args, players, permutations=2, seed=2, samples=2, max_graphs=25)
    assert calls == [2 * b] * (2 if use_wt else 1)                        # no wild-type draw without use_wt
    draws = [torch.randn(2 * b, 32, generator=torch.Generator().manual_seed(70 + i)).reshape(2, b, 32).to(DEV)
             for i in range(1, 3)]
    plan = _plan(c["g"], _edge_sizes(c["g"], players, 2)[0], 2, 2, 25, _edge_plan)
    g, seq, prop, samples, _ = _coalition_batch(c, plan, 0, plan["smp"].numel())
    gw_v = graph_batch(_gathered(aw, samples.cpu()), DEV)
    for k in range(2):
        inject_eps(c["model"], draws[0][k][samples], draws[1][k][samples] if use_wt else torch.zeros(len(samples), 32))
        with torch.no_grad():
            ref = c["model"].forward_comparative((g, gw_v), (seq, seq_w[samples]), (prop, prop_w[samples]))[4].reshape(-1)
        _close(cap.logits[0][:, k], ref, BATCH_TOL)
    del c["model"].sample_eps
    ref_base = predictive_pair(c["model"], *args, eps=(draws[0], draws[1] if use_wt else None))
    assert torch.equal(res.base.logits, ref_base.logits)


def _gathered(arr, samples):
    """Graph arrays of the graphs ``samples`` of a batch, in that order (the fixed wild type of each variant)."""
    off, eoff = _offsets(arr["node_counts"]), _offsets(arr["edge_counts"])
    pick = lambda key, o: torch.cat([arr[key][o[s]:o[s + 1]] for s in samples.tolist()])
    return {"x": pick("x", off), "src": pick("src", eoff), "dst": pick("dst", eoff), "edge_attr": pick("edge_attr", eoff),
            "node_counts": arr["node_counts"][samples], "edge_counts": arr["edge_counts"][samples]}


def test_chain_is_the_variant_order():
    """The plan's (sample, row, threshold) tables list the chains as ``chain`` does."""
    arr, ids = edge_group_case(9)
    _, plan = _device_plan(arr, ids, 6, 3)
    got = list(zip(plan["smp"].tolist(), plan["row"].tolist(), plan["thr"].tolist()))
    assert got == chain(plan["count"].cpu(), plan["ranks"].cpu(), plan["voff"].cpu())
