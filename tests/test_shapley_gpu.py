"""Shapley values of residues on the B200: the plan and expansion kernels against their contracts bit for bit, the
reduction within one fp32 ulp, chain entries against the fused eval forward of the host-built coalition batch and the
fp64 oracle, the j = 1 entries against occlusion, ``base`` against ``predictive``, determinism and pass-size independence,
the launches and the absence of host reads between passes, the pair form, gradients and injected draws.

An entry is held to 1e-6 relative against the same graph run in another batch: where a graph sits in a batch changes two
summation orders of the eval path (tests/test_mutscan_gpu.py, DESIGN 4.4c)."""
import numpy as np
import pytest
import torch

import immunostruct_b200 as I
from immunostruct_b200 import _C, shapley
from immunostruct_b200.occlusion import occlude_residues
from immunostruct_b200.predictive import predictive, predictive_pair
from immunostruct_b200.shapley import _plan, _sizes, residue_shapley, residue_shapley_pair
from immunostruct_b200.synthetic import synthetic_dense, synthetic_graph_arrays
from oracle import reference_ops as R

from helpers import graph_batch, inject_eps, log_error
from test_occlusion_host import _offsets
from test_shapley_host import (chain, coalitions, shapley_expand_contract, shapley_plan_contract,
                               shapley_reduce_contract)
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


def _close(got, ref, tol=TOL, what="shapley"):
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
    """Records what the Shapley kernels were handed: the plan's ranks and the variants' logits."""

    def __init__(self, monkeypatch):
        self.ranks, self.logits = [], []
        plan, reduce = _C.shapley_plan, _C.shapley_reduce

        def plan_(*a):
            plan(*a)
            self.ranks.append(a[8])

        def reduce_(*a):
            self.logits.append(a[0].clone())
            reduce(*a)

        monkeypatch.setattr(_C, "shapley_plan", plan_)
        monkeypatch.setattr(_C, "shapley_reduce", reduce_)


# ---- the kernels against their contracts ------------------------------------------------------------------------------
def _device_plan(arr, players, t, seed):
    g = graph_batch(arr, DEV)
    plan = _plan(g, _sizes(g, players, t), t, seed, 4096)
    return g, plan


@pytest.mark.parametrize("b,t", [(7, 64), (512, 64)])
def test_plan_against_contract(b, t):
    arr = _arrays(b, 3, big=True) if b == 7 else synthetic_graph_arrays(b, 200, 10, seed=4, n_pad=10)
    seed = 0xDEAD_BEEF_0123_4567
    g, plan = _device_plan(arr, None, t, seed)
    if b == 7:
        assert int(arr["node_counts"][0]) == 256 and int(plan["count"].max()) > 200
    ranks = torch.full(tuple(plan["ranks"].shape), -9, dtype=torch.int32)
    kept = torch.full((plan["kept"].numel(),), -9, dtype=torch.int64)
    flag = torch.zeros(1, dtype=torch.int32)
    shapley_plan_contract(_offsets(arr["node_counts"]), _offsets(arr["edge_counts"]), arr["src"], arr["dst"],
                          plan["ids32"].cpu(), plan["poff"].cpu(), plan["voff"].cpu(), seed, ranks, kept, flag)
    assert int(flag) == 0 and int(plan["flag"]) == 0
    assert torch.equal(plan["ranks"].cpu(), ranks)
    assert torch.equal(plan["kept"].cpu(), kept)


def _expand_both(arr, plan, lo, hi, max_graphs):
    """The expansion of variants lo .. hi-1 in passes of ``max_graphs``, device and contract -> per pass outputs."""
    g = graph_batch(arr, DEV)
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
            fn = _C.shapley_expand if dev == DEV else shapley_expand_contract
            fn(t_(arr["x"]), t_(off), t_(eoff), t_(arr["src"]), t_(arr["dst"]), t_(arr["edge_attr"]), t_(plan["ids32"]),
               t_(plan["ranks"]), t_(smp[j:j + r]), t_(row[j:j + r]), t_(thr[j:j + r]), t_(no), t_(eo), xo, so, do, ea,
               flag)
            outs.append([x.cpu() for x in (xo, so, do, ea, flag)])
        for a, b_ in zip(*outs):
            assert torch.equal(_bits(a), _bits(b_))
        assert int(outs[0][4]) == 0
    return g


@pytest.mark.parametrize("b", [7, 512])
def test_expand_against_contract(b):
    arr = _arrays(b, 5, big=True) if b == 7 else synthetic_graph_arrays(b, 200, 10, seed=6, n_pad=10)
    _, plan = _device_plan(arr, None, 4 if b == 7 else 64, 17)
    v = plan["smp"].numel()
    lo, hi = (0, v) if b == 7 else (v // 2, v // 2 + 3000)         # B = 512: a run of 3 000 variants mid-batch
    assert 2 * 1024 > 4 * _C.num_sms()                              # every CTA loops over several units
    _expand_both(arr, plan, lo, hi, 1024)


def test_expand_any_coalition_and_flags():
    arr = _arrays(6, 8)
    g = graph_batch(arr, DEV)
    ids = torch.full((g.n_nodes,), -1, dtype=torch.int32)
    off = _offsets(arr["node_counts"])
    for s in range(6):
        ids[off[s]:off[s] + 12] = torch.arange(12, dtype=torch.int32) // 3           # four groups of three rows
    ranks = torch.ones(3, 4, dtype=torch.int32)
    ranks[0, [0, 2]] = 0
    ranks[1, 3] = 0
    lib = [(0, 0, 1), (3, 1, 1), (5, 2, 1), (9, 0, 1), (1, 3, 1), (2, 0, 5), (4, 2, 0)]   # entries 3, 4, 5 are bad
    t = torch.tensor(lib).T.contiguous()
    nc = arr["node_counts"]
    fine = [v if v[0] < 6 and v[1] < 3 and v[2] <= 4 else (0, 0, 0) for v in lib]
    no = _offsets(nc[[v[0] for v in fine]])
    eo = _offsets(coalitions(arr, ids.long(), ranks, fine)["edge_counts"])
    outs = []
    for dev in (DEV, "cpu"):
        xo = torch.full((int(no[-1]), 23), float("nan"), device=dev)
        so, do = (torch.full((int(eo[-1]),), -7, dtype=torch.int64, device=dev) for _ in range(2))
        ea = torch.full((int(eo[-1]), 1), float("nan"), device=dev)
        flag = torch.zeros(1, dtype=torch.int32, device=dev)
        fn = _C.shapley_expand if dev == DEV else shapley_expand_contract
        fn(*(x.to(dev) for x in (arr["x"], g.node_off, g.edge_off, arr["src"], arr["dst"], arr["edge_attr"], ids, ranks,
                                 t[0], t[1], t[2], no, eo)), xo, so, do, ea, flag)
        outs.append([x.cpu() for x in (xo, so, do, ea, flag)])
    assert int(outs[0][4]) == int(outs[1][4]) == 1
    assert all(torch.equal(_bits(a), _bits(b_)) for a, b_ in zip(*outs))
    x0 = arr["x"][:int(nc[0])].clone()
    x0[[0, 1, 2, 6, 7, 8]] = 0.0
    assert torch.equal(outs[0][0][:int(nc[0])], x0)


def _ulp(x):
    return torch.nextafter(x.abs(), torch.tensor(float("inf"))) - x.abs()


def test_reduce_within_one_ulp():
    arr = synthetic_graph_arrays(40, 60, 10, seed=9, n_pad=5)
    players = _rows(arr, range(0, 60, 3))
    players[_offsets(arr["node_counts"])[3]:_offsets(arr["node_counts"])[4]] = False     # a sample without players
    _, plan = _device_plan(arr, players, 8, 21)
    gen = torch.Generator().manual_seed(5)
    k = 5
    logits = (torch.randn(plan["smp"].numel(), k, generator=gen) * 3).to(DEV)
    base = (torch.randn(40, k, generator=gen) * 3).to(DEV)
    outs = []
    for dev in (DEV, "cpu"):
        q = plan["q"]
        phi, se = torch.full((2, q), 7.0, device=dev), torch.full((2, q), 7.0, device=dev)
        gap, flag = torch.full((2, 40), 7.0, device=dev), torch.zeros(1, dtype=torch.int32, device=dev)
        fn = _C.shapley_reduce if dev == DEV else shapley_reduce_contract
        fn(*(x.to(dev) for x in (logits, base, plan["ranks"], plan["poff"], plan["voff"])), phi, se, gap, flag)
        outs.append([x.cpu() for x in (phi, se, gap, flag)])
    (phi, se, gap, flag), (phi_r, se_r, gap_r, flag_r) = outs
    assert int(flag) == int(flag_r) == 0
    for a, r in ((phi, phi_r), (se, se_r)):
        assert ((a - r).abs() <= _ulp(r)).all()
    assert float(gap.abs().max()) < 1e-12 and gap[:, 3].tolist() == [0.0, 0.0]


# ---- entries against the fused eval forward and the fp64 oracle ---------------------------------------------------------
def _coalition_batch(c, plan, lo, hi, pad_to=None):
    """The host-built coalition graphs of variants lo .. hi-1: (device batch, sequences, properties, device samples)."""
    ranks = plan["ranks"].cpu()
    variants = list(zip(plan["smp"][lo:hi].tolist(), plan["row"][lo:hi].tolist(), plan["thr"][lo:hi].tolist()))
    if pad_to:
        variants += variants[-1:] * (pad_to - len(variants))
    arr = coalitions(c["arr"], plan["ids"].cpu(), ranks, variants)
    samples = torch.tensor([v[0] for v in variants], device=DEV)
    return graph_batch(arr, DEV), c["seq"][samples], c["prop"][samples], samples, arr


def _fused_forward(c, plan, eps_k):
    """Logits of the fused eval forward of every coalition graph on draw ``eps_k``, B at a time (the passes of
    ``max_graphs`` = B, the last padded with repeats of its last variant)."""
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
    players = _rows(c["arr"], range(7))
    cap = _Capture(monkeypatch)
    res = residue_shapley(c["model"], c["g"], c["seq"], c["prop"], players=players, permutations=4, seed=3, eps=eps,
                          max_graphs=c["b"])
    g = c["g"]
    plan = _plan(g, _sizes(g, players, 4), 4, 3, c["b"])
    assert torch.equal(cap.ranks[0], plan["ranks"]) and plan["smp"].numel() == 12 * (1 + 4 * 6)
    logits = cap.logits[0]
    for k in (0, 2):
        _close(logits[:, k], _fused_forward(c, plan, eps[k]), BATCH_TOL)
    assert torch.equal(res.empty.logits, logits[plan["voff"][:-1]])


@pytest.mark.parametrize("precision", ["fp16x2", "bf16x3"], indirect=True)
def test_entries_match_fp64_oracle(precision, monkeypatch):
    c = _case(3, 31, ragged=False)
    eps = _eps(2, 3, 33)
    players = _rows(c["arr"], (0, 7, 100))
    cap = _Capture(monkeypatch)
    res = residue_shapley(c["model"], c["g"], c["seq"], c["prop"], players=players, permutations=2, seed=8, eps=eps,
                          max_graphs=4)
    plan = _plan(c["g"], _sizes(c["g"], players, 2), 2, 8, 4)
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


def test_first_entries_match_occlusion(monkeypatch):
    c = _case(9, 15)
    eps = _eps(2, 9, 16)
    players = _rows(c["arr"], range(0, 40, 4))
    cap = _Capture(monkeypatch)
    residue_shapley(c["model"], c["g"], c["seq"], c["prop"], players=players, permutations=6, seed=4, eps=eps)
    plan = _plan(c["g"], _sizes(c["g"], players, 6), 6, 4, 4096)
    occ = occlude_residues(c["model"], c["g"], c["seq"], c["prop"], nodes=players, eps=eps)
    first = (plan["thr"] == 1).nonzero().flatten()                        # j = 1: the first-ranked row removed alone
    smp, row = plan["smp"][first], plan["row"][first]
    ranks = plan["ranks"].reshape(-1, plan["ranks"].shape[-1])
    who = (ranks[row] == 0).int().argmax(1)                               # the player of rank 0
    rows = c["g"].node_off[smp] + torch.stack([(plan["ids"][c["g"].node_off[s]:c["g"].node_off[s + 1]] == w).nonzero()[0, 0]
                                               for s, w in zip(smp.tolist(), who.tolist())])
    _close(cap.logits[0][first], occ.logits[rows], BATCH_TOL)


# ---- base, determinism, pass size, gap ----------------------------------------------------------------------------------
def test_base_seed_and_pass_size(monkeypatch):
    b = 16
    c = _case(b, 41)
    eps = _eps(2, b, 43)
    players = _rows(c["arr"], range(0, 30, 2))
    cap = _Capture(monkeypatch)
    run = lambda m, seed=11: residue_shapley(c["model"], c["g"], c["seq"], c["prop"], players=players, permutations=8,
                                             seed=seed, eps=eps, max_graphs=m)
    a, a2, other = run(4096), run(4096), run(97)
    fields = ("logit", "prob", "logit_se", "prob_se", "gap_logit", "gap_prob")
    for f in fields:
        assert torch.equal(_bits(getattr(a, f)), _bits(getattr(a2, f))), f
    assert torch.equal(cap.ranks[0], cap.ranks[2]) and torch.equal(cap.logits[0], cap.logits[1])
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


# ---- launches, host reads, gradients, argument rules -------------------------------------------------------------------
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
    players = _rows(c["arr"], range(9))
    run = lambda: residue_shapley(model, c["g"], c["seq"], c["prop"], players=players, permutations=4, seed=1, eps=eps,
                                  max_graphs=max_graphs)
    run()                                                                              # warm-up
    base, _ = _names(lambda: predictive(model, c["g"], c["seq"], c["prop"], eps=eps), monkeypatch)
    plan = _plan(c["g"], _sizes(c["g"], players, 4), 4, 1, max_graphs)
    expected = list(base) + ["is_shapley_plan"]
    for j, r in plan["passes"]:
        g_r = _coalition_batch(c, plan, j, j + r)[0]
        with torch.no_grad():
            trunk, _ = _names(lambda: model.structure_embedding(g_r, project=False), monkeypatch)
        expected += ["is_shapley_expand", "is_collate_csr"] + trunk + ["is_head_mc_infer"]
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
    model.train()
    with pytest.raises(RuntimeError, match="eval"):
        run()
    model.eval()
    # an injected sampler is honoured: one call of [K*B, latent]
    calls = []
    model.sample_eps = lambda like: calls.append(tuple(like.shape)) or torch.zeros_like(like)
    inj = residue_shapley(model, c["g"], c["seq"], c["prop"], players=players, permutations=2, seed=1, samples=3)
    del model.sample_eps
    ref = residue_shapley(model, c["g"], c["seq"], c["prop"], players=players, permutations=2, seed=1,
                          eps=torch.zeros(3, b, 32, device=DEV))
    assert calls == [(3 * b, 32)] and torch.equal(inj.logit, ref.logit)


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
    players = _rows(c["arr"], range(5))
    cap = _Capture(monkeypatch)
    res = residue_shapley_pair(c["model"], *args, players=players, permutations=2, seed=2, samples=2, max_graphs=25)
    assert calls == [2 * b] * (2 if use_wt else 1)                        # no wild-type draw without use_wt
    draws = [torch.randn(2 * b, 32, generator=torch.Generator().manual_seed(70 + i)).reshape(2, b, 32).to(DEV)
             for i in range(1, 3)]
    plan = _plan(c["g"], _sizes(c["g"], players, 2), 2, 2, 25)
    g, seq, prop, samples, _ = _coalition_batch(c, plan, 0, plan["smp"].numel())
    gw_v = graph_batch({k: v for k, v in _gathered(aw, samples.cpu()).items()}, DEV)
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
