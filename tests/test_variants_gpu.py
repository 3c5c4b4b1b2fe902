"""Variant libraries on the B200: the gather-and-substitute kernel (is_variant_expand) against its contract bit for bit,
``score_variants`` bit-identical to ``predictive`` on the identity table and to ``mutational_scan`` on the scan's own
table, every variant against the fused eval forward of the host-built mutant batch and against the fp64 oracle,
independence of the pass size, the launch count per pass, the statistics, the draws, parameter gradients and the pair.

An entry is held to 1e-6 relative against the same variant run in another batch: where a graph sits in a batch changes
two summation orders of the eval path (tests/test_mutscan_gpu.py, DESIGN 4.4c)."""
import random

import pytest
import torch

import immunostruct_b200 as I
from immunostruct_b200 import _C
from immunostruct_b200.mutagenesis import mutational_scan, score_variants, score_variants_pair
from immunostruct_b200.predictive import predictive, predictive_pair
from immunostruct_b200.resident import variant_passes
from immunostruct_b200.synthetic import split_graphs, synthetic_dense, synthetic_graph_arrays
from oracle import reference_ops as R

from helpers import concat_graphs, graph_batch, inject_eps, log_error, slice_graphs
from test_variants_host import _explicit, library_tables, run_contract

pytestmark = pytest.mark.gpu
DEV = "cuda"
TOL = 1e-5
BATCH_TOL = 1e-6          # the same variant in another batch: summation order only (module docstring)
P = 12                    # peptide rows: node rows 0..11 and sequence rows 0..11 of every sample
HLA_ROWS = range(250, 257)  # sequence rows the graphs do not hold: substituted in the sequence only


@pytest.fixture
def precision(request):
    prev = I.get_precision()
    I.set_precision(request.param)
    yield request.param
    I.set_precision(prev)


def _close(got, ref, tol=TOL, what="variants"):
    ref = ref.detach().double().cpu()
    err = float((got.detach().double().cpu() - ref).abs().max())
    lim = tol * max(float(ref.abs().max()), 1e-30)
    log_error(f"{what}: err {err:.3e} err/bound {err / lim:.3f} (tol {tol:.0e})")
    assert err <= lim, (err, float(ref.abs().max()))


def _arrays(b, seed, ragged=True, big=False):
    """b graphs in three sizes (200 nodes with 10 padded rows, 120, 60 with 5 padded rows) in blocks, the first of 256
    nodes with ``big``, or (``ragged`` False: what the fp64 oracle takes) all of 200 nodes with 10 padded rows."""
    if not ragged:
        return synthetic_graph_arrays(b, 200, 10, seed=seed, n_pad=10)
    sizes = [(200, 10), (120, 0), (60, 5)]
    parts = [synthetic_graph_arrays((b - big + 2 - i) // 3, n, 10, seed=seed + i, n_pad=pad)
             for i, (n, pad) in enumerate(sizes) if (b - big + 2 - i) // 3 > 0]
    if big:
        parts.insert(0, synthetic_graph_arrays(1, 256, 10, seed=seed + 5, n_pad=6))
    return concat_graphs(*parts)


def _case(b, seed, name="HybridModelv2", ragged=True, big=False, **kw):
    """A batch whose sequence rows 0..11 carry the residues of node rows 0..11 under a permuted ``seq_columns``."""
    arr = _arrays(b, seed, ragged, big)
    dense = synthetic_dense(b, seed=seed)
    cols = torch.randperm(21, generator=torch.Generator().manual_seed(seed))[:20]
    off = torch.cat([torch.zeros(1, dtype=torch.int64), arr["node_counts"].cumsum(0)])
    seq = dense["seq"].clone()
    rows = (off[:-1].unsqueeze(1) + torch.arange(P)).reshape(-1)
    seq[:, :P] = torch.nn.functional.one_hot(cols[arr["x"][rows, :20].argmax(1)].reshape(b, P), 21).float()
    torch.manual_seed(seed)
    model = I.model_map[name](vae_input_dim=5943, device=DEV, **kw).to(DEV).eval()
    return dict(arr=arr, g=graph_batch(arr, DEV), seq_cpu=seq, seq=seq.to(DEV), prop=dense["prop"].to(DEV), cols=cols,
                model=model, b=b)


def _library(b, n_var, seed, max_subs=9):
    """Random variants: a random sample, 0..max_subs distinct peptide rows with random residues, every fifth variant one
    more substitution in the sequence only; variant 1 carries twelve substitutions."""
    rnd = random.Random(seed)
    lib = []
    for v in range(n_var):
        rows = rnd.sample(range(P), rnd.randint(0, max_subs))
        subs = [(p, p, rnd.randrange(20)) for p in rows]
        if v % 5 == 0:
            subs.append((-1, HLA_ROWS[v % len(HLA_ROWS)], rnd.randrange(20)))
        lib.append((rnd.randrange(b), subs))
    if n_var > 1:
        lib[1] = (b - 1, [(p, p, (7 * p) % 20) for p in range(P)])
    return lib


def _eps(k, b, seed):
    return torch.randn(k, b, 32, generator=torch.Generator().manual_seed(seed)).to(DEV)


def _score(c, lib, **kw):
    return score_variants(c["model"], c["g"], c["seq"], c["prop"], *library_tables(lib), seq_columns=c["cols"], **kw)


def _mutants(c, lib, arr=None, seq=None):
    """The host-built mutant batch of a library: (graph arrays, device batch, device sequences, samples)."""
    x, src, dst, ea, s, flag = _explicit(c["arr"] if arr is None else arr, c["seq_cpu"] if seq is None else seq, c["cols"], lib)
    assert flag == 0
    samples = torch.tensor([b for b, _ in lib])
    a = c["arr"] if arr is None else arr
    out = {"x": x, "src": src, "dst": dst, "edge_attr": ea, "node_counts": a["node_counts"][samples],
           "edge_counts": a["edge_counts"][samples]}
    return out, graph_batch(out, DEV), s.to(DEV), samples.to(DEV)


# ---- the kernel against its contract ---------------------------------------------------------------------------------
def _expand(c, lib, cols=None):
    g, seq = c["g"], c["seq"]
    sample, offsets, ni, si, res = (t.to(DEV) for t in library_tables(lib))
    r, (L, V) = sample.numel(), seq.shape[1:]
    zero = torch.zeros(1, dtype=torch.int64, device=DEV)
    node_out = torch.cat([zero, g.batch_num_nodes()[sample].cumsum(0)])
    edge_out = torch.cat([zero, g.batch_num_edges()[sample].cumsum(0)])
    n, e = int(node_out[-1]), int(edge_out[-1])
    xo, eo = torch.full((n, 23), float("nan"), device=DEV), torch.full((e, 1), float("nan"), device=DEV)
    so, do = (torch.full((e,), -7, dtype=torch.int64, device=DEV) for _ in range(2))
    sq = torch.full((r, L, V), float("nan"), device=DEV)
    flag = torch.zeros(1, dtype=torch.int32, device=DEV)
    _C.variant_expand(g.ndata["x"], g.node_off, g.edge_off, g._src_local, g._dst_local, g.edata["edge_attr"], seq, sample,
                      offsets, ni, si, res, (c["cols"] if cols is None else cols).to(DEV), node_out, edge_out, xo, so, do,
                      eo, sq, flag)
    return xo, so, do, eo, sq, int(flag)


@pytest.mark.parametrize("b", [7, 512])
def test_expand_kernel_against_contract(b):
    c = _case(b, 5, big=True)
    lib = _library(b, 4096, 6)
    assert 3 * len(lib) > 10 * 4 * _C.num_sms()                         # every CTA loops over many (variant, part) units
    assert int(c["arr"]["node_counts"][0]) == 256
    got = _expand(c, lib)
    ref = run_contract(c["arr"], c["seq_cpu"], c["cols"], *library_tables(lib))
    assert got[5] == ref[5] == 0
    for a, r_ in zip(got[:5], ref[:5]):
        assert torch.equal(a.cpu(), r_)
    again = _expand(c, lib)
    assert all(torch.equal(a, b_) for a, b_ in zip(got[:5], again[:5]))


def test_expand_kernel_flags_bad_substitutions():
    c = _case(9, 6)
    lib = _library(9, 64, 7)
    bad_libs = [lib + [(0, [(195, 3, 4)])],                               # graph 0: 200 nodes, the last 10 padded
                lib + [(1, [(-1, 5, 4)] + [(0, 0, 1)])]]
    seq2 = c["seq_cpu"].clone()
    seq2[1, 5, 0] = 1.0 - seq2[1, 5, 0]                                   # sequence row 5 of sample 1 is not one-hot
    for lib_, seq in zip(bad_libs, (c["seq_cpu"], seq2)):
        cc = dict(c, seq_cpu=seq, seq=seq.to(DEV))
        got = _expand(cc, lib_)
        ref = run_contract(c["arr"], seq, c["cols"], *library_tables(lib_))
        assert got[5] == ref[5] == 1
        for a, r_ in zip(got[:5], ref[:5]):
            assert torch.equal(a.cpu(), r_)
    got = _expand(c, lib, cols=c["cols"].roll(1))                         # a wrong map
    ref = run_contract(c["arr"], c["seq_cpu"], c["cols"].roll(1), *library_tables(lib))
    assert got[5] == ref[5] == 1 and all(torch.equal(a.cpu(), r_) for a, r_ in zip(got[:5], ref[:5]))


# ---- identities with predictive and the scan ---------------------------------------------------------------------------
@pytest.mark.parametrize("name", ["HybridModel", "HybridModelv2"])
def test_identity_table_equals_predictive(name):
    c = _case(40, 8, name)
    eps = _eps(3, 40, 9)
    res = _score(c, [(i, []) for i in range(40)], eps=eps, max_graphs=64)
    ref = predictive(c["model"], c["g"], c["seq"], c["prop"], eps=eps)
    for f in ("logits", "prob_mean", "prob_std"):
        assert torch.equal(getattr(res, f), getattr(ref, f)), f
        assert torch.equal(getattr(res.base, f), getattr(ref, f)), f


def test_single_site_table_equals_mutational_scan():
    b, n_sites, k = 24, 3, 2
    c = _case(b, 10)
    ni = torch.tensor([[3 * p + i % 4 for p in range(n_sites)] for i in range(b)])
    eps = _eps(k, b, 11)
    lib = [(i, [(int(ni[i, p]), int(ni[i, p]), col)]) for p in range(n_sites) for col in range(20) for i in range(b)]
    res = _score(c, lib, eps=eps, max_graphs=b * 7)
    scan = mutational_scan(c["model"], c["g"], c["seq"], c["prop"], ni, ni, seq_columns=c["cols"], eps=eps,
                           max_graphs=b * 7)
    assert torch.equal(res.logits, scan.logits.permute(1, 2, 0, 3).reshape(-1, k))
    assert torch.equal(res.prob_mean, scan.prob_mean.permute(1, 2, 0).reshape(-1))
    assert torch.equal(res.prob_std, scan.prob_std.permute(1, 2, 0).reshape(-1))
    assert torch.equal(res.base.logits, scan.base.logits)


# ---- entries against the fused eval forward and the fp64 oracle ---------------------------------------------------------
@pytest.mark.parametrize("precision", ["fp16x2", "bf16x3", "bf16"], indirect=True)
@pytest.mark.parametrize("name", ["HybridModel", "HybridModelv2", "HybridModel_SSL", "HybridModelv2_SSL"])
def test_entries_match_the_fused_forward(precision, name):
    c = _case(24, 12, name)
    lib = _library(24, 40, 13)
    eps = _eps(3, 24, 14)
    res = _score(c, lib, eps=eps, max_graphs=16)
    _, g, seq, samples = _mutants(c, lib)
    for k in (0, 2):
        inject_eps(c["model"], eps[k][samples])
        with torch.no_grad():
            ref = c["model"](g, seq, c["prop"][samples])[3].reshape(-1)
        # (the last Linear of the SSL forward runs in torch, after the fused head: 1e-5 as in predictive)
        _close(res.logits[:, k], ref, TOL if name.endswith("_SSL") else BATCH_TOL)
    del c["model"].sample_eps


def _og64(arr):
    og = R.dgl_batch(split_graphs(arr))
    return dict(og, x=og["x"].double(), edge_attr=og["edge_attr"].double())


@pytest.mark.parametrize("precision", ["fp16x2", "bf16x3", "fp32"], indirect=True)
def test_entries_match_fp64_oracle(precision):
    c = _case(5, 31, ragged=False)
    lib = _library(5, 10, 32)
    eps = _eps(2, 5, 33)
    res = _score(c, lib, eps=eps, max_graphs=4)
    arr, _, seq, samples = _mutants(c, lib)
    p64 = {k: v.detach().double().cpu() for k, v in c["model"].state_dict().items()}
    for k in range(2):
        ref = R.hybrid_forward(p64, _og64(arr), seq.double().cpu(), c["prop"][samples].double().cpu(),
                               eps[k][samples].double().cpu(), version="v2")[3].reshape(-1)
        _close(res.logits[:, k].cpu(), ref)


# ---- pass size ----------------------------------------------------------------------------------------------------------
def test_pass_size_independence():
    b = 64
    c = _case(b, 41)
    lib = _library(b, 300, 42)
    eps = _eps(2, b, 43)
    sizes = (4096, 128, 37)
    assert [len(variant_passes(300, m)) for m in sizes] == [1, 3, 9]
    runs = [_score(c, lib, eps=eps, max_graphs=m) for m in sizes]
    # the statistics follow from the logits: sigmoid' <= 1/4 bounds how far a logit error moves them (test_mutscan_gpu)
    stat_lim = BATCH_TOL * float(runs[0].logits.abs().max()) / 4
    for other in runs[1:]:
        _close(other.logits, runs[0].logits, BATCH_TOL)
        for f in ("prob_mean", "prob_std"):
            err = float((getattr(other, f) - getattr(runs[0], f)).abs().max())
            log_error(f"variants: {f} err {err:.3e} err/bound {err / stat_lim:.3f}")
            assert err <= stat_lim, (f, err, stat_lim)
        assert torch.equal(other.base.logits, runs[0].base.logits)


# ---- launches, statistics, draws, gradients ---------------------------------------------------------------------------
def _launches(fn):
    before = _C.LAUNCHES
    out = fn()
    return _C.LAUNCHES - before, out


@pytest.mark.parametrize("k,max_graphs", [(1, 4096), (16, 4096), (1, 16)])
def test_launches_per_pass_statistics_and_draws(k, max_graphs):
    b = 16
    c = _case(b, 51)
    model = c["model"]
    lib = _library(b, 50, 52)
    params = list(model.parameters())
    for i, q in enumerate(params[::3]):
        q.grad = torch.full_like(q, float(i + 1))
    before = [None if q.grad is None else q.grad.clone() for q in params]
    eps = _eps(k, b, 53)
    _score(c, lib, eps=eps, max_graphs=max_graphs)                                       # warm-up
    trunk_head, _ = _launches(lambda: predictive(model, c["g"], c["seq"], c["prop"], eps=eps))
    arr, _, seq, samples = _mutants(c, lib)
    per_pass = 0                        # one eval trunk + head on the pass's r graphs (its vae_fc1 K split is that of r rows)
    for j, r in variant_passes(len(lib), max_graphs):
        g_r = graph_batch(slice_graphs(arr, j, j + r), DEV)
        run = lambda: predictive(model, g_r, seq[j:j + r], c["prop"][samples[j:j + r]], eps=eps[:, samples[j:j + r]])
        run()
        per_pass += _launches(run)[0] + 2                                                # + expansion + collation
    n, res = _launches(lambda: _score(c, lib, eps=eps, max_graphs=max_graphs))
    assert n == trunk_head + per_pass, (n, trunk_head, per_pass)
    pr = torch.sigmoid(res.logits.double())
    assert float((res.prob_mean.double() - pr.mean(-1)).abs().max()) <= 1e-7
    assert float((res.prob_std.double() - pr.std(-1, unbiased=False)).abs().max()) <= 1e-7
    if k > 1:
        assert float(res.prob_std.min()) > 0
    calls = []
    model.sample_eps = lambda like: calls.append(tuple(like.shape)) or torch.randn_like(like)
    drawn = _score(c, lib, samples=k, max_graphs=max_graphs)
    assert calls == [(k * b, 32)] and drawn.logits.shape == (len(lib), k)
    del model.sample_eps
    for q, b_ in zip(params, before):
        assert (q.grad is None) == (b_ is None) and (b_ is None or torch.equal(q.grad, b_))
    assert not res.logits.requires_grad


@pytest.mark.parametrize("use_wt", [True, False])
def test_pair_launches_and_wild_type(use_wt):
    b, max_graphs = 12, 8
    c = _case(b, 61, "HybridModelv2_Comparative", use_wt_for_downstream=use_wt)
    cancer_only = I.model_map["HybridModelv2_Comparative"](vae_input_dim=5943, device=DEV,
                                                          use_wt_for_downstream=False).to(DEV).eval()
    aw = _arrays(b, 62)
    dw = synthetic_dense(b, seed=62)
    gw, seq_w, prop_w = graph_batch(aw, DEV), dw["seq"].to(DEV), dw["prop"].to(DEV)
    lib = _library(b, 30, 63)
    args = ((c["g"], gw), (c["seq"], seq_w), (c["prop"], prop_w))
    eps = (_eps(4, b, 64), _eps(4, b, 65))
    run = lambda **kw: score_variants_pair(c["model"], *args, *library_tables(lib), seq_columns=c["cols"],
                                           max_graphs=max_graphs, **kw)
    res = run(eps=eps)                                                                   # warm-up (cached weight planes)
    base, _ = _launches(lambda: predictive_pair(c["model"], *args, samples=4))
    arr, _, seq, samples = _mutants(c, lib)
    _, gw_m, seq_wm, _ = _mutants(c, [(i, []) for i, _ in lib], arr=aw, seq=dw["seq"])
    # every variant against predictive_pair on the host-built pair batch (the wild type gathered by sample)
    ref = predictive_pair(c["model"], (graph_batch(arr, DEV), gw_m), (seq, seq_wm), (c["prop"][samples], prop_w[samples]),
                          eps=(eps[0][:, samples], eps[1][:, samples]))
    _close(res.logits, ref.logits, BATCH_TOL)
    per_pass = 0                        # one cancer trunk + pair head on the pass's r graphs
    for j, r in variant_passes(len(lib), max_graphs):
        g_r = graph_batch(slice_graphs(arr, j, j + r), DEV)
        s_r = samples[j:j + r]
        pair_r = ((g_r, g_r), (seq[j:j + r], seq[j:j + r]), (c["prop"][s_r], c["prop"][s_r]))
        predictive_pair(cancer_only, *pair_r, samples=4)                                  # cached weight planes
        per_pass += _launches(lambda: predictive_pair(cancer_only, *pair_r, samples=4))[0] + 2
    calls = []
    c["model"].sample_eps = lambda like: calls.append(tuple(like.shape)) or torch.randn_like(like)
    n, res = _launches(lambda: run(samples=4))
    assert calls == [(4 * b, 32)] * (2 if use_wt else 1)                                  # no wild-type draw without use_wt
    assert n == base + per_pass, (n, base, per_pass)                                    # the wild type runs once or never
    assert res.logits.shape == (len(lib), 4)
