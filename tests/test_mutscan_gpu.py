"""Single-residue mutational scan on the B200: the expansion kernel (is_mutscan_expand) against its contract bit for bit,
every entry against the fused eval forward of the host-built mutant batch, the native column against the unmutated
score, the fp64 oracle per mutant, independence of the pass size, the launch count per pass, the statistics, the draws
and no side effects on parameter gradients.

Pass size: two kernels of the eval path make a sample's logit depend on the batch it shares.  The edge kernel sums a
node's messages with a tensor-core MMA over the 128 in-edges of its tile (csrc/egnn_tc2.cu, hn = S m), and where a graph
sits in the batch decides where its edges fall in a tile; the vae_fc1 GEMM (csrc/gemm_tma.cu) splits K into a number of
slices that follows the row count (is_gemm_tma_split_k).  Both change summation orders only, so a scan entry is held to
1e-6 relative against the same variant run in another batch (the forward of the B-sample mutant batch, another pass
size, a single-graph forward)."""
import pytest
import torch
import torch.nn.functional as F

import immunostruct_b200 as I
from immunostruct_b200 import _C
from immunostruct_b200.mutagenesis import mutational_scan, mutational_scan_pair, scan_sites
from immunostruct_b200.predictive import predictive, predictive_pair
from immunostruct_b200.resident import scan_passes
from immunostruct_b200.synthetic import split_graphs, synthetic_dense, synthetic_graph_arrays
from oracle import reference_ops as R

from helpers import concat_graphs, graph_batch, inject_eps, log_error
from test_mutscan_host import mutscan_expand_contract

pytestmark = pytest.mark.gpu
DEV = "cuda"
TOL = 1e-5
BATCH_TOL = 1e-6          # the same variant in another batch: summation order only (module docstring)


@pytest.fixture
def precision(request):
    prev = I.get_precision()
    I.set_precision(request.param)
    yield request.param
    I.set_precision(prev)


def _close(got, ref, tol=TOL):
    ref = ref.detach().double().cpu()
    err = float((got.detach().double().cpu() - ref).abs().max())
    lim = tol * max(float(ref.abs().max()), 1e-30)
    log_error(f"mutscan: err {err:.3e} err/bound {err / lim:.3f} (tol {tol:.0e})")
    assert err <= lim, (err, float(ref.abs().max()))


def _gen(seed):
    return torch.Generator().manual_seed(seed)


def _arrays(b, seed, ragged=True):
    """b graphs in three sizes (200 nodes with 10 padded rows, 120, 60 with 5 padded rows) in blocks, or (``ragged``
    False: what the fp64 oracle takes, like the reference) all of 200 nodes with 10 padded rows."""
    if not ragged:
        return synthetic_graph_arrays(b, 200, 10, seed=seed, n_pad=10)
    sizes = [(200, 10), (120, 0), (60, 5)]
    parts = [synthetic_graph_arrays((b + 2 - i) // 3, n, 10, seed=seed + i, n_pad=pad) for i, (n, pad) in enumerate(sizes)
             if (b + 2 - i) // 3 > 0]
    return concat_graphs(*parts)


def _sites(arr, seq, n_sites, seed):
    """Sites on real residues, the last absent for every seventh sample; the sequence rows at the sites follow
    ``seq_columns`` (20 of the 21 sequence columns, permuted)."""
    b = arr["node_counts"].numel()
    off = torch.cat([torch.zeros(1, dtype=torch.int64), arr["node_counts"].cumsum(0)])
    ni = torch.tensor([[3 * p + i % 5 for p in range(n_sites)] for i in range(b)])
    si = torch.tensor([[p + 1 + i % 3 for p in range(n_sites)] for i in range(b)])
    ni[3::7, -1] = si[3::7, -1] = -1
    cols = torch.randperm(21, generator=_gen(seed))[:20]
    seq = seq.clone()
    for i in range(b):
        for p in range(n_sites):
            if ni[i, p] >= 0:
                seq[i, si[i, p]] = F.one_hot(cols[arr["x"][off[i] + ni[i, p], :20].argmax()], 21).float()
    return ni, si, cols, seq, off


def _case(b, seed, name="HybridModelv2", n_sites=3, ragged=True, **kw):
    arr = _arrays(b, seed, ragged)
    dense = synthetic_dense(b, seed=seed)
    ni, si, cols, seq, off = _sites(arr, dense["seq"], n_sites, seed)
    torch.manual_seed(seed)
    model = I.model_map[name](vae_input_dim=5943, device=DEV, **kw).to(DEV).eval()
    return dict(arr=arr, g=graph_batch(arr, DEV), seq=seq.to(DEV), prop=dense["prop"].to(DEV), ni=ni, si=si, cols=cols,
                off=off, model=model)


def _mutant(c, p, col):
    """The B-sample batch with residue column ``col`` at site p of every sample (host-built)."""
    arr, seq = dict(c["arr"]), c["seq"].cpu().clone()
    x = arr["x"].clone()
    for i in range(c["ni"].shape[0]):
        if c["ni"][i, p] >= 0:
            x[c["off"][i] + c["ni"][i, p], :20] = F.one_hot(torch.tensor(col), 20).float()
            seq[i, c["si"][i, p]] = F.one_hot(c["cols"][col], 21).float()
    arr["x"] = x
    return arr, graph_batch(arr, DEV), seq.to(DEV)


def _eps(k, b, seed):
    return torch.randn(k, b, 32, generator=_gen(seed)).to(DEV)


def _scan(c, **kw):
    return mutational_scan(c["model"], c["g"], c["seq"], c["prop"], c["ni"], c["si"], seq_columns=c["cols"], **kw)


# ---- the kernel against its contract ---------------------------------------------------------------------------------
def _expand(g, seq, ni, si, cols, sites):
    r, n, (b, L, V) = sites.shape[0], g.n_nodes, seq.shape
    dev = lambda t: t.to(DEV).contiguous()
    xo = torch.full((r * n, 23), float("nan"), device=DEV)
    so = torch.full((r * b, L, V), float("nan"), device=DEV)
    flag = torch.zeros(1, dtype=torch.int32, device=DEV)
    _C.mutscan_expand(g.ndata["x"], g.node_off, dev(ni), dev(seq), dev(si), dev(cols), dev(sites), xo, so, flag)
    return xo, so, flag


def _contract(g, seq, ni, si, cols, sites):
    r, n, (b, L, V) = sites.shape[0], g.n_nodes, seq.shape
    xo, so, flag = torch.empty(r * n, 23), torch.empty(r * b, L, V), torch.zeros(1, dtype=torch.int32)
    mutscan_expand_contract(g.ndata["x"].cpu(), g.node_off.cpu(), ni, seq.cpu(), si, cols, sites, xo, so, flag)
    return xo, so, flag


@pytest.mark.parametrize("b,which", [(7, "one"), (512, "one"), (512, "three"), (512, "twenty")])
def test_expand_kernel_against_contract(b, which):
    c = _case(b, 5, n_sites=3)
    sites = scan_sites(3)
    sites = {"one": sites[37:38], "three": sites[20:23], "twenty": sites[10:30]}[which]
    cap = 6 * _C.num_sms()                                              # the launcher's grid cap
    if which == "twenty":
        assert 2 * sites.shape[0] * b > 20 * cap                      # every CTA loops over many (copy, graph) units
    got = _expand(c["g"], c["seq"], c["ni"], c["si"], c["cols"], sites)
    ref = _contract(c["g"], c["seq"], c["ni"], c["si"], c["cols"], sites)
    for a, r_ in zip(got, ref):
        assert torch.equal(a.cpu(), r_)
    assert int(got[2]) == 0
    again = _expand(c["g"], c["seq"], c["ni"], c["si"], c["cols"], sites)
    assert all(torch.equal(a, b_) for a, b_ in zip(got, again))


def test_expand_kernel_flags_bad_sites():
    c = _case(9, 6, n_sites=2)
    sites = scan_sites(2)
    padded = c["ni"].clone()
    padded[0, 0] = 195                                                  # graph 0: 200 nodes, the last 10 padded
    wrong = c["cols"].roll(1)
    for ni, cols in ((padded, c["cols"]), (c["ni"], wrong)):
        got = _expand(c["g"], c["seq"], ni, c["si"], cols, sites)
        ref = _contract(c["g"], c["seq"], ni, c["si"], cols, sites)
        assert int(got[2]) == 1 and int(ref[2]) == 1
        assert torch.equal(got[0].cpu(), ref[0]) and torch.equal(got[1].cpu(), ref[1])


# ---- entries against the fused eval forward ---------------------------------------------------------------------------
@pytest.mark.parametrize("precision", ["fp16x2", "bf16x3", "bf16"], indirect=True)
@pytest.mark.parametrize("name", ["HybridModel", "HybridModelv2", "HybridModel_SSL", "HybridModelv2_SSL"])
def test_entries_match_the_fused_forward(precision, name):
    c = _case(40, 11, name)
    eps = _eps(3, 40, 12)
    res = _scan(c, eps=eps)
    for p, col in ((0, 0), (1, 13), (2, 19), (2, 7)):
        _, g, seq = _mutant(c, p, col)
        for k in (0, 2):
            inject_eps(c["model"], eps[k])
            with torch.no_grad():
                ref = c["model"](g, seq, c["prop"])[3].reshape(-1)
            keep = (c["ni"][:, p] >= 0).to(DEV)
            got = res.logits[:, p, col, k]
            assert torch.isnan(got[~keep]).all()
            # (the last Linear of the SSL forward runs in torch, after the fused head: 1e-5 as in predictive)
            _close(got[keep], ref[keep], TOL if name.endswith("_SSL") else BATCH_TOL)
    present = (c["ni"] >= 0).to(DEV)
    i, p = present.nonzero(as_tuple=True)
    _close(res.logits[i, p, res.native[i, p]], res.base.logits[i], BATCH_TOL)
    assert (res.native[~present] == -1).all()


@pytest.mark.parametrize("name", ["HybridModel_Comparative", "HybridModel_Comparative_SSL", "HybridModelv2_Comparative",
                                  "HybridModelv2_Comparative_SSL"])
def test_pair_entries_equal_predictive_pair(name):
    c = _case(24, 21, name)
    aw = _arrays(24, 22)
    dw = synthetic_dense(24, seed=22)
    gw, seq_w, prop_w = graph_batch(aw, DEV), dw["seq"].to(DEV), dw["prop"].to(DEV)
    eps = (_eps(2, 24, 23), _eps(2, 24, 24))
    res = mutational_scan_pair(c["model"], (c["g"], gw), (c["seq"], seq_w), (c["prop"], prop_w), c["ni"], c["si"],
                               seq_columns=c["cols"], eps=eps, max_graphs=24 * 7)
    base = predictive_pair(c["model"], (c["g"], gw), (c["seq"], seq_w), (c["prop"], prop_w), eps=eps)
    assert torch.equal(res.base.logits, base.logits)
    for p, col in ((0, 4), (2, 11)):
        _, g, seq = _mutant(c, p, col)
        ref = predictive_pair(c["model"], (g, gw), (seq, seq_w), (c["prop"], prop_w), eps=eps)
        keep = (c["ni"][:, p] >= 0).to(DEV)
        _close(res.logits[:, p, col][keep], ref.logits[keep], BATCH_TOL)
        _close(res.prob_mean[:, p, col][keep], ref.prob_mean[keep], BATCH_TOL)


# ---- the fp64 oracle --------------------------------------------------------------------------------------------------
def _og64(arr):
    og = R.dgl_batch(split_graphs(arr))
    return dict(og, x=og["x"].double(), edge_attr=og["edge_attr"].double())


@pytest.mark.parametrize("precision", ["fp16x2", "bf16x3", "fp32"], indirect=True)
def test_entries_match_fp64_oracle(precision):
    c = _case(5, 31, n_sites=2, ragged=False)
    eps = _eps(2, 5, 32)
    res = _scan(c, eps=eps)
    p64 = {k: v.detach().double().cpu() for k, v in c["model"].state_dict().items()}
    for p, col in ((0, 2), (1, 17), (0, 9)):
        arr, _, seq = _mutant(c, p, col)
        for k in range(2):
            ref = R.hybrid_forward(p64, _og64(arr), seq.double().cpu(), c["prop"].double().cpu(), eps[k].double().cpu(),
                                   version="v2")[3].reshape(-1)
            keep = c["ni"][:, p] >= 0
            _close(res.logits[:, p, col, k].cpu()[keep], ref[keep])


# ---- pass size ----------------------------------------------------------------------------------------------------------
def test_pass_size_independence():
    b = 200
    c = _case(b, 41, n_sites=2)
    eps = _eps(2, b, 42)
    runs = [_scan(c, eps=eps, max_graphs=m) for m in (b, 3 * b, 4096)]
    assert [len(scan_passes(40, b, m)) for m in (b, 3 * b, 4096)] == [40, 14, 2]
    present = (c["ni"] >= 0).to(DEV)
    # the statistics follow from the logits: sigmoid' <= 1/4 bounds how far a logit error moves a probability, its mean and
    # its spread (the spread is small next to the probabilities, so its own scale would be too tight a yardstick)
    stat_lim = BATCH_TOL * float(runs[0].logits[present].abs().max()) / 4
    for other in runs[1:]:
        assert all(torch.isnan(getattr(other, f)[~present]).all() for f in ("logits", "prob_mean", "prob_std"))
        _close(other.logits[present], runs[0].logits[present], BATCH_TOL)
        for f in ("prob_mean", "prob_std"):
            err = float((getattr(other, f)[present] - getattr(runs[0], f)[present]).abs().max())
            log_error(f"mutscan: {f} err {err:.3e} err/bound {err / stat_lim:.3f}")
            assert err <= stat_lim, (f, err, stat_lim)
        assert torch.equal(other.native, runs[0].native)
        assert torch.equal(other.base.logits, runs[0].base.logits)
    for i in (0, 3, 100):
        one = {k: v for k, v in split_graphs(c["arr"])[i].items()}
        for p, col in ((0, 5), (1, 12)):
            if c["ni"][i, p] < 0:
                continue
            x = one["x"].clone()
            x[c["ni"][i, p], :20] = F.one_hot(torch.tensor(col), 20).float()
            seq = c["seq"][i:i + 1].clone()
            seq[0, c["si"][i, p]] = F.one_hot(c["cols"][col], 21).float().to(DEV)
            g1 = graph_batch({"x": x, "src": one["src"], "dst": one["dst"], "edge_attr": one["edge_attr"],
                              "node_counts": torch.tensor([x.shape[0]]), "edge_counts": torch.tensor([one["src"].numel()])},
                             DEV)
            single = predictive(c["model"], g1, seq, c["prop"][i:i + 1], eps=eps[:, i:i + 1])
            _close(runs[0].logits[i, p, col], single.logits[0], BATCH_TOL)


# ---- launches, statistics, draws, gradients ---------------------------------------------------------------------------
def _launches(fn):
    before = _C.LAUNCHES
    out = fn()
    return _C.LAUNCHES - before, out


@pytest.mark.parametrize("n_sites,k,max_graphs", [(1, 1, 4096), (3, 16, 4096), (3, 1, 16 * 7)])
def test_launches_per_pass_statistics_and_draws(n_sites, k, max_graphs):
    c = _case(16, 51, n_sites=n_sites)
    model = c["model"]
    params = list(model.parameters())
    for i, q in enumerate(params[::3]):
        q.grad = torch.full_like(q, float(i + 1))
    before = [None if q.grad is None else q.grad.clone() for q in params]
    eps = _eps(k, 16, 52)
    _scan(c, eps=eps, max_graphs=max_graphs)                                           # warm-up
    trunk_head, _ = _launches(lambda: predictive(model, c["g"], c["seq"], c["prop"], eps=eps))
    passes = scan_passes(n_sites * 20, 16, max_graphs)
    per_pass = {}                       # one eval trunk + head on the r-copy batch (its vae_fc1 K split is that of r*B rows)
    for r in {r for _, r in passes}:
        g_r = c["g"].replicate(r)
        per_pass[r] = _launches(lambda: predictive(model, g_r, c["seq"].repeat(r, 1, 1), c["prop"].repeat(r, 1),
                                                   eps=eps.repeat(1, r, 1)))[0]
    n, res = _launches(lambda: _scan(c, eps=eps, max_graphs=max_graphs))
    assert n == trunk_head + len(per_pass) + sum(per_pass[r] + 1 for _, r in passes)
    pr = torch.sigmoid(res.logits.double())
    keep = ~torch.isnan(pr[..., 0])
    assert float((res.prob_mean.double()[keep] - pr.mean(-1)[keep]).abs().max()) <= 1e-7
    assert float((res.prob_std.double()[keep] - pr.std(-1, unbiased=False)[keep]).abs().max()) <= 1e-7
    if k > 1:
        assert float(res.prob_std[keep].min()) > 0
    calls = []
    model.sample_eps = lambda like: calls.append(tuple(like.shape)) or torch.randn_like(like)
    drawn = _scan(c, samples=k, max_graphs=max_graphs)
    assert calls == [(k * 16, 32)] and drawn.logits.shape == (16, n_sites, 20, k)
    del model.sample_eps
    for q, b_ in zip(params, before):
        assert (q.grad is None) == (b_ is None) and (b_ is None or torch.equal(q.grad, b_))
    assert not res.logits.requires_grad


@pytest.mark.parametrize("use_wt", [True, False])
def test_pair_launches_and_wild_type(use_wt):
    b, max_graphs = 12, 12 * 9
    c = _case(b, 61, "HybridModelv2_Comparative", n_sites=2, use_wt_for_downstream=use_wt)
    cancer_only = I.model_map["HybridModelv2_Comparative"](vae_input_dim=5943, device=DEV,
                                                          use_wt_for_downstream=False).to(DEV).eval()
    aw = _arrays(b, 62)
    dw = synthetic_dense(b, seed=62)
    gw, seq_w, prop_w = graph_batch(aw, DEV), dw["seq"].to(DEV), dw["prop"].to(DEV)
    args = ((c["g"], gw), (c["seq"], seq_w), (c["prop"], prop_w))
    scan = lambda: mutational_scan_pair(c["model"], *args, c["ni"], c["si"], seq_columns=c["cols"], samples=4,
                                        max_graphs=max_graphs)
    scan()                                                                              # warm-up (and cached weight planes)
    base, _ = _launches(lambda: predictive_pair(c["model"], *args, samples=4))
    passes = scan_passes(40, b, max_graphs)
    per_pass = {}                       # one cancer trunk + pair head on the r-copy batch
    for r in {r for _, r in passes}:
        rep = lambda t: t.repeat(r, *([1] * (t.dim() - 1)))
        g_r = c["g"].replicate(r)
        pair_r = ((g_r, gw.replicate(r)), (rep(c["seq"]), rep(seq_w)), (rep(c["prop"]), rep(prop_w)))
        predictive_pair(cancer_only, *pair_r, samples=4)                                # cached weight planes
        per_pass[r] = _launches(lambda: predictive_pair(cancer_only, *pair_r, samples=4))[0]
    calls = []
    c["model"].sample_eps = lambda like: calls.append(tuple(like.shape)) or torch.randn_like(like)
    n, res = _launches(scan)
    assert calls == [(4 * b, 32)] * (2 if use_wt else 1)                                  # no wild-type draw without use_wt
    assert n == base + len(per_pass) + sum(per_pass[r] + 1 for _, r in passes)         # the wild type runs once or never
    assert res.logits.shape == (b, 2, 20, 4)
