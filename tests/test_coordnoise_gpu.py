"""Structural uncertainty on the B200: the expansion kernel (is_coord_noise_expand) against its contract, the distribution
of its normals, independence of the pass size and of the run, every entry against the fused eval forward of the
perturbed batch and against the fp64 oracle, ``base`` against ``predictive``, sigma 0 and isolated rows, the variance
split, the launches of each pass with no host read between them, the pair form, gradients and argument rules.

An entry is held to 1e-6 relative against the same graph run in another batch: where a graph sits in a batch changes two
summation orders of the eval path (tests/test_mutscan_gpu.py, DESIGN 4.4c)."""
import numpy as np
import pytest
import torch
from scipy import stats

import immunostruct_b200 as I
from immunostruct_b200 import _C
from immunostruct_b200.coordnoise import coordinate_ensemble, coordinate_ensemble_pair
from immunostruct_b200.predictive import predictive, predictive_pair
from immunostruct_b200.resident import scan_passes
from immunostruct_b200.synthetic import synthetic_dense, synthetic_graph_arrays
from oracle import reference_ops as R

from helpers import concat_graphs, graph_batch, inject_eps, log_error
from test_coordnoise_host import _offsets, coord_noise_expand_contract, normals, perturbed_batches
from test_variants_gpu import _arrays, _case, _og64

pytestmark = pytest.mark.gpu
DEV = "cuda"
TOL = 1e-5
BATCH_TOL = 1e-6          # the same graph in another batch: summation order only (module docstring)
Z_TOL = 2.0 ** -21        # 4 fp32 ulps: the rounding of logf, sqrtf, sincospif and one product
SEED = 2 ** 63 + 0x1234567


@pytest.fixture
def precision(request):
    prev = I.get_precision()
    I.set_precision(request.param)
    yield request.param
    I.set_precision(prev)


def _close(got, ref, tol=TOL, what="coordnoise"):
    ref = ref.detach().double().cpu()
    err = float((got.detach().double().cpu() - ref).abs().max())
    lim = tol * max(float(ref.abs().max()), 1e-30)
    log_error(f"{what}: err {err:.3e} err/bound {err / lim:.3f} (tol {tol:.0e})")
    assert err <= lim, (err, float(ref.abs().max()))


def _eps(k, b, seed):
    return torch.randn(k, b, 32, generator=torch.Generator().manual_seed(seed)).to(DEV)


def _bits(t):
    return t.view(torch.int32)


def _sigma(arr, seed, zero_every=5):
    """Per-row sigma in [0.25, 1.75), 0 on every ``zero_every``-th row."""
    n = int(arr["node_counts"].sum())
    s = 0.25 + 1.5 * torch.rand(n, generator=torch.Generator().manual_seed(seed))
    s[::zero_every] = 0.0
    return s


def _keys(arr):
    """(graph b, graph-local row a) of every node row."""
    counts = arr["node_counts"].numpy()
    b = np.repeat(np.arange(counts.size), counts)
    return b, np.arange(b.size) - _offsets(arr["node_counts"]).numpy()[b]


def _expand(arr, sigma, seed, item, draw0, r, x=None):
    """The device kernel on a graph-array batch -> x23_out [r N, 23] on the host."""
    x = (arr["x"] if x is None else x).to(DEV).contiguous()
    out = torch.full((r * x.shape[0], 23), float("nan"), device=DEV)
    _C.coord_noise_expand(x, _offsets(arr["node_counts"]).to(DEV), sigma.to(DEV), seed, item, draw0, out)
    return out.cpu()


# ---- the kernel against its contract -----------------------------------------------------------------------------------
@pytest.mark.parametrize("case", ["b7", "b512", "big"])
def test_expand_kernel_against_contract(case):
    arr = {"b7": lambda: _arrays(7, 3), "b512": lambda: synthetic_graph_arrays(512, 200, 10, seed=4, n_pad=10),
           "big": lambda: concat_graphs(_arrays(48, 5, big=True), _arrays(5, 6))}[case]()
    if case == "big":
        assert int(arr["node_counts"][0]) == 256
    n = int(arr["node_counts"].sum())
    sigma = _sigma(arr, 7)
    b, a = _keys(arr)
    live = sigma.numpy() != 0
    for r, draw0, item in {"b7": [(1, 0, 0), (3, 2, 1), (16, 0, 0)], "b512": [(8, 8, 0)], "big": [(5, 1, 1)]}[case]:
        dev = _expand(arr, sigma, SEED, item, draw0, r)
        ref = torch.empty(r * n, 23)
        coord_noise_expand_contract(arr["x"], _offsets(arr["node_counts"]), sigma, SEED, item, draw0, ref)
        assert torch.equal(_bits(dev[:, :20]), _bits(ref[:, :20]))
        for k in range(r):
            blk, rblk = dev[k * n:(k + 1) * n], ref[k * n:(k + 1) * n]
            assert torch.equal(_bits(blk[~torch.from_numpy(live)]), _bits(arr["x"][~torch.from_numpy(live)]))
            z = normals(SEED, item, draw0 + k, b[live], a[live])
            step = np.abs(sigma.numpy()[live, None].astype(np.float64) * z)
            err = np.abs(blk[live, 20:].double().numpy() - rblk[live, 20:].double().numpy())
            # the z of the two differ by Z_TOL relative at most; the final fmaf / fp32 rounding by one ulp
            lim = Z_TOL * step + 2.0 ** -23 * np.abs(rblk[live, 20:].double().numpy())
            log_error(f"coord_noise_expand {case} r={r}: err/bound {float((err / np.maximum(lim, 1e-300)).max()):.3f}")
            assert (err <= lim).all()


def test_expand_kernel_normals_are_the_contract():
    """x = 0, sigma = 1: the output is z; within 4 fp32 ulps of the fp64 Box-Muller on the same uniforms."""
    arr = _arrays(7, 8)
    x = arr["x"].clone()
    x[:, 20:] = 0.0
    n = x.shape[0]
    b, a = _keys(arr)
    for r, draw0, item in ((1, 0, 0), (4, 3, 1)):
        out = _expand(arr, torch.ones(n), SEED, item, draw0, r, x=x)
        for k in range(r):
            z = normals(SEED, item, draw0 + k, b, a)
            got = out[k * n:(k + 1) * n, 20:].double().numpy()
            err = np.abs(got - z)
            lim = Z_TOL * np.maximum(np.abs(z), 2.0 ** -126)
            log_error(f"coord_noise_expand z r={r}: err/bound {float((err / lim).max()):.3f}")
            assert (err <= lim).all()


def test_device_normals_distribution():
    b, m = 512, 16
    arr = synthetic_graph_arrays(b, 200, 10, seed=9, n_pad=10)
    x = arr["x"].clone()
    x[:, 20:] = 0.0
    out = _expand(arr, torch.ones(x.shape[0]), 20260101, 0, 0, m, x=x)
    z = out[:, 20:].double().numpy()
    flat = z.reshape(-1)
    n = flat.size
    assert n == b * 200 * m * 3
    assert abs(flat.mean()) < 5 / np.sqrt(n)
    assert abs(flat.var() - 1) < 5 * np.sqrt(2 / n)
    assert abs(stats.skew(flat)) < 5 * np.sqrt(6 / n) and abs(stats.kurtosis(flat)) < 5 * np.sqrt(24 / n)
    assert np.abs(np.corrcoef(z.T) - np.eye(3)).max() < 5 / np.sqrt(z.shape[0])
    rows = z.reshape(m, b, 200, 3)
    for x0, x1 in ((rows[:, :, :-1], rows[:, :, 1:]), (rows[:, :-1], rows[:, 1:]), (rows[:-1], rows[1:])):   # a, b, m
        assert abs(np.corrcoef(x0.reshape(-1), x1.reshape(-1))[0, 1]) < 5 / np.sqrt(x0.size)
    assert stats.kstest(flat, "norm").pvalue > 1e-3


# ---- entries against the fused eval forward and the fp64 oracle ---------------------------------------------------------
def _fused(c, x_m, eps_k):
    """Logit of the fused eval forward of batch ``c`` with node features ``x_m`` on draw ``eps_k`` [B, latent]."""
    g = graph_batch(dict(c["arr"], x=x_m.cpu()), DEV)
    inject_eps(c["model"], eps_k)
    with torch.no_grad():
        out = c["model"](g, c["seq"], c["prop"])[3].reshape(-1)
    del c["model"].sample_eps
    return out


@pytest.mark.parametrize("precision", ["fp16x2", "bf16x3"], indirect=True)
@pytest.mark.parametrize("name", ["HybridModel", "HybridModelv2"])
def test_entries_match_the_fused_forward(precision, name):
    c = _case(12, 12, name)
    eps = _eps(3, 12, 14)
    sigma = _sigma(c["arr"], 15)
    m_count = 5
    # max_graphs = B: every structure is one pass of the B graphs at their own positions, with the encoder at B rows
    res = coordinate_ensemble(c["model"], c["g"], c["seq"], c["prop"], sigma=sigma.to(DEV), structures=m_count,
                              seed=SEED, eps=eps, max_graphs=c["b"])
    for m in range(m_count):
        x_m = _expand(c["arr"], sigma, SEED, 0, m, 1)                  # structure m written alone
        for k in (0, 2):
            _close(res.logits[:, m, k], _fused(c, x_m, eps[k]), BATCH_TOL)
    assert float((res.logits - res.base.logits[:, None]).abs().max()) > 1e-6      # the coordinates reach the score


@pytest.mark.parametrize("precision", ["fp16x2", "bf16x3"], indirect=True)
def test_entries_match_fp64_oracle(precision):
    c = _case(3, 31, ragged=False)
    eps = _eps(2, 3, 33)
    sigma = _sigma(c["arr"], 34)
    m_count = 3
    res = coordinate_ensemble(c["model"], c["g"], c["seq"], c["prop"], sigma=sigma.to(DEV), structures=m_count,
                              seed=SEED, eps=eps, max_graphs=4)
    p64 = {k: v.detach().double().cpu() for k, v in c["model"].state_dict().items()}
    for m, pert in enumerate(perturbed_batches(c["arr"], sigma, SEED, 0, m_count)):
        for k in range(2):
            ref = R.hybrid_forward(p64, _og64(pert), c["seq"].double().cpu(), c["prop"].double().cpu(),
                                   eps[k].double().cpu(), version="v2")[3].reshape(-1)
            _close(res.logits[:, m, k].cpu(), ref)


# ---- pass size, seeds, sigma 0, isolated rows, base, the variance split ------------------------------------------------
def _record(monkeypatch):
    """Wrap the expansion: every call's output copied out."""
    seen, expand = [], _C.coord_noise_expand

    def rec(*a):
        expand(*a)
        seen.append(a[-1].clone())

    monkeypatch.setattr(_C, "coord_noise_expand", rec)
    return seen


def test_pass_size_seed_and_base(monkeypatch):
    b, m_count = 24, 16
    c = _case(b, 41)
    eps = _eps(4, b, 43)
    sigma = _sigma(c["arr"], 44).to(DEV)
    runs, coords = [], []
    for mg in (4096, 5 * b):
        seen = _record(monkeypatch)
        runs.append(coordinate_ensemble(c["model"], c["g"], c["seq"], c["prop"], sigma=sigma, structures=m_count,
                                        seed=SEED, eps=eps, max_graphs=mg))
        coords.append(torch.cat(seen))
        monkeypatch.undo()
    assert len(scan_passes(m_count, b, 5 * b)) == 4
    assert torch.equal(_bits(coords[0]), _bits(coords[1]))              # the same structures, whatever the passes
    _close(runs[1].logits, runs[0].logits, BATCH_TOL)
    again = coordinate_ensemble(c["model"], c["g"], c["seq"], c["prop"], sigma=sigma, structures=m_count, seed=SEED,
                                eps=eps, max_graphs=4096)
    assert torch.equal(again.logits, runs[0].logits) and again.seed == SEED
    other = coordinate_ensemble(c["model"], c["g"], c["seq"], c["prop"], sigma=sigma, structures=m_count, seed=SEED + 1,
                                eps=eps, max_graphs=4096)
    assert not torch.equal(other.logits, runs[0].logits)
    ref = predictive(c["model"], c["g"], c["seq"], c["prop"], eps=eps)
    for run in runs + [other]:
        for f in ("logits", "prob_mean", "prob_std"):
            assert torch.equal(getattr(run.base, f), getattr(ref, f)), f
    res = runs[0]
    p = torch.sigmoid(res.logits.double())
    total = res.prob_std.double().square()
    split = res.std_structure.double().square() + res.std_latent.double().square()
    assert float((total - split).abs().max()) <= 1e-6 * float(total.max())
    assert float((res.prob_mean.double() - p.mean((1, 2))).abs().max()) < 1e-7
    assert float((res.std_structure.double() - p.mean(2).std(1, unbiased=False)).abs().max()) < 1e-7
    assert float(res.std_structure.min()) > 0 and float(res.std_latent.min()) > 0


def test_sigma_zero_and_isolated_rows():
    b = 24
    c = _case(b, 45)
    eps = _eps(2, b, 46)
    g = c["g"]
    zero = coordinate_ensemble(c["model"], g, c["seq"], c["prop"], sigma=0.0, structures=6, seed=SEED, eps=eps)
    _close(zero.logits, zero.base.logits[:, None].expand(-1, 6, -1), BATCH_TOL)
    x = g.ndata["x"]
    touched = torch.zeros(g.n_nodes, dtype=torch.bool, device=DEV)
    touched[g.edge_index[0]] = True
    touched[g.edge_index[1]] = True
    isolated = ~touched
    assert int(isolated.sum()) > 0 and bool((x[isolated] == 0).all())   # the padded rows
    sigma = torch.where(isolated, 3.0, 0.0).float()
    pad = coordinate_ensemble(c["model"], g, c["seq"], c["prop"], sigma=sigma, structures=6, seed=SEED, eps=eps)
    assert torch.equal(pad.logits, zero.logits)                        # an isolated row's coordinates reach nothing


# ---- launches, host reads, gradients, argument rules -------------------------------------------------------------------
def _names(fn, monkeypatch):
    names = []
    call = _C._call
    monkeypatch.setattr(_C, "_call", lambda name, *a: names.append(name) or call(name, *a))
    try:
        out = fn()
    finally:
        monkeypatch.setattr(_C, "_call", call)
    return names, out


def test_launches_host_reads_and_gradients(monkeypatch):
    b, m_count, max_graphs = 16, 7, 48
    c = _case(b, 51)
    model = c["model"]
    params = list(model.parameters())
    for i, q in enumerate(params[::3]):
        q.grad = torch.full_like(q, float(i + 1))
    before = [None if q.grad is None else q.grad.clone() for q in params]
    eps = _eps(4, b, 53)
    sigma = _sigma(c["arr"], 54).to(DEV)
    run = lambda: coordinate_ensemble(model, c["g"], c["seq"], c["prop"], sigma=sigma, structures=m_count, seed=SEED,
                                      eps=eps, max_graphs=max_graphs)
    res = run()                                                                        # warm-up
    base, _ = _names(lambda: predictive(model, c["g"], c["seq"], c["prop"], eps=eps), monkeypatch)
    passes = scan_passes(m_count, b, max_graphs)
    assert passes == [(0, 3), (3, 3), (6, 1)]
    sizes = sorted({r for _, r in passes})
    expected = list(base) + ["is_collate_csr"] * len(sizes)
    for _, r in passes:
        g_r = c["g"].replicate(r)
        with torch.no_grad():
            trunk, _ = _names(lambda: model.structure_embedding(g_r, project=False), monkeypatch)
        expected += ["is_coord_noise_expand"] + trunk + ["is_head_mc_infer"]
    names, again = _names(run, monkeypatch)
    assert names == expected
    assert names.count("is_vae_mid_infer") == 1                                        # the encoder ran once
    assert torch.equal(again.logits, res.logits)
    # no host read from the first expansion to the result
    expand = _C.coord_noise_expand

    def expand_(*a):
        torch.cuda.set_sync_debug_mode("error")
        expand(*a)

    monkeypatch.setattr(_C, "coord_noise_expand", expand_)
    try:
        quiet = run()
    finally:
        torch.cuda.set_sync_debug_mode("default")
    monkeypatch.setattr(_C, "coord_noise_expand", expand)
    assert torch.equal(quiet.logits, res.logits)
    for q, b_ in zip(params, before):
        assert (q.grad is None) == (b_ is None) and (b_ is None or torch.equal(q.grad, b_))
    assert not res.logits.requires_grad
    torch.manual_seed(3)
    s1 = coordinate_ensemble(model, c["g"], c["seq"], c["prop"], sigma=sigma, structures=2, eps=eps).seed
    torch.manual_seed(3)
    assert coordinate_ensemble(model, c["g"], c["seq"], c["prop"], sigma=sigma, structures=2, eps=eps).seed == s1
    model.train()
    with pytest.raises(RuntimeError, match="eval"):
        run()
    model.eval()
    with pytest.raises(NotImplementedError, match="HybridModelv2_SSL"):
        coordinate_ensemble(I.model_map["StructureModelv2"](vae_input_dim=5943, device=DEV).to(DEV).eval(), c["g"],
                            c["seq"], c["prop"], sigma=1.0)
    with pytest.raises(ValueError, match="finite and >= 0 in every row"):
        coordinate_ensemble(model, c["g"], c["seq"], c["prop"], sigma=-sigma)


@pytest.mark.parametrize("use_wt,perturb_wt", [(True, True), (True, False), (False, False)])
def test_pair_against_forward_comparative(use_wt, perturb_wt, monkeypatch):
    b, m_count = 10, 3
    c = _case(b, 61, "HybridModelv2_Comparative", use_wt_for_downstream=use_wt)
    aw = _arrays(b, 62)
    dw = synthetic_dense(b, seed=62)
    gw, seq_w, prop_w = graph_batch(aw, DEV), dw["seq"].to(DEV), dw["prop"].to(DEV)
    args = ((c["g"], gw), (c["seq"], seq_w), (c["prop"], prop_w))
    calls = []
    c["model"].sample_eps = lambda like: calls.append(like.shape[0]) or torch.randn(
        like.shape, generator=torch.Generator().manual_seed(70 + len(calls))).to(like.device)
    s_c, s_w = _sigma(c["arr"], 63), _sigma(aw, 64, zero_every=3)
    names, res = _names(lambda: coordinate_ensemble_pair(
        c["model"], *args, sigma=(s_c.to(DEV), s_w.to(DEV) if perturb_wt else None), structures=m_count, seed=SEED,
        samples=2, max_graphs=25), monkeypatch)
    assert calls == [2 * b] * (2 if use_wt else 1)                        # no wild-type draw without use_wt
    assert names.count("is_coord_noise_expand") == len(scan_passes(m_count, b, 25)) * (2 if perturb_wt else 1)
    assert names.count("is_vae_mid_infer") == (2 if use_wt else 1)
    draws = [torch.randn(2 * b, 32, generator=torch.Generator().manual_seed(70 + i)).reshape(2, b, 32).to(DEV)
             for i in range(1, 3)]
    del c["model"].sample_eps
    for m in range(m_count):
        gc_m = graph_batch(dict(c["arr"], x=_expand(c["arr"], s_c, SEED, 0, m, 1)), DEV)
        gw_m = graph_batch(dict(aw, x=_expand(aw, s_w, SEED, 1, m, 1)), DEV) if perturb_wt else gw
        for k in range(2):
            inject_eps(c["model"], draws[0][k], draws[1][k] if use_wt else torch.zeros(b, 32))
            with torch.no_grad():
                ref = c["model"].forward_comparative((gc_m, gw_m), (c["seq"], seq_w), (c["prop"], prop_w))[4].reshape(-1)
            _close(res.logits[:, m, k], ref, BATCH_TOL)
    del c["model"].sample_eps
    ref_base = predictive_pair(c["model"], *args, eps=(draws[0], draws[1] if use_wt else None))
    assert torch.equal(res.base.logits, ref_base.logits)
    if not use_wt:
        with pytest.raises(ValueError, match="use_wt_for_downstream"):
            coordinate_ensemble_pair(c["model"], *args, sigma=(s_c.to(DEV), 1.0))
