"""Structural uncertainty (immunostruct_b200/coordnoise.py), host logic on CPU: the contract of the expansion kernel
(is_coord_noise_expand: numpy uint32 Philox4x32-10, fp64 Box-Muller rounded to fp32) against the Random123 known-answer
vectors, the independence of its streams, the layout of r copies, the distribution of its normals, every error raised
before a kernel call, the pass split, and whole runs through the per-kernel contracts against the fp64 oracle's forward
on each contract-perturbed batch, single and pair.  The device kernel is checked in tests/test_coordnoise_gpu.py, which
shares ``coord_noise_expand_contract``."""
import numpy as np
import pytest
import torch
from scipy import stats

import immunostruct_b200 as I
from immunostruct_b200 import _C, trunk
from immunostruct_b200.coordnoise import coordinate_ensemble, coordinate_ensemble_pair
from immunostruct_b200.resident import scan_passes
from oracle import kernel_contracts as KC
from oracle import reference_ops as R

from conftest import load_golden, oracle_graph, rel_err
from helpers import build_model, graph_batch
from test_predictive_host import _comparative, head_mc_infer_contract

TOL = 1e-4
_M0, _M1 = np.uint64(0xD2511F53), np.uint64(0xCD9E8D57)
_W0, _W1 = 0x9E3779B9, 0xBB67AE85
_LO = np.uint64(0xFFFFFFFF)


# ---- the kernel's contract ----------------------------------------------------------------------------------------------
def philox4x32_10(counter, key):
    """Philox4x32-10 (Salmon et al. 2011) on uint32 arrays: counter = four arrays (or ints) broadcast together, key = two
    ints -> four uint32 arrays."""
    c = [np.asarray(v, dtype=np.uint32) for v in np.broadcast_arrays(*[np.asarray(v, dtype=np.uint32) for v in counter])]
    k0, k1 = int(key[0]), int(key[1])
    for rnd in range(10):
        if rnd:
            k0, k1 = (k0 + _W0) & 0xFFFFFFFF, (k1 + _W1) & 0xFFFFFFFF
        p0, p1 = c[0].astype(np.uint64) * _M0, c[2].astype(np.uint64) * _M1
        c = [(p1 >> np.uint64(32)).astype(np.uint32) ^ c[1] ^ np.uint32(k0), (p1 & _LO).astype(np.uint32),
             (p0 >> np.uint64(32)).astype(np.uint32) ^ c[3] ^ np.uint32(k1), (p0 & _LO).astype(np.uint32)]
    return c


def uniforms(v):
    """u = ((v >> 8) + 0.5) 2^-24 as the kernel forms it: (2 (v >> 8) + 1) rounded to fp32 once, times 2^-25."""
    return (((v >> np.uint32(8)) << np.uint32(1)) | np.uint32(1)).astype(np.float32) * np.float32(2.0 ** -25)


def normals(seed, item, m, b, a):
    """z [.., 3] of the stream keys (seed, item, m, b, a) (arrays broadcast), fp64 Box-Muller on the fp32 uniforms, in
    fp64 (the kernel differs by the rounding of logf, sqrtf, sincospif and one product)."""
    v = philox4x32_10((a, b, m, item), (seed & 0xFFFFFFFF, seed >> 32))
    u = [uniforms(w).astype(np.float64) for w in v]
    r0, r2 = np.sqrt(-2.0 * np.log(u[0])), np.sqrt(-2.0 * np.log(u[2]))
    return np.stack([r0 * np.cos(2.0 * np.pi * u[1]), r0 * np.sin(2.0 * np.pi * u[1]), r2 * np.cos(2.0 * np.pi * u[3])], -1)


def coord_noise_expand_contract(x23, node_off, sigma, seed, item, draw0, x23_out):
    """Contract of is_coord_noise_expand (signature of ``_C.coord_noise_expand``): x23_out [r N, 23] = r copies of x23,
    copy k being structure draw m = draw0 + k; in copy k, columns 20..22 of graph-local row a of graph b with
    sigma != 0 become fp32(sigma z + x), z = ``normals(seed, item, m, b, a)`` rounded to fp32."""
    x = x23.detach().cpu().numpy()
    n = x.shape[0]
    r = x23_out.shape[0] // n
    off = node_off.cpu().numpy()
    counts = np.diff(off)
    b = np.repeat(np.arange(counts.size), counts)
    a = np.arange(n) - off[b]
    s = sigma.detach().cpu().numpy().astype(np.float64)
    out = np.tile(x, (r, 1))
    live = s != 0
    for k in range(r):
        z = normals(seed, item, draw0 + k, b[live], a[live]).astype(np.float32).astype(np.float64)
        rows = k * n + np.flatnonzero(live)
        out[rows, 20:] = (s[live, None] * z + x[live, 20:].astype(np.float64)).astype(np.float32)
    x23_out.copy_(torch.from_numpy(out))


def _offsets(counts):
    return torch.cat([torch.zeros(1, dtype=torch.int64), torch.as_tensor(counts, dtype=torch.int64).cumsum(0)])


def perturbed_batches(arr, sigma, seed, item, structures):
    """The contract's structure draws m = 0 .. M-1 of a graph-array batch, one graph-array dict each."""
    x = arr["x"].float()
    out = []
    for m in range(structures):
        xo = torch.empty_like(x)
        coord_noise_expand_contract(x, _offsets(arr["node_counts"]), sigma, seed, item, m, xo)
        out.append(dict(arr, x=xo))
    return out


def test_known_answer_vectors():
    cases = [((0, 0, 0, 0), (0, 0), (0x6627e8d5, 0xe169c58d, 0xbc57ac4c, 0x9b00dbd8)),
             ((0xffffffff,) * 4, (0xffffffff,) * 2, (0x408f276d, 0x41c83b0e, 0xa20bc7c6, 0x6d5451fd)),
             ((0x243f6a88, 0x85a308d3, 0x13198a2e, 0x03707344), (0xa4093822, 0x299f31d0),
              (0xd16cfe09, 0x94fdcceb, 0x5001e420, 0x24126ea1))]
    for ctr, key, want in cases:
        assert [int(v) for v in philox4x32_10(ctr, key)] == list(want)


def test_uniforms_exact_and_open():
    v = np.array([0, 255, 256, 0x7FFFFFFF, 0x80000000, 0xFFFFFFFF], dtype=np.uint32)
    u = uniforms(v).astype(np.float64)
    assert u[0] == u[1] == 2.0 ** -25 and u[2] == 3 * 2.0 ** -25
    assert (u > 0).all() and (u <= 1).all()
    exact = ((v >> 8).astype(np.float64) + 0.5) * 2.0 ** -24
    assert (u[exact < 0.5] == exact[exact < 0.5]).all()            # below 1/2 the uniform is exact
    assert (np.abs(u - exact) <= 2.0 ** -25).all()                  # above, one rounding of a 25-bit integer


def test_streams_are_distinct():
    a = np.arange(64)
    ref = philox4x32_10((a, 3, 5, 0), (7, 0))
    words = lambda ctr, key: np.stack(philox4x32_10(ctr, key), 1)
    base = np.stack(ref, 1)
    for ctr, key in [((a, 4, 5, 0), (7, 0)), ((a, 3, 6, 0), (7, 0)), ((a, 3, 5, 1), (7, 0)), ((a, 3, 5, 0), (8, 0)),
                     ((a, 3, 5, 0), (7, 1)), ((a + 1, 3, 5, 0), (7, 0))]:
        assert not (words(ctr, key) == base).all(1).any()
    assert len({tuple(w) for w in base.tolist()}) == a.size
    z = normals(2 ** 40 + 7, 0, 0, 0, np.arange(8))
    assert not np.allclose(z, normals(7, 0, 0, 0, np.arange(8)))    # the seed's high half is part of the key


def _hand_batch():
    counts = [5, 33, 1, 70]                                            # chunks of 32 rows: one, two and three per graph
    gen = torch.Generator().manual_seed(0)
    x = torch.randn(sum(counts), 23, generator=gen) * 10
    x[3, 20:] = torch.tensor([-0.0, 0.0, 1.5])
    return x, _offsets(counts), counts


@pytest.mark.parametrize("r,draw0", [(1, 0), (3, 0), (2, 5)])
def test_layout_of_r_copies(r, draw0):
    x, off, counts = _hand_batch()
    n = x.shape[0]
    sigma = torch.rand(n, generator=torch.Generator().manual_seed(1))
    sigma[[0, 3, 40, n - 1]] = 0.0
    out = torch.full((r * n, 23), float("nan"))
    coord_noise_expand_contract(x, off, sigma, 99, 0, draw0, out)
    for k in range(r):
        blk = out[k * n:(k + 1) * n]
        assert torch.equal(blk[:, :20], x[:, :20])
        zero = sigma == 0
        assert torch.equal(blk[zero].view(torch.int32), x[zero].view(torch.int32))   # -0.0 kept
        moved = (blk[~zero, 20:] - x[~zero, 20:]).abs()
        assert (moved > 0).all()
        one = torch.empty(n, 23)
        coord_noise_expand_contract(x, off, sigma, 99, 0, draw0 + k, one)             # copy k = draw draw0 + k alone
        assert torch.equal(blk, one)
        for row, b, a in ((37, 1, 32), (38, 2, 0), (41, 3, 2), (108, 3, 69)):   # graph-local rows key the stream
            z = normals(99, 0, draw0 + k, b, a).astype(np.float32).astype(np.float64)
            want = (float(sigma[row]) * z + x[row, 20:].double().numpy()).astype(np.float32)
            assert np.array_equal(blk[row, 20:].numpy(), want)


def test_normals_distribution():
    a, b = np.meshgrid(np.arange(1000), np.arange(100), indexing="ij")
    z = normals(123456789, 0, 0, b.reshape(-1), a.reshape(-1)).astype(np.float32).astype(np.float64)
    flat = z.reshape(-1)
    n = flat.size
    assert n == 300000
    assert abs(flat.mean()) < 5 / np.sqrt(n)
    assert abs(flat.var() - 1) < 5 * np.sqrt(2 / n)
    assert abs(stats.skew(flat)) < 5 * np.sqrt(6 / n) and abs(stats.kurtosis(flat)) < 5 * np.sqrt(24 / n)
    corr = np.corrcoef(z.T)
    assert np.abs(corr - np.eye(3)).max() < 5 / np.sqrt(z.shape[0])
    rows = z.reshape(1000, 100, 3)                                    # [a, b, 3]: neighbouring rows, then graphs
    for x0, x1 in ((rows[:-1], rows[1:]), (rows[:, :-1], rows[:, 1:])):
        assert abs(np.corrcoef(x0.reshape(-1), x1.reshape(-1))[0, 1]) < 5 / np.sqrt(x0.size)
    assert stats.kstest(flat, "norm").pvalue > 1e-3


# ---- whole runs through the kernel contracts ------------------------------------------------------------------------
@pytest.fixture
def cpu_backend(monkeypatch):
    for name in KC.ALL:
        monkeypatch.setattr(_C, name, getattr(KC, name))
    monkeypatch.setattr(_C, "head_mc_infer", head_mc_infer_contract)
    monkeypatch.setattr(_C, "coord_noise_expand", coord_noise_expand_contract)
    monkeypatch.setattr(trunk, "_require_device_batch", lambda g: None)
    yield


def test_errors_before_any_kernel_call(cpu_backend, monkeypatch):
    gd = load_golden("hybrid_v2")
    model = build_model("HybridModelv2", gd)
    d = gd["dense"]
    g = graph_batch(gd["graph"])
    gc = load_golden("comparative_v2")
    gcb, gwb = graph_batch(gc["graph_c"]), graph_batch(gc["graph_w"])         # collated before the count starts
    launched = []
    for name in ("coord_noise_expand", "head_mc_infer", "collate_csr", "linear_tc", "vae_mid_infer"):
        monkeypatch.setattr(_C, name, lambda *a, **k: launched.append(1))
    n = g.n_nodes

    def bad(exc, match, m=model, fn=coordinate_ensemble, sigma=0.5, **kw):
        with pytest.raises(exc, match=match):
            fn(m, g, d["seq"], d["prop"], sigma=sigma, **kw)

    neg = torch.full((n,), 0.5)
    neg[4] = -1e-3
    nan = torch.full((n,), 0.5)
    nan[7] = float("nan")
    for s in (-0.1, float("nan"), float("inf")):
        bad(ValueError, "finite and >= 0", sigma=s)
    for s in (neg, nan, torch.full((n,), float("inf"))):
        bad(ValueError, "finite and >= 0 in every row", sigma=s)
    for s in (torch.ones(n, dtype=torch.float64), torch.ones(n + 1), torch.ones(n, 1), [0.5] * n, True, None):
        bad(ValueError, "float32 tensor", sigma=s)
    for m in (0, -1, 2.0, True):
        bad(ValueError, "structures", structures=m)
    bad(ValueError, "structures", structures=2 ** 32 + 1)
    for sd in (-1, 2 ** 64, 1.5, True):
        bad(ValueError, "seed", seed=sd)
    bad(ValueError, "max_graphs", max_graphs=2)
    bad(ValueError, "samples", samples=0)
    bad(ValueError, "eps", eps=torch.zeros(2, 2, 32))
    for name in ("StructureModel", "StructureModelv2", "SequenceModel", "DualModel"):
        bad(NotImplementedError, "HybridModelv2_SSL", m=I.model_map[name](vae_input_dim=231, device="cpu").eval())
    model.train()
    bad(RuntimeError, "eval")
    model.eval()
    bad(NotImplementedError, "HybridModel_Comparative", fn=lambda m, g_, s_, p_, **kw: coordinate_ensemble_pair(
        m, (g_, g_), (s_, s_), (p_, p_), **kw), sigma=(0.5, None))
    for use_wt in (True, False):
        cm = _comparative(use_wt, gc)
        dc = gc["dense"]
        pair = lambda **kw: coordinate_ensemble_pair(cm, (gcb, gwb), (dc["seq_c"], dc["seq_w"]),
                                                     (dc["prop_c"], dc["prop_w"]), **kw)
        for s in (0.5, (0.5,), (None, 0.5), [0.5, 0.5, 0.5]):
            with pytest.raises(ValueError, match="pair"):
                pair(sigma=s)
        if use_wt:
            with pytest.raises(ValueError, match="sigma_w must be finite"):
                pair(sigma=(0.5, -1.0))
            with pytest.raises(ValueError, match="sigma_w"):
                pair(sigma=(0.5, torch.zeros(3)))
        else:
            with pytest.raises(ValueError, match="use_wt_for_downstream"):
                pair(sigma=(0.5, 0.5))
        with pytest.raises(ValueError, match="eps"):
            pair(sigma=(0.5, None), eps=torch.zeros(1, 4, 32))
        cm.train()
        with pytest.raises(RuntimeError, match="eval"):
            pair(sigma=(0.5, None))
    assert not launched


def _og64(arrays):
    g = oracle_graph(arrays)
    return dict(g, x=g["x"].double(), edge_attr=g["edge_attr"].double())


def _peptide_sigma(arr, rows, scale, seed):
    """Per-row sigma: random in [scale/2, scale) on the first ``rows`` rows of every graph, 0 elsewhere."""
    off = _offsets(arr["node_counts"])
    s = torch.zeros(int(off[-1]))
    gen = torch.Generator().manual_seed(seed)
    for b in range(arr["node_counts"].numel()):
        s[off[b]:off[b] + rows] = scale * (0.5 + 0.5 * torch.rand(rows, generator=gen))
    return s


def _check_statistics(res):
    p = torch.sigmoid(res.logits.double())
    b = p.shape[0]
    pf = p.reshape(b, -1)
    assert float((res.prob_mean.double() - pf.mean(1)).abs().max()) < 1e-7
    assert float((res.prob_std.double() - pf.std(1, unbiased=False)).abs().max()) < 1e-7
    assert float((res.std_structure.double() - p.mean(2).std(1, unbiased=False)).abs().max()) < 1e-7
    assert float((res.std_latent.double() - p.var(2, unbiased=False).mean(1).sqrt()).abs().max()) < 1e-7
    total = res.prob_std.double().square()
    split = res.std_structure.double().square() + res.std_latent.double().square()
    assert float((total - split).abs().max()) <= 1e-6 * float(total.max())   # the law of total variance


@pytest.mark.parametrize("max_graphs,sigma", [(4096, "rows"), (4, "rows"), (7, "scalar")])
def test_matches_fp64_oracle_per_structure(cpu_backend, max_graphs, sigma):
    gd = load_golden("hybrid_v2")
    model = build_model("HybridModelv2", gd)
    d = gd["dense"]
    arr = gd["graph"]
    g = graph_batch(arr)
    eps = torch.randn(2, 3, 32, generator=torch.Generator().manual_seed(3))
    s = _peptide_sigma(arr, 5, 1.5, 4) if sigma == "rows" else 0.8
    m_count = 5
    res = coordinate_ensemble(model, g, d["seq"], d["prop"], sigma=s, structures=m_count, seed=2 ** 40 + 11, eps=eps,
                              max_graphs=max_graphs)
    assert res.logits.shape == (3, m_count, 2) and res.seed == 2 ** 40 + 11
    s_rows = s if sigma == "rows" else torch.full((g.n_nodes,), 0.8)
    p64 = {k: v.detach().double() for k, v in model.state_dict().items()}
    for m, pert in enumerate(perturbed_batches(arr, s_rows, res.seed, 0, m_count)):
        for k in range(2):
            ref = R.hybrid_forward(p64, _og64(pert), d["seq"].double(), d["prop"].double(), eps[k].double(),
                                   version="v2", n_layers=int(gd["meta"]["gcn_layers"]))[3].reshape(-1)
            assert rel_err(res.logits[:, m, k], ref) < TOL, (m, k)
    spread = (res.logits - res.base.logits[:, None, :]).abs().max()
    assert float(spread) > 1e-4                                       # the coordinates reach the score
    _check_statistics(res)
    assert all(q.grad is None for q in model.parameters())


def test_pass_split_and_seed(cpu_backend, monkeypatch):
    gd = load_golden("hybrid_v2")
    model = build_model("HybridModelv2", gd)
    d = gd["dense"]
    g = graph_batch(gd["graph"])
    calls = []

    def expand(x23, node_off, sigma, seed, item, draw0, x23_out):
        coord_noise_expand_contract(x23, node_off, sigma, seed, item, draw0, x23_out)
        calls.append((draw0, x23_out.shape[0] // x23.shape[0], x23_out.clone()))

    monkeypatch.setattr(_C, "coord_noise_expand", expand)
    s = _peptide_sigma(gd["graph"], 4, 1.0, 5)
    eps = torch.randn(1, 3, 32, generator=torch.Generator().manual_seed(6))
    runs = {}
    for mg in (4096, 7, 3):
        calls.clear()
        runs[mg] = coordinate_ensemble(model, g, d["seq"], d["prop"], sigma=s, structures=10, seed=77, eps=eps,
                                       max_graphs=mg)
        assert [(j, r) for j, r, _ in calls] == scan_passes(10, 3, mg)
        assert [(j, r) for j, r, _ in calls] == {4096: [(0, 10)], 7: [(0, 2), (2, 2), (4, 2), (6, 2), (8, 2)],
                                                 3: [(j, 1) for j in range(10)]}[mg]
        runs[mg].coords = torch.cat([c for _, _, c in calls])
    for mg in (7, 3):
        assert torch.equal(runs[mg].coords, runs[4096].coords)        # a structure does not depend on the pass split
        assert rel_err(runs[mg].logits, runs[4096].logits) < 1e-6
    torch.manual_seed(5)
    one = coordinate_ensemble(model, g, d["seq"], d["prop"], sigma=s, structures=2, eps=eps)
    torch.manual_seed(5)
    two = coordinate_ensemble(model, g, d["seq"], d["prop"], sigma=s, structures=2, eps=eps)
    assert one.seed == two.seed and 0 <= one.seed < 2 ** 63 and torch.equal(one.logits, two.logits)
    other = coordinate_ensemble(model, g, d["seq"], d["prop"], sigma=s, structures=2, eps=eps, seed=one.seed + 1)
    assert not torch.equal(other.logits, one.logits)
    zero = coordinate_ensemble(model, g, d["seq"], d["prop"], sigma=0.0, structures=3, eps=eps)
    assert rel_err(zero.logits, zero.base.logits[:, None, :].expand(-1, 3, -1)) < 1e-6
    assert float(zero.std_structure.abs().max()) < 1e-7


@pytest.mark.parametrize("use_wt,sigma_w", [(True, "rows"), (True, None), (False, None)])
def test_pair_matches_fp64_oracle_and_draws_once_per_item(cpu_backend, monkeypatch, use_wt, sigma_w):
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
    s_c = _peptide_sigma(arr_c, 4, 1.2, 8)
    s_w = None if sigma_w is None else _peptide_sigma(arr_w, 6, 0.9, 9)
    expands = []
    monkeypatch.setattr(_C, "coord_noise_expand", lambda *a: expands.append(a[4]) or coord_noise_expand_contract(*a))
    m_count, seed = 3, 31337
    res = coordinate_ensemble_pair(model, (gc, gw), (d["seq_c"], d["seq_w"]), (d["prop_c"], d["prop_w"]),
                                   sigma=(s_c, s_w), structures=m_count, seed=seed, samples=2, max_graphs=4)
    b = arr_c["node_counts"].numel()
    assert expands == ([0, 1] if s_w is not None else [0]) * m_count    # one expansion per perturbed item and pass
    assert [tuple(c.shape) for c in calls] == [(2 * b, 32)] * (2 if use_wt else 1)
    eps_c = calls[0].reshape(2, b, 32)
    eps_w = calls[1].reshape(2, b, 32) if use_wt else torch.zeros(2, b, 32)
    pert_c = perturbed_batches(arr_c, s_c, seed, 0, m_count)
    pert_w = perturbed_batches(arr_w, s_w, seed, 1, m_count) if s_w is not None else [arr_w] * m_count
    p64 = {k: v.detach().double() for k, v in model.state_dict().items()}
    for m in range(m_count):
        for k in range(2):
            ref = R.comparative_forward(p64, (_og64(pert_c[m]), _og64(pert_w[m])),
                                        (d["seq_c"].double(), d["seq_w"].double()),
                                        (d["prop_c"].double(), d["prop_w"].double()),
                                        (eps_c[k].double(), eps_w[k].double()),
                                        n_layers=int(gd["meta"]["gcn_layers"]), use_wt=use_wt)[4].reshape(-1)
            assert rel_err(res.logits[:, m, k], ref) < TOL, (m, k)
    _check_statistics(res)
