"""Nearest neighbours in the classifier's feature space on the B200: the search kernels (is_knn) against the fp64
contract of tests/test_neighbors_host.py, bit-exact ties, slicing and subset invariance, exclude, NaN rows, the launch
sequence; the feature kernel (is_head_features_infer) against the models' own hidden layer in both tensor-core modes,
its determinism, its identity with the fused head, and an end-to-end self search."""
import pytest
import torch

import immunostruct_b200 as I
from immunostruct_b200 import _C
from immunostruct_b200.neighbors import embed, embed_pair, nearest
from immunostruct_b200.synthetic import split_graphs, synthetic_dense, synthetic_graph_arrays

from helpers import graph_batch
from test_neighbors_host import knn_contract

pytestmark = pytest.mark.gpu
DEV = "cuda"
TOL = 1e-5
BATCH_TOL = 1e-6


def _gen(seed):
    return torch.Generator().manual_seed(seed)


# ---- the search against its contract ----------------------------------------------------------------------------------
def _bound(d64, dim):
    """fp32 error bound of one pair's distance: D + 2 roundings of at most 2^-24 relative each (the difference, the
    fused square-add chain), with margin."""
    return 2 * (dim + 4) * 2.0 ** -24 * d64


def _check_contract(query, bank, k, idx, dist, exclude=None):
    n_q, dim = query.shape
    ref_i, ref_d = knn_contract(query, bank, k + 1, exclude)
    ref_i, ref_d, nxt = ref_i[:, :k], ref_d[:, :k], ref_d[:, k]
    assert idx.shape == (n_q, k) and dist.shape == (n_q, k) and idx.dtype == torch.int64 and dist.dtype == torch.float32
    filled = idx >= 0
    assert torch.equal(filled, ref_i >= 0)
    assert torch.isinf(dist[~filled]).all() and (dist[~filled] > 0).all()
    assert (dist[:, 1:] >= dist[:, :-1]).all()
    if exclude is not None:
        assert not ((idx == exclude[:, None]) & filled).any()
    # every returned row: its fp32 distance within the bound of its fp64 distance
    rows = bank.double()[idx.clamp_min(0)]
    own = ((query.double()[:, None, :] - rows) ** 2).sum(-1)
    assert ((dist.double() - own).abs() <= _bound(own, dim) + 1e-300)[filled].all()
    # the order statistics within the bound; the index wherever the fp64 gaps on both sides exceed twice the bound
    assert ((dist.double() - ref_d).abs() <= _bound(ref_d, dim) + 1e-300)[filled].all()
    both = torch.cat([ref_d, nxt[:, None]], 1)
    gap = both[:, 1:] - both[:, :-1]
    prev = torch.cat([torch.full_like(gap[:, :1], float("inf")), gap[:, :-1]], 1)
    clear = (torch.isinf(both[:, 1:]) | (gap > 2 * _bound(both[:, 1:], dim))) & (prev > 2 * _bound(ref_d, dim)) & filled
    assert torch.equal(idx[clear], ref_i[clear])
    return clear


@pytest.mark.parametrize("dim", [1, 32, 33, 104, 256])
@pytest.mark.parametrize("k", [1, 16, 64])
def test_search_against_contract(dim, k):
    g = _gen(dim * 100 + k)
    clear = total = 0
    for n_q in (1, 7, 129, 4099):
        for r in (1, 31, 128, 129, 30011):
            query = torch.randn(n_q, dim, generator=g).to(DEV)
            bank = torch.randn(r, dim, generator=g).to(DEV)
            res = nearest(query, bank, k)
            c = _check_contract(query, bank, k, res.index, res.distance)
            clear, total = clear + int(c.sum()), total + int((res.index >= 0).sum())
    assert clear >= 0.9 * total                  # the check above is not vacuous


def _integer_case(n_q, r, dim, seed, distinct=40):
    """Integer-valued features with many duplicate rows: every difference, square and partial sum is exact in fp32."""
    g = _gen(seed)
    rows = torch.randint(-3, 4, (distinct, dim), generator=g).float()
    bank = rows[torch.randint(0, distinct, (r,), generator=g)]
    query = torch.cat([rows, torch.randint(-3, 4, (max(0, n_q - distinct), dim), generator=g).float()])[:n_q]
    return query.to(DEV), bank.to(DEV)


@pytest.mark.parametrize("dim", [1, 33, 104])
@pytest.mark.parametrize("k", [1, 16, 64])
def test_exact_ties_bit_for_bit(dim, k):
    for n_q, r in ((7, 129), (4099, 30011)):
        query, bank = _integer_case(n_q, r, dim, seed=dim + k)
        ref_i, ref_d = knn_contract(query, bank, k)
        for s in sorted({1, min(3, _C.knn_max_slices(r)), _C.knn_max_slices(r)}):
            idx, dist = _C.knn(query, bank, k, slices=s)
            assert torch.equal(idx, ref_i), (n_q, r, s)
            assert torch.equal(dist, ref_d.float()), (n_q, r, s)


@pytest.mark.parametrize("integer", [False, True])
def test_slicing_and_subset_invariance(integer):
    dim, k, r = 32, 16, 30011
    if integer:
        query, bank = _integer_case(4099, r, dim, seed=5)
    else:
        g = _gen(6)
        query, bank = torch.randn(4099, dim, generator=g).to(DEV), torch.randn(r, dim, generator=g).to(DEV)
    runs = [_C.knn(query, bank, k, slices=s) for s in (1, 2, 7, _C.knn_max_slices(r))]
    for idx, dist in runs[1:]:
        assert torch.equal(idx, runs[0][0]) and torch.equal(dist, runs[0][1])
    g = _gen(7)
    for subset in ([0], [4098], [17, 3, 17], torch.randperm(4099, generator=g)[:129].tolist(),
                   torch.randperm(4099, generator=g)[:1000].tolist()):
        res = nearest(query[subset], bank, k)           # another Q: another tile layout and slice count
        assert torch.equal(res.index, runs[0][0][subset]) and torch.equal(res.distance, runs[0][1][subset])


def test_exclude_leave_self_out():
    g = _gen(8)
    bank = torch.randn(30011, 32, generator=g).to(DEV)
    ex = torch.arange(30011, device=DEV)
    res = nearest(bank, bank, 16, exclude=ex)
    _check_contract(bank, bank, 16, res.index, res.distance, ex)
    ref_i, _ = knn_contract(bank, bank, 17)
    assert torch.equal(ref_i[:, 0], ex)                # brute force: the diagonal first, then the same rows
    assert (res.index == ref_i[:, 1:]).float().mean() > 0.999
    # -1 entries exclude nothing, mixed with real ones
    plain = nearest(bank[:500], bank, 16)
    none = nearest(bank[:500], bank, 16, exclude=torch.full((500,), -1, device=DEV))
    assert torch.equal(plain.index, none.index) and torch.equal(plain.distance, none.distance)
    mixed = ex[:500].clone()
    mixed[::2] = -1
    res = nearest(bank[:500], bank, 16, exclude=mixed)
    assert torch.equal(res.index[::2], plain.index[::2])
    assert torch.equal(res.index[1::2, :15], plain.index[1::2, 1:])        # the own row (distance 0) left out


def test_nan_rows_and_queries():
    g = _gen(9)
    bank = torch.randn(3000, 33, generator=g)
    nan_rows = torch.randperm(3000, generator=g)[:400]
    bank[nan_rows, torch.randint(0, 33, (400,), generator=g)] = float("nan")
    query = torch.randn(300, 33, generator=g)
    query[::7, 5] = float("nan")
    query, bank = query.to(DEV), bank.to(DEV)
    for s in (1, 5):
        idx, dist = _C.knn(query, bank, 64, slices=s)
        assert not torch.isin(idx, nan_rows.to(DEV)).any()
        assert (idx[::7] == -1).all() and torch.isinf(dist[::7]).all()
        keep = torch.ones(300, dtype=torch.bool, device=DEV)
        keep[::7] = False
        _check_contract(query[keep], bank, 64, idx[keep], dist[keep])
    # fewer eligible rows than k: the rest is -1 / +inf
    idx, dist = _C.knn(query[1:2], bank[nan_rows[:10]].clone().index_fill_(0, torch.tensor([3], device=DEV), 0.0), 8)
    assert idx[0].tolist() == [3] + [-1] * 7 and torch.isinf(dist[0, 1:]).all()


def test_launches():
    g = _gen(10)
    bank = torch.randn(27000, 32, generator=g).to(DEV)
    for n_q, want in ((27000, ["knn_partial_kernel"]), (5, ["knn_partial_kernel", "knn_merge_kernel"])):
        query = bank[:n_q].contiguous()
        nearest(query, bank, 16)                                        # warm-up (module load)
        torch.cuda.synchronize()
        with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
            nearest(query, bank, 16)
            torch.cuda.synchronize()
        names = [e.name for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA and "knn" in e.name]
        assert len(names) == len(want) and all(any(w in n for n in names) for w in want), names


# ---- features ----------------------------------------------------------------------------------------------------------
@pytest.fixture
def precision(request):
    prev = I.get_precision()
    I.set_precision(request.param)
    yield request.param
    I.set_precision(prev)


def _close(got, ref, tol=TOL):
    ref = ref.detach().double().cpu()
    err = float((got.detach().double().cpu() - ref).abs().max())
    assert err <= tol * max(float(ref.abs().max()), 1e-30), (err, float(ref.abs().max()))


def _scaled(model, seed):
    """Scaled-up weights (the latent mean x 3, the classifier's input layer x 4): at default initialisation the hidden
    layer hardly depends on the input, and a comparison of features would pass vacuously."""
    torch.manual_seed(seed)
    with torch.no_grad():
        for name, p in model.named_parameters():
            if name in ("vae_fc21.weight", "vae_fc21.bias"):
                p.mul_(3.0)
            if name == "classifier.1.weight":
                p.mul_(4.0)
    I.invalidate_caches()
    return model.eval()


def _case(b, seed, name, **kw):
    arr = synthetic_graph_arrays(b, 200, 10, seed=seed, n_pad=10)
    dense = synthetic_dense(b, seed=seed)
    torch.manual_seed(seed)
    model = _scaled(I.model_map[name](vae_input_dim=5943, device=DEV, **kw).to(DEV), seed)
    return graph_batch(arr, DEV), arr, dense["seq"].to(DEV), dense["prop"].to(DEV), model


def _module_hidden(model, fn):
    """The classifier's hidden layer of the model's own module path, with the latent at its mean."""
    got = []
    h = model.classifier[2].register_forward_hook(lambda m, i, o: got.append(o.detach().clone()))
    model.reparameterize = lambda mu, logvar: mu
    try:
        with torch.no_grad():
            fn()
    finally:
        h.remove()
        del model.reparameterize
    assert len(got) == 1
    return got[0]


def _varies(f):
    """The features are not (nearly) constant over the batch."""
    assert float(f.std(0).max()) > 1e-2 * float(f.abs().max())


SINGLE = ["HybridModel", "HybridModelv2", "HybridModel_SSL", "HybridModelv2_SSL", "HybridModel_Comparative",
          "HybridModel_Comparative_SSL", "HybridModelv2_Comparative", "HybridModelv2_Comparative_SSL"]


@pytest.mark.parametrize("precision", ["fp16x2", "bf16x3"], indirect=True)
@pytest.mark.parametrize("name", SINGLE)
def test_embed_matches_the_module_hidden_layer(precision, name):
    g, _, seq, prop, model = _case(64, 11, name)
    f = embed(model, g, seq, prop)
    assert f.shape == (64, 32) and f.dtype == torch.float32
    ref = _module_hidden(model, lambda: model(g, seq, prop))
    _close(f, ref)
    _varies(f)


@pytest.mark.parametrize("precision", ["fp16x2", "bf16x3"], indirect=True)
@pytest.mark.parametrize("name", ["HybridModel_Comparative", "HybridModelv2_Comparative_SSL"])
@pytest.mark.parametrize("use_wt", [True, False])
def test_embed_pair_matches_forward_comparative(precision, name, use_wt):
    gc, _, seq_c, prop_c, model = _case(48, 21, name, use_wt_for_downstream=use_wt)
    arr_w = synthetic_graph_arrays(48, 200, 10, seed=22, n_pad=10)
    dw = synthetic_dense(48, seed=22)
    gw, seq_w, prop_w = graph_batch(arr_w, DEV), dw["seq"].to(DEV), dw["prop"].to(DEV)
    f = embed_pair(model, (gc, gw), (seq_c, seq_w), (prop_c, prop_w))
    ref = _module_hidden(model, lambda: model.forward_comparative((gc, gw), (seq_c, seq_w), (prop_c, prop_w)))
    _close(f, ref)
    _varies(f)
    if not use_wt:                                   # the wild type is not read
        assert torch.equal(f, embed_pair(model, (gc, None), (seq_c, None), (prop_c, None)))


def _arrays_of(graphs):
    cat = lambda key: torch.cat([gr[key] for gr in graphs])
    return {"x": cat("x"), "src": cat("src"), "dst": cat("dst"), "edge_attr": cat("edge_attr"),
            "node_counts": torch.tensor([gr["num_nodes"] for gr in graphs]),
            "edge_counts": torch.tensor([gr["src"].numel() for gr in graphs])}


def test_embed_is_deterministic_and_batch_independent():
    g, arr, seq, prop, model = _case(96, 31, "HybridModelv2")
    f = embed(model, g, seq, prop)
    assert torch.equal(f, embed(model, g, seq, prop))
    order = list(range(95, -1, -3))                  # another batch: a subset in another order
    g2 = graph_batch(_arrays_of([split_graphs(arr)[i] for i in order]), DEV)
    _close(embed(model, g2, seq[order], prop[order]), f[order], BATCH_TOL)


@pytest.mark.parametrize("name", ["HybridModel", "HybridModelv2", "HybridModel_SSL", "HybridModelv2_SSL"])
def test_feature_kernel_equals_the_fused_head(name):
    from immunostruct_b200.predictive import _encode, _head_params
    g, _, seq, prop, model = _case(40, 41, name)
    with torch.no_grad():
        pooled, mu, _, zv = _encode(model, g, seq, prop)
        wc, bc, coef, n_head, w1, b1, _, _ = _head_params(model)
        _, hid = _C.head_infer(pooled, wc, bc, zv, coef, n_head, w1, b1, None, None)
        assert torch.equal(_C.head_features_infer([(pooled, mu, zv)], wc, bc, coef, n_head, w1, b1), hid)
    assert torch.equal(embed(model, g, seq, prop), hid)


def test_self_search_end_to_end():
    g, arr, seq, prop, model = _case(200, 51, "HybridModelv2")
    f = embed(model, g, seq, prop)
    res = nearest(f, f, 4)
    own = torch.arange(200, device=DEV)
    dup = (f[:, None, :] == f[None, :, :]).all(-1).sum(1) > 1            # identical feature rows tie at 0.0
    assert torch.equal(res.index[~dup, 0], own[~dup])
    assert (res.distance[:, 0] == 0.0).all()
    left = nearest(f, f, 3, exclude=own)
    assert (left.index != own[:, None]).all()
    assert torch.equal(left.index[~dup], res.index[~dup, 1:]) and torch.equal(left.distance[~dup], res.distance[~dup, 1:])


def test_embed_needs_eval_and_leaves_grads():
    g, _, seq, prop, model = _case(8, 61, "HybridModelv2_Comparative")
    for p in model.parameters():
        p.grad = torch.full_like(p, 0.5)
    before = {n: p.grad.clone() for n, p in model.named_parameters()}
    with torch.enable_grad():
        f = embed(model, g, seq, prop)
        embed_pair(model, (g, g), (seq, seq), (prop, prop))
    assert not f.requires_grad
    assert all(torch.equal(p.grad, before[n]) for n, p in model.named_parameters())
    model.train()
    with pytest.raises(RuntimeError, match="eval"):
        embed(model, g, seq, prop)
    with pytest.raises(RuntimeError, match="eval"):
        embed_pair(model, (g, g), (seq, seq), (prop, prop))
