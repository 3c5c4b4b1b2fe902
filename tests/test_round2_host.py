"""Host logic of the round-2 components on CPU (``_C`` monkeypatched with the kernel contracts): segment pooling,
the contrastive module's BatchNorm bookkeeping, the fused Adam wrapper against torch.optim, flat gradients and the
bucketed reducer's hook path (world_size 2, gloo), the augmentations' composite, and the PyG-free graph ingest."""
import copy
import os
import socket
import sys
import types

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

import immunostruct_b200 as I
from immunostruct_b200 import _C, augment, ingest, trunk
from immunostruct_b200 import functional as IF
from immunostruct_b200.optim import FusedAdam, FusedAdamW, flatten_gradients
from oracle import kernel_contracts as KC
from oracle import reference_ops as R

from conftest import load_golden, rel_err
from helpers import graph_batch


@pytest.fixture
def cpu_backend(monkeypatch):
    for name in KC.ALL:
        monkeypatch.setattr(_C, name, getattr(KC, name))
    monkeypatch.setattr(trunk, "_require_device_batch", lambda g: None)
    monkeypatch.setattr(augment, "_x", lambda b: b.ndata["x"])
    yield


# ---- segment pooling -----------------------------------------------------------------------------
def test_segment_pool_modes_and_tie_gradient(cpu_backend):
    off = torch.tensor([0, 3, 3, 7])                        # ragged, with an empty segment
    x = torch.tensor([[1., 5.], [4., 5.], [4., 0.], [2., 2.], [9., 2.], [0., 2.], [9., 1.]], requires_grad=True)
    mx = IF.segment_pool(off, x, "max")
    assert mx.tolist() == [[4., 5.], [0., 0.], [9., 2.]]
    mx.sum().backward()
    # ties share the gradient evenly (scatter_reduce 'amax')
    want = torch.tensor([[0., .5], [.5, .5], [.5, 0.], [0., 1 / 3], [.5, 1 / 3], [0., 1 / 3], [.5, 0.]])
    assert torch.allclose(x.grad, want, atol=1e-7)
    mean = IF.segment_pool(off, x.detach(), "mean")
    assert torch.allclose(mean[0], x[:3].mean(0).detach()) and mean[1].abs().sum() == 0
    assert torch.allclose(IF.segment_pool(off, x.detach(), "sum")[2], x[3:].sum(0).detach())
    assert torch.allclose(mean, R.global_mean_pool(x.detach(), torch.tensor([0, 0, 0, 2, 2, 2, 2]))[:3])


# ---- contrastive module ----------------------------------------------------------------------------
def test_contrastive_module_matches_reference_module_including_bn_buffers(cpu_backend):
    """The reference's PairedContrastiveLoss as stored in comparative_v2.npz (tests/golden/make_golden.py): its initial
    state_dict, the embeddings it was called on and the loss it returned.  Over two further steps on seeded inputs the
    BatchNorm buffers are held to a default torch.nn.BatchNorm1d (the reference's projector module, run in fp64 on the
    cancer, then the wild-type projection, as the reference's forward calls it), losses and gradients to fp64 autograd of the restatement
    (oracle/reference_ops.py paired_contrastive, itself checked against the same stored loss in tests/test_oracle.py)."""
    gd = load_golden("comparative_v2")
    state = gd["projector"]
    mine = I.PairedContrastiveLoss(embedding_dim=104)
    mine.load_state_dict(state)
    assert rel_err(mine(gd["out"]["emb_c"], gd["out"]["emb_w"], gd["dense"]["target"]), gd["out"]["loss_contrastive"]) < 1e-5

    mine = I.PairedContrastiveLoss(embedding_dim=104)
    mine.load_state_dict(state)
    bn = torch.nn.Sequential(torch.nn.Linear(104, 128, bias=False), torch.nn.BatchNorm1d(128)).double()
    bn.load_state_dict({k[len("projector."):]: v for k, v in state.items() if k.startswith(("projector.0.", "projector.1."))})
    p64 = {k: v.double().requires_grad_(True) for k, v in state.items() if k.endswith(("weight", "bias"))}
    torch.manual_seed(5)
    ec, ew = torch.randn(12, 104) * 2, torch.randn(12, 104) * 2
    t = (torch.arange(12) % 3 == 0).float()
    e1, e2 = ec.double().requires_grad_(True), ew.double().requires_grad_(True)
    f1, f2 = ec.clone().requires_grad_(True), ew.clone().requires_grad_(True)
    l_ref = R.paired_contrastive(p64, e1, e2, t)
    for step in range(2):                                   # two steps: running statistics accumulate
        l_mine = mine(f1, f2, t)
        bn(ec.double()), bn(ew.double())
        assert rel_err(l_mine, l_ref) < 1e-5
    l_ref.backward(); l_mine.backward()
    assert rel_err(f1.grad, e1.grad) < 1e-4 and rel_err(f2.grad, e2.grad) < 1e-4
    ref_state = {"projector." + k: v for k, v in bn.state_dict().items()}
    for k, a in mine.state_dict().items():
        b = ref_state.get(k, state[k])
        assert torch.allclose(a.double(), b.double(), rtol=1e-5, atol=1e-6), k
    assert int(mine.projector[1].num_batches_tracked) == 4
    for k, p in mine.named_parameters():
        assert rel_err(p.grad, p64[k].grad) < 1e-4, k
    # gated-off batches leave the BatchNorm buffers alone, like the reference (which returns before the projector)
    before = copy.deepcopy(mine.state_dict())
    assert float(mine(f1, f2, torch.ones(12))) == 0.0
    for k, v in mine.state_dict().items():
        assert torch.equal(v, before[k]), k
    # a single pair cannot hold two classes: zero, nothing launched (reference: python 0)
    assert float(mine(f1[:1], f2[:1], t[:1])) == 0.0


# ---- fused Adam ------------------------------------------------------------------------------------
def _toy(seed=0):
    torch.manual_seed(seed)
    return torch.nn.Sequential(torch.nn.Linear(7, 5), torch.nn.Tanh(), torch.nn.Linear(5, 3), torch.nn.Linear(3, 3))


@pytest.mark.parametrize("capturable", [False, True])
@pytest.mark.parametrize("decoupled,wd", [(False, 0.0), (False, 1e-2), (True, 1e-2)])
def test_fused_adam_matches_torch_and_skips_gradless_parameters(cpu_backend, decoupled, wd, capturable):
    a, b = _toy(), _toy()
    opt_t = (torch.optim.AdamW if decoupled else torch.optim.Adam)(a.parameters(), lr=1e-2, weight_decay=wd)
    opt_f = (FusedAdamW if decoupled else FusedAdam)(b.parameters(), lr=1e-2, weight_decay=wd, capturable=capturable)
    sched_t = torch.optim.lr_scheduler.StepLR(opt_t, 2, 0.5)
    sched_f = torch.optim.lr_scheduler.StepLR(opt_f, 2, 0.5)
    x = torch.randn(16, 7)
    unused_before = b[3].weight.detach().clone()
    for step in range(5):
        for m, o in ((a, opt_t), (b, opt_f)):
            o.zero_grad()
            m[2](m[1](m[0](x))).pow(2).mean().backward()       # m[3] unused: grad None
            o.step()
        sched_t.step(); sched_f.step()
    for (k, p), (_, q) in zip(b.named_parameters(), a.named_parameters()):
        assert torch.allclose(p, q, rtol=1e-5, atol=1e-7), k
    assert b[3].weight.grad is None and torch.equal(b[3].weight, unused_before)      # never touched (no decay either)
    # parameters are views of one flat buffer; state_dict round-trips; optimizer state uses torch's keys
    sd = b.state_dict()
    c = _toy(1); c.load_state_dict(sd)
    assert torch.equal(c[0].weight, b[0].weight)
    st = opt_f.state[b[0].weight]
    assert set(st) == {"step", "exp_avg", "exp_avg_sq"}
    assert float(st["step"]) == 5 if not capturable else float(opt_f._flat[0]["step_dev"]) == 5
    assert torch.allclose(st["exp_avg"], opt_t.state[a[0].weight]["exp_avg"], rtol=1e-5, atol=1e-8)


def test_flat_gradients_gather_point_and_sharing(cpu_backend):
    m = _toy()
    x = torch.randn(4, 7)
    m[2](m[0](x)).sum().backward()
    fg = flatten_gradients(m.parameters())
    assert flatten_gradients(m.parameters()) is fg                 # one object per live parameter set
    assert [p is q for p, q in zip(fg.params, [m[2].bias, m[2].weight, m[0].bias, m[0].weight])] == [True] * 4
    g0 = m[0].weight.grad.clone()
    assert m[0].weight.grad.data_ptr() != fg.views[3].data_ptr()   # not aliased by default
    fg.gather()
    assert torch.equal(fg.views[3], g0)
    fg.point()
    assert m[0].weight.grad.data_ptr() == fg.views[3].data_ptr()
    m.zero_grad(set_to_none=True)
    m[2](m[0](2 * x)).sum().backward()                             # fresh .grad tensors again
    fg.gather([3])                                                 # a single slot
    assert torch.equal(fg.views[3], m[0].weight.grad) and not torch.equal(fg.views[1], m[2].weight.grad)
    fg.realias()
    assert all(p.grad.data_ptr() == v.data_ptr() for p, v in zip(fg.params, fg.views))


def _reducer_worker(rank, world, port, q):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    from immunostruct_b200.distributed import BucketedGradientReducer, broadcast_parameters, shard_range
    torch.manual_seed(7)
    model = torch.nn.Sequential(torch.nn.Linear(6, 8), torch.nn.Tanh(), torch.nn.Linear(8, 4), torch.nn.Linear(4, 4))
    broadcast_parameters(model)
    red = BucketedGradientReducer(model.parameters(), bucket_bytes=64)     # several buckets
    data = torch.arange(48, dtype=torch.float32).reshape(8, 6) / 10
    lo, hi = shard_range(8, rank, world)
    out = []
    for step in range(3):
        if step == 2:
            model.zero_grad(set_to_none=True)              # default torch behaviour: fresh .grad tensors
        else:
            red.zero_grad() if step else None
        (model[2](model[1](model[0](data[lo:hi] + step))).pow(2).sum() / 8).backward()
        red.step()
        # plain lists: tensors would travel as file descriptors that die with this process
        out.append((model[0].weight.grad.tolist(), model[2].bias.grad.tolist(), red.overlapped_last_step, len(red.buckets)))
    q.put((rank, out, model[3].weight.grad is None))
    dist.barrier()
    dist.destroy_process_group()


def test_bucketed_reducer_overlaps_and_matches_full_batch_world2_gloo():
    s = socket.socket(); s.bind(("127.0.0.1", 0)); port = s.getsockname()[1]; s.close()
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    procs = [ctx.Process(target=_reducer_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    res = sorted([q.get(timeout=180) for _ in procs], key=lambda t: t[0])
    for p in procs:
        p.join(60)
        assert p.exitcode == 0
    torch.manual_seed(7)
    model = torch.nn.Sequential(torch.nn.Linear(6, 8), torch.nn.Tanh(), torch.nn.Linear(8, 4), torch.nn.Linear(4, 4))
    data = torch.arange(48, dtype=torch.float32).reshape(8, 6) / 10
    for step in range(3):
        model.zero_grad()
        (model[2](model[1](model[0](data + step))).pow(2).sum() / 8).backward()
        for r in range(2):
            gw, gb, overlapped, nb = res[r][1][step]
            assert torch.allclose(torch.tensor(gw) * 2, model[0].weight.grad, rtol=1e-5, atol=1e-6)
            assert torch.allclose(torch.tensor(gb) * 2, model[2].bias.grad, rtol=1e-5, atol=1e-6)
            assert nb >= 2
            assert overlapped == (0 if step == 0 else nb)       # from step 2 on every bucket is launched from a hook
    assert res[0][2] and res[1][2]                               # unused layer: grad stays None


# ---- augmentations ---------------------------------------------------------------------------------
def _toy_batch():
    from immunostruct_b200.synthetic import synthetic_graph_arrays
    arr = synthetic_graph_arrays(3, 12, 3, seed=3, n_pad=2)
    return graph_batch(arr)


def test_train_augment_composite_on_contracts(cpu_backend):
    gb = _toy_batch()
    x0 = gb.ndata["x"].clone()
    g = torch.Generator().manual_seed(11)
    seq = torch.nn.functional.one_hot(torch.randint(0, 20, (3, 30)), 21).float()
    seq0 = seq.clone()
    q = augment.random_rotation_(gb, g, return_q=True)
    assert torch.allclose(q @ q.transpose(1, 2), torch.eye(3).expand(3, 3, 3), atol=1e-5)
    off = gb.node_off.tolist()
    for i in range(3):
        a, b = off[i], off[i + 1]
        assert torch.allclose(gb.ndata["x"][a:b, 20:], x0[a:b, 20:] @ q[i], atol=1e-5)
        # rotations preserve pairwise distances
        assert torch.allclose(torch.cdist(gb.ndata["x"][a:b, 20:], gb.ndata["x"][a:b, 20:]), torch.cdist(x0[a:b, 20:], x0[a:b, 20:]), atol=1e-3)
    aa = augment.mask_single_structure_(gb, generator=g)
    ones_rows = (gb.ndata["x"][:, :20].sum(1) == 20).nonzero().flatten()
    assert ones_rows.numel() == 3
    for i, r in enumerate(ones_rows.tolist()):
        assert off[i] <= r < off[i + 1] and int(x0[r, :20].argmax()) == int(aa[i]) and x0[r, :20].sum() == 1
    augment.mask_structure_(gb, 2, g)
    zeroed = ((gb.ndata["x"][:, :20].sum(1) == 0) & (x0[:, :20].sum(1) == 1)).nonzero().flatten()
    assert 3 * 2 - 3 <= zeroed.numel() <= 3 * 2           # padded / SSL-masked picks change nothing
    # sequence masking: 3 distinct positions among the first 30 - 9 rows become the padding token
    augment.mask_sequence_(seq, 9, 3, generator=g)
    changed = (seq != seq0).any(-1)
    assert changed[:, 21:].sum() == 0 and bool((seq[changed].argmax(-1) == 20).all())
    assert bool(((seq.argmax(-1) == 20).sum(1) == 3).all())
    # the composite applies the same steps in the reference's order and hands back the SSL targets
    gb2 = _toy_batch()
    aug = I.TrainAugment(structure_pad_count=2, sequence_pad_count=3, return_amino_acid=True, peptide_len=9,
                         generator=torch.Generator().manual_seed(11))
    seq2 = seq0.clone()
    _, _, aa2 = aug(gb2, seq2)
    assert torch.equal(aa2, aa) and torch.equal(gb2.ndata["x"], gb.ndata["x"]) and torch.equal(seq2, seq)


def test_pair_masking_picks_the_same_residue_type(cpu_backend):
    gc, gw = _toy_batch(), _toy_batch()
    gw.ndata["x"][:, :20] = gw.ndata["x"][:, :20].roll(5, 0)
    xw0 = gw.ndata["x"].clone()
    aa = augment.mask_single_structure_(gc, gw, torch.Generator().manual_seed(2))
    off = gw.node_off.tolist()
    for i in range(3):
        rows = (gw.ndata["x"][off[i]:off[i + 1], :20].sum(1) == 20).nonzero().flatten()
        if rows.numel():
            assert int(xw0[off[i] + int(rows[0]), :20].argmax()) == int(aa[i])


# ---- PyG-free ingest ---------------------------------------------------------------------------------
def _write_fake_pyg_files(tmp_path):
    """Pickle graphs with stand-in torch_geometric classes laid out like PyG 2.5.3's (Data -> _store ->
    GlobalStorage._mapping, storage pickled with its parent), in a subprocess-free way: the fake modules are
    registered only while writing and removed before reading."""
    tg = types.ModuleType("torch_geometric")
    tgd = types.ModuleType("torch_geometric.data")
    tgdd = types.ModuleType("torch_geometric.data.data")
    tgds = types.ModuleType("torch_geometric.data.storage")

    class GlobalStorage:
        def __init__(self, parent, **kw):
            self._mapping = dict(kw)
            self._parent = parent

        def __getstate__(self):
            return dict(self.__dict__)

    class Data:
        def __init__(self, **kw):
            self.__dict__["_edge_attr_cls"] = GlobalStorage
            self.__dict__["_tensor_attr_cls"] = GlobalStorage
            self.__dict__["_store"] = GlobalStorage(self, **kw)

    GlobalStorage.__module__, GlobalStorage.__qualname__ = "torch_geometric.data.storage", "GlobalStorage"
    Data.__module__, Data.__qualname__ = "torch_geometric.data.data", "Data"
    tgds.GlobalStorage, tgdd.Data = GlobalStorage, Data
    mods = {"torch_geometric": tg, "torch_geometric.data": tgd, "torch_geometric.data.data": tgdd,
            "torch_geometric.data.storage": tgds}
    sys.modules.update(mods)
    try:
        gen = torch.Generator().manual_seed(0)
        specs = [("0_ImmunoAAAPEPTIDE_HLA-A0201", 7), ("1_ImmunoCCCPEPTIDE_HLA-B0702", 5),
                 ("2_ImmunoAAAPEPTIDE_HLA-A0201", 6),        # duplicate key -> dropped
                 ("3_ImmunoNXVPMVATV_HLA-A0201", 4)]         # filtered name
        for name, n in specs:
            x = torch.zeros(n, 22)
            x[torch.arange(n), torch.randint(0, 20, (n,), generator=gen)] = 1
            x[:, 20:] = torch.rand(n, 2, generator=gen)
            d = Data(x=x, coords=torch.randn(n, 3, generator=gen), name=name, num_nodes=n,
                     edge_index=torch.stack([torch.arange(n - 1), torch.arange(1, n)]), node_id=[f"A:{i}" for i in range(n)])
            torch.save(d, os.path.join(tmp_path, name + ".pt"))
    finally:
        for k in mods:
            sys.modules.pop(k, None)


def test_ingest_reads_pyg_pickles_without_torch_geometric(tmp_path):
    _write_fake_pyg_files(tmp_path)
    assert "torch_geometric" not in sys.modules
    files = sorted(f for f in os.listdir(tmp_path) if f.endswith(".pt"))
    graphs = ingest.preprocess_graphs(str(tmp_path), files)
    assert "torch_geometric" not in sys.modules
    assert [g.name for g in graphs] == ["0_ImmunoAAAPEPTIDE_HLA-A0201", "1_ImmunoCCCPEPTIDE_HLA-B0702"]
    assert graphs[0].x.shape == (7, 20) and graphs[0].coords.shape == (7, 3) and graphs[0].num_nodes == 7
    mapper = {g.name.split("Immuno")[1]: ingest.append_coords(g) for g in graphs}
    dgl_graphs = ingest.preprocess_graph(mapper, 23, 3)
    g0, g1 = dgl_graphs["AAAPEPTIDE_HLA-A0201"], dgl_graphs["CCCPEPTIDE_HLA-B0702"]
    assert g0.num_nodes() == g1.num_nodes() == 7                       # padded to the set's maximum
    assert g1.ndata["x"].shape == (7, 23) and g1.ndata["x"][5:].abs().sum() == 0 and g1.ndata["x"].dtype == torch.float32
    assert g1.num_edges() == 4 and g1.edata["edge_attr"].shape == (4, 1) and bool((g1.edata["edge_attr"] == 1).all())
    s, d = g1.edges()
    assert s.tolist() == [0, 1, 2, 3] and d.tolist() == [1, 2, 3, 4]    # directed exactly as stored
    batch = I.batch([g0, g1])                                          # feeds the normal collate path
    assert batch.n_nodes == 14 and batch.n_edges == 10 and batch.max_nodes == 7
    with pytest.raises(ValueError):
        ingest.pad_graph(ingest.PygData(x=torch.zeros(3, 22), coords=torch.zeros(3, 3), edge_index=torch.zeros(2, 0, dtype=torch.long)), 5, 23, 3)
