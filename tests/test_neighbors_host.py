"""Nearest neighbours in the classifier's feature space (immunostruct_b200/neighbors.py), host side: the search contract
restated in fp64 (``knn_contract``) on hand cases, every argument rule of ``nearest`` and of the ``_C.knn`` binding
raised before anything is enqueued, the argument rules of ``embed`` / ``embed_pair``, and the SASS of the existing head
kernels pinned against the feature kernel's addition.  The device search is checked against the same contract in
tests/test_neighbors_gpu.py."""
import hashlib
import json
import os
import re
import shutil
import subprocess

import pytest
import torch

import immunostruct_b200 as I
from immunostruct_b200 import _C, build, neighbors
from immunostruct_b200.neighbors import embed, embed_pair, nearest
from oracle import kernel_contracts as KC

from conftest import ROOT, load_golden
from helpers import build_model, graph_batch


# ---- the search contract ----------------------------------------------------------------------------------------------
def knn_contract(query, bank, k, exclude=None, chunk=256):
    """The contract of is_knn in fp64, on the device of its inputs: squared Euclidean distances, ascending by
    (distance, bank index); a pair with a NaN distance (a NaN feature on either side) and the excluded row are not
    eligible; slots past the eligible rows hold -1 / +inf.  -> (index [Q, k] int64, distance [Q, k] float64)."""
    q64, b64 = query.double(), bank.double()
    n_q, r = q64.shape[0], b64.shape[0]
    index = torch.full((n_q, k), -1, dtype=torch.int64, device=query.device)
    dist = torch.full((n_q, k), float("inf"), dtype=torch.float64, device=query.device)
    cols = torch.arange(r, device=query.device)
    for s in range(0, n_q, chunk):
        d = ((q64[s:s + chunk, None, :] - b64[None, :, :]) ** 2).sum(-1) if b64.shape[1] <= 8 else \
            torch.cdist(q64[s:s + chunk], b64, compute_mode="donot_use_mm_for_euclid_dist") ** 2
        bad = torch.isnan(d)
        if exclude is not None:
            bad |= cols[None, :] == exclude[s:s + chunk, None]
        # NaN sorts after every number in torch.sort; stable: ties keep the smaller index first
        d = torch.where(bad, torch.full_like(d, float("nan")), d)
        val, idx = torch.sort(d, dim=1, stable=True)
        m = min(k, r)
        val, idx = val[:, :m], idx[:, :m]
        ok = ~torch.isnan(val)
        index[s:s + chunk, :m] = torch.where(ok, idx, torch.full_like(idx, -1))
        dist[s:s + chunk, :m] = torch.where(ok, val, torch.full_like(val, float("inf")))
    return index, dist


def test_contract_orders_ties_by_index():
    bank = torch.tensor([[1.0, 0.0], [0.0, 1.0], [0.0, 0.0], [-1.0, 0.0], [0.0, -1.0], [2.0, 0.0]])
    idx, d = knn_contract(torch.zeros(1, 2), bank, 6)
    assert idx.tolist() == [[2, 0, 1, 3, 4, 5]]
    assert d.tolist() == [[0.0, 1.0, 1.0, 1.0, 1.0, 4.0]]


def test_contract_nan_rows_queries_and_padding():
    bank = torch.tensor([[0.0, 0.0], [float("nan"), 0.0], [3.0, 0.0]])
    idx, d = knn_contract(torch.tensor([[1.0, 0.0], [0.0, float("nan")]]), bank, 4)
    assert idx.tolist() == [[0, 2, -1, -1], [-1, -1, -1, -1]]
    assert d[0].tolist() == [1.0, 4.0, float("inf"), float("inf")]
    assert torch.isinf(d[1]).all()
    # an infinite feature is a finite-or-infinite distance, not a missing one
    idx, d = knn_contract(torch.zeros(1, 2), torch.tensor([[float("inf"), 0.0], [1.0, 1.0]]), 3)
    assert idx.tolist() == [[1, 0, -1]] and d.tolist() == [[2.0, float("inf"), float("inf")]]


def test_contract_k_larger_than_the_bank_and_exclude():
    bank = torch.arange(5, dtype=torch.float32)[:, None]
    idx, d = knn_contract(bank, bank, 7, exclude=torch.arange(5))
    assert idx[0].tolist() == [1, 2, 3, 4, -1, -1, -1]
    assert idx[2].tolist() == [1, 3, 0, 4, -1, -1, -1]
    assert d[2].tolist()[:4] == [1.0, 1.0, 4.0, 4.0]
    idx, _ = knn_contract(bank, bank, 2, exclude=torch.tensor([-1, -1, 3, -1, 0]))
    assert idx.tolist() == [[0, 1], [1, 0], [2, 1], [3, 2], [4, 3]]


def test_contract_matches_brute_force_on_random_data():
    g = torch.Generator().manual_seed(3)
    q, b = torch.randn(9, 5, generator=g), torch.randn(40, 5, generator=g)
    idx, d = knn_contract(q, b, 6, chunk=4)
    for i in range(9):
        full = sorted((float(((q[i].double() - b[j].double()) ** 2).sum()), j) for j in range(40))[:6]
        assert idx[i].tolist() == [j for _, j in full]
        assert d[i].tolist() == pytest.approx([v for v, _ in full], rel=1e-12)


# ---- argument rules ---------------------------------------------------------------------------------------------------
@pytest.fixture
def no_launch(monkeypatch):
    calls = []
    monkeypatch.setattr(_C, "_call", lambda name, *a: calls.append(name))
    monkeypatch.setattr(_C, "num_sms", lambda: 148)
    yield calls
    assert not calls


def test_knn_binding_argument_rules(no_launch):
    q, b = torch.zeros(3, 4), torch.zeros(5, 4)

    def bad(exc, match, *args, **kw):
        with pytest.raises(exc, match=match):
            _C.knn(*args, **kw)

    bad(ValueError, "2-D", torch.zeros(3), b, 1)
    bad(ValueError, "2-D", q, torch.zeros(5, 4, 1), 1)
    bad(ValueError, "2-D", q.numpy(), b, 1)
    bad(ValueError, "float32", q.double(), b, 1)
    bad(ValueError, "float32", q, b.half(), 1)
    bad(ValueError, "contiguous", torch.zeros(4, 3).t(), b, 1)
    bad(ValueError, "contiguous", q, torch.zeros(4, 5).t(), 1)
    bad(ValueError, "same feature count", q, torch.zeros(5, 3), 1)
    bad(ValueError, "D <= 256", torch.zeros(3, 0), torch.zeros(5, 0), 1)
    bad(ValueError, "D <= 256", torch.zeros(3, 257), torch.zeros(5, 257), 1)
    bad(ValueError, "at least one query", torch.zeros(0, 4), b, 1)
    bad(ValueError, "R < 2", q, torch.zeros(0, 4), 1)
    for k in (0, 65, -1, 2.0, True, None):
        bad(ValueError, "k must be", q, b, k)
    big = torch.zeros(300, 4)
    for s in (0, 4, 1.0, True):
        bad(ValueError, "slices", q, big, 1, slices=s)
    bad(ValueError, "slices", q, b, 1, slices=2)
    for ex in (torch.zeros(3, dtype=torch.int32), torch.zeros(4, dtype=torch.int64), torch.zeros(3, 1, dtype=torch.int64),
               [0, 1, 2]):
        bad(ValueError, "exclude must be", q, b, 1, ex)
    bad(ValueError, r"\[-1, 5\)", q, b, 1, torch.tensor([0, 5, 1]))
    bad(ValueError, r"\[-1, 5\)", q, b, 1, torch.tensor([0, -2, 1]))
    bad(RuntimeError, "CUDA", q, b, 1)
    bad(RuntimeError, "CUDA", q, b, 1, torch.tensor([-1, 4, 0]), slices=1)
    assert _C.knn_max_slices(1) == 1 and _C.knn_max_slices(128) == 1 and _C.knn_max_slices(129) == 2
    assert _C.knn_max_slices(2 ** 31 - 1) == 65535


def test_nearest_argument_rules(no_launch):
    q, b = torch.zeros(3, 4), torch.zeros(5, 4)
    for args in ((torch.zeros(3), b), (q, torch.zeros(5)), (q.numpy(), b)):
        with pytest.raises(ValueError, match="query"):
            nearest(*args, 1)
    with pytest.raises(ValueError, match="k must be"):
        nearest(q, b, 65)
    with pytest.raises(ValueError, match="exclude"):
        nearest(q, b, 1, exclude=torch.tensor([0, 1, 9]))
    with pytest.raises(ValueError, match="float32"):
        nearest(q.double(), b, 1)
    with pytest.raises(RuntimeError, match="CUDA"):
        nearest(q, b, 2, exclude=torch.tensor([0, 1, 2]))


def test_slice_count_fills_the_device(monkeypatch):
    monkeypatch.setattr(_C, "num_sms", lambda: 148)
    assert neighbors._slices(1, 27000) == 148
    assert neighbors._slices(1, 300) == 3                        # never a slice without a full tile
    assert neighbors._slices(129, 30011) == 50                   # 3 query tiles x 50 slices >= 148 CTAs
    assert neighbors._slices(27000, 27000) == 1
    assert neighbors._slices(262144, 27000) == 1


def test_embed_argument_rules(monkeypatch):
    for name in KC.ALL:
        monkeypatch.setattr(_C, name, getattr(KC, name))
    gd = load_golden("hybrid_v2")
    model = build_model("HybridModelv2", gd)
    d, g = gd["dense"], graph_batch(gd["graph"])
    launched = []
    for name in ("head_features_infer", "collate_csr", "linear_tc", "vae_mid_infer"):
        monkeypatch.setattr(_C, name, lambda *a, _n=name, **k: launched.append(_n))
    for name in ("StructureModel", "StructureModelv2", "SequenceModel", "DualModel"):
        m = I.model_map[name](vae_input_dim=231, device="cpu").eval()
        with pytest.raises(NotImplementedError, match="HybridModelv2_SSL"):
            embed(m, g, d["seq"], d["prop"])
    with pytest.raises(NotImplementedError, match="HybridModel_Comparative"):
        embed_pair(model, (g, g), (d["seq"], d["seq"]), (d["prop"], d["prop"]))
    model.train()
    with pytest.raises(RuntimeError, match="eval"):
        embed(model, g, d["seq"], d["prop"])
    assert not launched


# ---- the existing head kernels keep their SASS ------------------------------------------------------------------------
HEAD_SASS = os.path.join(ROOT, "tests", "golden", "head_sass.json")


def _kernel_sass(obj, names):
    text = subprocess.run([os.path.join(os.path.dirname(build.NVCC), "cuobjdump"), "-sass", obj], check=True,
                          stdout=subprocess.PIPE, text=True).stdout
    out, cur = {}, None
    for line in text.splitlines():
        m = re.match(r"\s+Function : (\S+)", line)
        if m:
            cur = m.group(1)
            out[cur] = hashlib.sha1()
        elif cur is not None:
            out[cur].update(line.encode())
    return {n: out[n].hexdigest() for n in names}


def _nvcc_release():
    v = subprocess.run([build.NVCC, "--version"], check=True, stdout=subprocess.PIPE, text=True).stdout
    return re.search(r"release (\S+),", v).group(1)


def test_existing_head_kernels_keep_their_sass(tmp_path):
    """SHA-1 of the cuobjdump -sass text of every kernel that csrc/head.cu had before the feature kernel was added,
    recorded from that source with the nvcc release named in the file (another compiler release emits other SASS)."""
    if not os.path.exists(build.NVCC) or shutil.which(os.path.join(os.path.dirname(build.NVCC), "cuobjdump")) is None:
        pytest.skip("the CUDA toolkit is not installed")
    ref = json.load(open(HEAD_SASS))
    if _nvcc_release() != ref["nvcc_release"]:
        pytest.skip(f"the SASS was recorded with nvcc {ref['nvcc_release']}")
    obj = str(tmp_path / "head.o")
    subprocess.run([build.NVCC, *build.FLAGS, "-I", build.CSRC, "-I",
                    os.path.join(ROOT, "include"), "-c", os.path.join(build.CSRC, "head.cu"), "-o", obj], check=True,
                   stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL)
    assert _kernel_sass(obj, ref["kernels"]) == ref["kernels"]
