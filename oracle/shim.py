"""Import the UNMODIFIED reference model/loss files from ``/root/reference`` on a box that has
neither ``dgl`` nor ``torch_geometric``.  TEST INFRASTRUCTURE ONLY (see reference_ops.py header).

``install()`` puts minimal stand-ins for the absent third-party packages into ``sys.modules``
(``dgl``, ``dgl.nn``, ``dgl.dataloading``, ``torch_geometric.nn``, ``matplotlib.pyplot``,
``lifelines``) and prepends ``/root/reference/immunostruct`` to ``sys.path`` so that
``import models`` / ``import utils`` resolve to the reference's own packages.  The stand-ins'
arithmetic (EGNNConv, batch, pooling) is the restatement in ``oracle/reference_ops.py``; everything
else the imported classes execute is the reference's literal code.  Used by
``tests/golden/make_golden.py`` / ``make_golden_r2.py`` to generate the committed vectors, which the tests
read instead of the reference tree.
"""
from __future__ import annotations

import os
import sys
import types

import torch
import torch.nn as nn

from . import reference_ops as R

# The reference tree: /root/reference in the build container; on the GPU box (where /root/reference does not exist) the
# copy that oracle/install_ref.py placed under baseline/_ref/ (git-ignored, travels with the snapshot).
_REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
_CANDIDATES = ("/root/reference/immunostruct", os.path.join(_REPO, "baseline", "_ref", "immunostruct"))
REFERENCE_ROOT = next((c for c in _CANDIDATES if os.path.isdir(os.path.join(c, "models"))), _CANDIDATES[0])


def reference_available() -> bool:
    return os.path.isdir(os.path.join(REFERENCE_ROOT, "models"))


class ShimGraph:
    """Just enough of ``dgl.DGLGraph`` for the reference model code (hybrid_models.py:82,86-87)."""

    def __init__(self, src, dst, num_nodes, batch_num_nodes=None):
        self._src, self._dst, self._n = src, dst, int(num_nodes)
        self.ndata, self.edata = {}, {}
        self._bnn = batch_num_nodes if batch_num_nodes is not None else torch.tensor([self._n])

    @property
    def device(self):
        return self._src.device

    def to(self, device):
        return self

    def num_nodes(self):
        return self._n

    def num_edges(self):
        return int(self._src.numel())

    def edges(self):
        return self._src, self._dst

    def batch_num_nodes(self):
        return self._bnn


def shim_graph(data, num_nodes=None):
    src, dst = data
    return ShimGraph(torch.as_tensor(src), torch.as_tensor(dst), num_nodes)


def shim_batch(graphs):
    b = R.dgl_batch([{"src": g._src, "dst": g._dst, "num_nodes": g._n, "x": g.ndata["x"],
                      "edge_attr": g.edata["edge_attr"]} for g in graphs])
    out = ShimGraph(b["src"], b["dst"], b["num_nodes"], b["batch_num_nodes"])
    out.ndata["x"], out.edata["edge_attr"] = b["x"], b["edge_attr"]
    return out


def graph_from_dict(b: dict) -> ShimGraph:
    g = ShimGraph(b["src"], b["dst"], b["num_nodes"], b["batch_num_nodes"])
    g.ndata["x"], g.edata["edge_attr"] = b["x"], b["edge_attr"]
    return g


class ShimEGNNConv(nn.Module):
    """Parameter container with upstream DGL's layout; forward = reference_ops.egnn_conv."""

    def __init__(self, in_size, hidden_size, out_size, edge_feat_size=0):
        super().__init__()
        act = nn.SiLU()
        self.edge_mlp = nn.Sequential(nn.Linear(in_size * 2 + edge_feat_size + 1, hidden_size), act,
                                      nn.Linear(hidden_size, hidden_size), act)
        self.node_mlp = nn.Sequential(nn.Linear(in_size + hidden_size, hidden_size), act,
                                      nn.Linear(hidden_size, out_size))
        self.coord_mlp = nn.Sequential(nn.Linear(hidden_size, hidden_size), act,
                                       nn.Linear(hidden_size, 1, bias=False))

    def forward(self, graph, node_feat, coord_feat, edge_feat=None):
        p = dict(self.named_parameters())
        src, dst = graph.edges()
        return R.egnn_conv(p, "", src, dst, node_feat, coord_feat, edge_feat)


def install():
    """Idempotently install the stand-ins and make the reference importable."""
    if "dgl" not in sys.modules:
        dgl = types.ModuleType("dgl")
        dgl.DGLGraph = ShimGraph
        dgl.graph = shim_graph
        dgl.batch = shim_batch
        dgl_nn = types.ModuleType("dgl.nn")
        dgl_nn.EGNNConv = ShimEGNNConv
        dgl_dl = types.ModuleType("dgl.dataloading")
        dgl_dl.GraphDataLoader = torch.utils.data.DataLoader
        dgl.nn, dgl.dataloading = dgl_nn, dgl_dl
        sys.modules.update({"dgl": dgl, "dgl.nn": dgl_nn, "dgl.dataloading": dgl_dl})
    if "torch_geometric" not in sys.modules:
        tg = types.ModuleType("torch_geometric")
        tg_nn = types.ModuleType("torch_geometric.nn")
        tg_nn.global_mean_pool = R.global_mean_pool
        tg_nn.global_max_pool = R.global_max_pool
        tg.nn = tg_nn
        sys.modules.update({"torch_geometric": tg, "torch_geometric.nn": tg_nn})
    for name in ("matplotlib", "matplotlib.pyplot", "lifelines", "lifelines.statistics", "wandb"):
        if name not in sys.modules:
            try:
                __import__(name)
            except Exception:
                sys.modules[name] = types.ModuleType(name)
    if REFERENCE_ROOT not in sys.path:
        sys.path.insert(0, REFERENCE_ROOT)


def load_reference():
    """Returns (model_map, Losses, PairedContrastiveLoss) from the reference's own files."""
    if not reference_available():
        raise RuntimeError("no reference tree on this box (/root/reference or baseline/_ref, see oracle/install_ref.py)")
    install()
    import importlib
    mapping = importlib.import_module("models.mapping")
    loss = importlib.import_module("utils.loss")
    contrastive = importlib.import_module("utils.contrastive")
    return mapping.model_map, loss.Losses, contrastive.PairedContrastiveLoss
