"""Graph containers: the drop-in for the ``dgl`` objects the reference's data and model code touch.

* ``graph((src, dst), num_nodes=n)`` / ``Graph`` -- one sample, as built by ``to_dgl``
  (immunostruct/data/utils.py:54-67): directed multigraph, edge i = src[i] -> dst[i], ``ndata['x']``
  [n,23], ``edata['edge_attr']`` [E,1].
* ``batch(graphs)`` -- replaces ``dgl.batch`` in ``collate`` / ``collate_amino_acid``
  (data/utils.py:163,169-170,181,187-188).  On the host it only concatenates the per-sample arrays
  (graph-LOCAL endpoints, no offsetting, no sorting).  ``GraphBatch.to(device)`` (the call at
  procedures/train.py:20) ships them and runs the on-device collation kernel
  (csrc/collate.cu): global ``edge_index``, ``batch`` vector, destination-sorted CSR, CSC transpose,
  per-graph segment offsets -- all cached on the batch for every layer and for the backward pass.

``GraphBatch`` serves both vocabularies: PyG's ``x / edge_index / edge_attr / batch`` (the north star)
and the DGL accessors the reference code uses (``ndata``, ``edata``, ``batch_num_nodes()``,
``num_nodes()``, ``num_edges()``, ``edges()``, ``device``, ``to``).
"""
from __future__ import annotations

from typing import Optional, Sequence

import torch

from . import _C

MAX_IN_DEGREE = 128     # edge tiles hold <= 128 in-edges of whole destination nodes (csrc/egnn.cu)
MAX_GRAPH_NODES = 256   # largest graph the per-graph attention kernels stage on chip (csrc/attn_pool*.cu)

# Collation statistics are checked by default, without a per-batch host synchronisation: the first batch of a
# process is validated synchronously; every later batch copies its four statistics words to pinned host memory
# asynchronously and they are inspected when the NEXT batch is collated (or at validate()).  A bad batch therefore
# raises one batch late at the latest instead of silently producing garbage.  set_validation("off") disables it.
_validation = {"mode": "deferred", "first_done": False, "pending": []}


def set_validation(mode: str) -> None:
    """"deferred" (default), "sync" (check every batch immediately: one host sync per batch) or "off"."""
    if mode not in ("deferred", "sync", "off"):
        raise ValueError("validation mode must be 'deferred', 'sync' or 'off'")
    _validation["mode"] = mode


def _raise_on_stats(max_deg, bad, max_nodes, n_empty, status, claimed_max_nodes=None):
    if bad:
        raise ValueError(f"{bad} edge endpoints fall outside their graph's node range")
    if max_deg > MAX_IN_DEGREE:
        raise ValueError(f"max in-degree {max_deg} exceeds the supported {MAX_IN_DEGREE}")
    if claimed_max_nodes is not None and max_nodes > claimed_max_nodes:
        raise ValueError(f"a graph has {max_nodes} nodes but the batch was built with max_nodes={claimed_max_nodes}")
    if status:
        raise RuntimeError("an EGNN kernel met a node with more than 128 in-edges")


def _drain_pending(block: bool = False) -> None:
    keep = []
    pend = _validation["pending"]
    for i, (ev, host, claimed, owner) in enumerate(pend):
        if block:
            ev.synchronize()
        elif not ev.query():
            keep.append((ev, host, claimed, owner))
            continue
        vals = host.tolist()
        if vals[1] or vals[0] > MAX_IN_DEGREE or vals[4] or (claimed is not None and vals[2] > claimed):
            _validation["pending"] = keep + pend[i + 1:]          # drop before raising: the error is reported once
            _raise_on_stats(vals[0], vals[1], vals[2], vals[3], vals[4], claimed)
    _validation["pending"] = keep


_PINNED_SLOTS = 64


def _pinned_slot():
    """Round-robin slot of a small pinned ring for the asynchronous statistics read-back (allocating pinned memory per
    batch would cost more than the copy)."""
    ring = _validation.get("ring")
    if ring is None:
        ring = _validation["ring"] = torch.empty(_PINNED_SLOTS, 5, dtype=torch.int32).pin_memory()
        _validation["next"] = 0
    if len(_validation["pending"]) >= _PINNED_SLOTS - 1:
        _drain_pending(block=True)
    i = _validation["next"]
    _validation["next"] = (i + 1) % _PINNED_SLOTS
    return ring[i]


class Graph:
    """A single host-side sample graph (``dgl.graph`` stand-in for the data pipeline)."""

    def __init__(self, data, num_nodes: Optional[int] = None):
        src, dst = data
        self._src = torch.as_tensor(src, dtype=torch.int64).reshape(-1)
        self._dst = torch.as_tensor(dst, dtype=torch.int64).reshape(-1)
        if self._src.numel() != self._dst.numel():
            raise ValueError("src and dst must have the same length")
        if num_nodes is None:
            num_nodes = int(max(self._src.max(), self._dst.max())) + 1 if self._src.numel() else 0
        self._n = int(num_nodes)
        self.ndata, self.edata = {}, {}

    @property
    def device(self):
        return self._src.device

    def num_nodes(self) -> int:
        return self._n

    def num_edges(self) -> int:
        return int(self._src.numel())

    def edges(self):
        return self._src, self._dst

    def batch_num_nodes(self):
        return torch.tensor([self._n], dtype=torch.int64)

    def to(self, device, non_blocking: bool = False):
        return batch([self]).to(device, non_blocking=non_blocking)


def graph(data, num_nodes: Optional[int] = None) -> Graph:
    return Graph(data, num_nodes)


class GraphBatch:
    """A batch of graphs; device-resident instances carry the cached CSR / CSC / segment offsets."""

    _CSR_FIELDS = ("node_off", "edge_off", "edge_index", "batch", "indptr", "csr_src", "csr_dst", "csr_eid",
                   "outptr", "csc_pos", "stats")

    def __init__(self, x, src_local, dst_local, edge_attr, node_counts, edge_counts,
                 max_nodes: Optional[int] = None, collate_now: bool = True):
        self.ndata = {"x": x}
        self.edata = {"edge_attr": edge_attr}
        self._src_local = src_local
        self._dst_local = dst_local
        self._node_counts = node_counts
        self._edge_counts = edge_counts
        self.n_graphs = int(node_counts.numel())
        self.n_nodes = int(x.shape[0])
        self.n_edges = int(src_local.numel())
        self.max_nodes = max_nodes
        self.status = None
        for f in self._CSR_FIELDS:
            setattr(self, self._attr(f), None)
        if x.is_cuda and collate_now:
            self._collate()

    @staticmethod
    def _attr(f):
        return "_" + f if f in ("edge_index", "batch") else f

    # ---- construction ---------------------------------------------------------------------------
    @classmethod
    def from_arrays(cls, x, src_local, dst_local, edge_attr, node_counts, edge_counts, max_nodes=None):
        """Device-resident (or host) concatenated arrays with graph-local endpoints."""
        return cls(x, src_local.to(torch.int64), dst_local.to(torch.int64), edge_attr,
                   node_counts.to(torch.int64), edge_counts.to(torch.int64), max_nodes)

    def _collate(self):
        dev = self.ndata["x"].device
        n, e, b = self.n_nodes, self.n_edges, self.n_graphs
        i64 = dict(dtype=torch.int64, device=dev)
        i32 = dict(dtype=torch.int32, device=dev)
        out = {
            "node_off": torch.empty(b + 1, **i64), "edge_off": torch.empty(b + 1, **i64),
            "edge_index": torch.empty(2, e, **i64), "batch": torch.empty(n, **i64),
            "indptr": torch.empty(n + 1, **i32), "csr_src": torch.empty(e, **i32),
            "csr_dst": torch.empty(e, **i32), "csr_eid": torch.empty(e, **i32),
            "outptr": torch.empty(n + 1, **i32), "csc_pos": torch.empty(e, **i32),
            "scratch": torch.empty(2 * n, **i32), "stats": torch.empty(4, **i32),
        }
        _C.collate_csr(self._src_local, self._dst_local, self._node_counts, self._edge_counts, n, e, out)
        for f in self._CSR_FIELDS:
            setattr(self, self._attr(f), out[f])
        self.status = torch.zeros(1, **i32)
        if self.max_nodes is None:
            self.max_nodes = int(self._node_counts.max()) if b else 0
        mode = _validation["mode"]
        if mode == "off" or not self.stats.is_cuda or torch.cuda.is_current_stream_capturing():
            return
        if mode == "sync" or not _validation["first_done"]:
            _validation["first_done"] = True
            self.validate()
            return
        _drain_pending()
        host = _pinned_slot()
        host[:4].copy_(self.stats, non_blocking=True)
        host[4:].copy_(self.status, non_blocking=True)
        ev = torch.cuda.Event()
        ev.record()
        _validation["pending"].append((ev, host, self.max_nodes, id(self)))

    def validate(self):
        """Host check of the collation statistics and the EGNN status flag (one device->host read)."""
        if self.stats is None:
            raise RuntimeError("validate() needs a device-resident batch")
        max_deg, bad, max_nodes, n_empty = self.stats.tolist()
        _validation["pending"] = [e for e in _validation["pending"] if e[3] != id(self)]     # reported here, not again later
        _raise_on_stats(max_deg, bad, max_nodes, n_empty, int(self.status.item()), self.max_nodes)
        return self

    def replicate(self, r: int) -> "GraphBatch":
        """``r`` copies of the batch, one after another, collated on its device (features detached; callers that evaluate
        many variants of one batch replace the copies' features and keep the topology)."""
        ea = self.edata["edge_attr"]
        out = GraphBatch(self.ndata["x"].detach().repeat(r, 1), self._src_local.repeat(r), self._dst_local.repeat(r),
                         ea.detach().repeat(r, *([1] * (ea.dim() - 1))), self._node_counts.repeat(r),
                         self._edge_counts.repeat(r), max_nodes=self.max_nodes, collate_now=False)
        out._collate()
        return out

    # ---- DGL vocabulary -------------------------------------------------------------------------
    @property
    def device(self):
        return self.ndata["x"].device

    def to(self, device, non_blocking: bool = False):
        device = torch.device(device)
        if device.type == self.device.type and (device.index is None or device.index == self.device.index):
            return self
        mv = lambda t: t.to(device, non_blocking=non_blocking)
        return GraphBatch(mv(self.ndata["x"]), mv(self._src_local), mv(self._dst_local),
                          mv(self.edata["edge_attr"]), mv(self._node_counts), mv(self._edge_counts),
                          self.max_nodes)

    def pin_memory(self):
        if self.device.type != "cpu":
            return self
        p = lambda t: t.pin_memory()
        return GraphBatch(p(self.ndata["x"]), p(self._src_local), p(self._dst_local), p(self.edata["edge_attr"]),
                          p(self._node_counts), p(self._edge_counts), self.max_nodes)

    def batch_num_nodes(self):
        return self._node_counts

    def batch_num_edges(self):
        return self._edge_counts

    @property
    def batch_size(self) -> int:
        return self.n_graphs

    def num_nodes(self) -> int:
        return self.n_nodes

    def num_edges(self) -> int:
        return self.n_edges

    def edges(self):
        ei = self.edge_index
        return ei[0], ei[1]

    # ---- PyG vocabulary -------------------------------------------------------------------------
    @property
    def x(self):
        return self.ndata["x"]

    @property
    def edge_attr(self):
        return self.edata["edge_attr"]

    def host_edge_index(self):
        """Global endpoints for a HOST batch (integer bookkeeping for data utilities; the model
        itself only accepts device batches)."""
        off = torch.zeros(self.n_graphs + 1, dtype=torch.int64)
        off[1:] = torch.cumsum(self._node_counts, 0)
        shift = torch.repeat_interleave(off[:-1], self._edge_counts)
        return torch.stack([self._src_local + shift, self._dst_local + shift])

    @property
    def edge_index(self):
        if self._edge_index is None and not self.ndata["x"].is_cuda:
            return self.host_edge_index()
        return self._edge_index

    @property
    def batch(self):
        if self._batch is None and not self.ndata["x"].is_cuda:
            return torch.repeat_interleave(torch.arange(self.n_graphs), self._node_counts)
        return self._batch


def batch(graphs: Sequence[Graph], pin_memory: bool = False) -> GraphBatch:
    """``dgl.batch`` replacement for ``collate`` (data/utils.py:163): concatenate per-sample arrays."""
    if len(graphs) == 0:
        raise ValueError("batch() needs at least one graph")
    if isinstance(graphs[0], GraphBatch):
        raise TypeError("batch() expects single graphs")
    x = torch.cat([g.ndata["x"] for g in graphs], 0)
    ea = torch.cat([g.edata["edge_attr"] for g in graphs], 0)
    src = torch.cat([g._src for g in graphs])
    dst = torch.cat([g._dst for g in graphs])
    nc = torch.tensor([g.num_nodes() for g in graphs], dtype=torch.int64)
    ec = torch.tensor([g.num_edges() for g in graphs], dtype=torch.int64)
    if x.is_cuda:
        nc, ec = nc.to(x.device), ec.to(x.device)
    out = GraphBatch(x.float(), src, dst, ea.float(), nc, ec, max_nodes=int(nc.max()))
    return out.pin_memory() if pin_memory and not x.is_cuda else out


def collate(samples):
    """Drop-in for ``immunostruct/data/utils.py:160-176``: (graph | (graph, graph), seq, label, labelf)."""
    graphs, seq_data, labels, labelsf = map(list, zip(*samples))
    if isinstance(graphs[0], Graph):
        return (batch(graphs), torch.stack(seq_data, 0), torch.stack(labels, 0), torch.stack(labelsf, 0))
    return ((batch([g[0] for g in graphs]), batch([g[1] for g in graphs])),
            (torch.stack([s[0] for s in seq_data], 0), torch.stack([s[1] for s in seq_data], 0)),
            torch.stack(labels, 0),
            (torch.stack([l[0] for l in labelsf], 0), torch.stack([l[1] for l in labelsf], 0)))


def collate_amino_acid(samples):
    """Drop-in for ``immunostruct/data/utils.py:178-196`` (SSL variant with the masked residue id)."""
    amino = torch.stack([s[4] for s in samples], 0).flatten()
    return (*collate([s[:4] for s in samples]), amino)
