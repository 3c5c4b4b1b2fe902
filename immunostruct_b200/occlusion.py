"""Structural occlusion: the score of the batch with one residue, or one contact, removed from the structure.

The residue-identity analyses (``mutagenesis``, ``design``) keep the coordinates and contacts of the input structure, and
the integrated-gradients attribution of ``edge_attr`` measures the sensitivity to a constant scalar feature, not the
effect of a contact.  Occlusion answers "which residues and which contacts of the structure does the call depend on"
exactly, by removing each one and scoring the result:

* residue occlusion of graph-local row i of sample b: the 23 floats of the row become 0.0 (features and coordinates) and
  every edge with src == i or dst == i is dropped, multi-edges and a self-loop included.  The row stays, so node counts
  and the mean pool's denominator are unchanged: the residue becomes an absent (padded) one, as ``pad_graph`` writes it.
* contact occlusion of the unordered pair {u, v}, u != v: every edge between u and v in either direction is dropped.
  Rows are unchanged; a self-loop is not a contact.  The contacts of a graph are the distinct unordered pairs of its
  non-self-loop edges.

The kept edges keep their base order, so a variant is exactly the graph a boolean edge mask would build.  The sequence
branch is not touched: a variant has the sequence, the properties and the draws of its base sample, so variants of one
sample share their latent tokens and differ by their structural effect alone.  That is also why the VAE encoder runs
once per call, at batch B, and each pass gathers its encoded tensors by sample instead of re-encoding.

One host read before the first launch checks the selection and sizes every pass.  A pass is a run of up to
``max_graphs`` variants in (sample, u, v) order: ``is_occlusion_expand`` (csrc/occlusion.cu) writes their rows and
compacted edges from the resident batch, the pass's topology is collated, the structure trunk runs, and the multi-draw
head scores every draw.  The expansion flag is read once, after the last pass.

An entry agrees with the fused eval forward of the host-built occluded batch on the same draws to rounding, not bit for
bit: where a graph sits in a batch changes two summation orders (mutagenesis module docstring, DESIGN 4.4c).
"""
from __future__ import annotations

from dataclasses import dataclass
from typing import Optional

import torch

from . import functional as IF
from .comparative_models import _Comparative
from .hybrid_models import _Hybrid
from .predictive import _CLASSES, _PAIR_CLASSES, Predictive, _check, _scorer, _scorer_pair
from .resident import pass_totals, score_gathered, variant_passes

Tensor = torch.Tensor


@dataclass
class ResidueOcclusion:
    """Scores of the batch with one residue occluded, aligned with the graph's node rows; rows not scanned are NaN."""
    logits: Tensor        # [ΣN, K]  logit with row i occluded, draw k of its sample
    prob_mean: Tensor     # [ΣN]     mean of sigmoid(logit) over the draws
    prob_std: Tensor      # [ΣN]     population standard deviation of sigmoid(logit) over the draws
    base: Predictive      # the unmodified batch on the same draws


@dataclass
class ContactOcclusion:
    """Scores of the batch with one contact occluded, one entry per contact, ordered by (sample, u, v)."""
    sample: Tensor        # [C]   int64, the contact's sample
    u: Tensor             # [C]   int64, graph-local endpoint, u < v
    v: Tensor             # [C]   int64, graph-local endpoint
    edge_contact: Tensor  # [ΣE]  int64, contact id of each edge of the batch; -1 for self-loops and unselected contacts
    logits: Tensor        # [C, K]
    prob_mean: Tensor     # [C]
    prob_std: Tensor      # [C]
    base: Predictive


def _degrees(graph):
    """(global src, global dst, edges touching each node row [N]: in + out degree, a self-loop counted once)."""
    gs, gd = graph.edge_index
    n = graph.n_nodes
    loops = torch.zeros(n, dtype=torch.int64, device=gs.device).scatter_add_(0, gs, (gs == gd).long())
    return gs, gd, torch.bincount(gs, minlength=n) + torch.bincount(gd, minlength=n) - loops


def _selection(graph, nodes, touch):
    """The checked node-row selection, bool [ΣN] on the batch's device (default: every row that is not already absent,
    i.e. not all-zero with no edge)."""
    n = graph.n_nodes
    x = graph.ndata["x"]
    if nodes is None:
        return ~((x == 0).all(1) & (touch == 0))
    if not isinstance(nodes, Tensor) or nodes.dtype != torch.bool or tuple(nodes.shape) != (n,):
        raise ValueError(f"nodes must be a bool tensor [ΣN={n}] over the batch's node rows")
    return nodes.to(x.device)


def _first_selected(keep):
    """Indices of the True entries first, in order, then the others: a stable sort, so no host read."""
    return torch.sort((~keep).to(torch.int32), stable=True).indices


def _finish_tables(graph, smp, na, nb, kept, n_var, n_slots, max_graphs, what):
    """Running sums and the one host read -> (sample, node_a, node_b, node count, kept edges, node offsets, edge offsets,
    passes, pass node totals, pass edge totals, C), trimmed to the C variants."""
    nv = graph.batch_num_nodes().to(smp.device)[smp]
    ncs, ecs, node_tot, edge_tot = pass_totals(nv, kept, n_var, n_slots, max_graphs)
    vals = torch.cat([n_var.reshape(1), node_tot, edge_tot]).tolist()
    c = vals[0]
    if c == 0:
        raise ValueError(f"the selection holds no {what}: nothing to occlude")
    passes = variant_passes(c, max_graphs)
    return (smp[:c].contiguous(), na[:c].contiguous(), nb[:c].contiguous(), nv[:c].contiguous(), kept[:c].contiguous(),
            ncs[:c + 1], ecs[:c + 1], passes, vals[1:1 + len(passes)], vals[1 + n_slots:1 + n_slots + len(passes)], c)


def _residue_tables(graph, nodes, max_graphs):
    """Residue variants in row order: (tables, selected rows [C])."""
    variant_passes(1, max_graphs)
    gs, gd, touch = _degrees(graph)
    sel = _selection(graph, nodes, touch)
    n = graph.n_nodes
    if n == 0:
        raise ValueError("the selection holds no residue: nothing to occlude")
    rows = _first_selected(sel)
    smp = graph.batch[rows]
    na = rows - graph.node_off[smp]
    kept = graph.batch_num_edges().to(rows.device)[smp] - touch[rows]
    tables = _finish_tables(graph, smp, na, torch.full_like(na, -1), kept, sel.sum(), -(-n // max_graphs), max_graphs,
                            "residue")
    return tables, rows[:tables[-1]]


def _contacts(gs, gd, sel, n):
    """The contacts of the global edges (gs, gd) [E > 0] with at least one endpoint selected by ``sel`` [N], numbered in
    (sample, u, v) order, without a host read -> (edge_contact [E]: the contact id of each edge, -1 for self-loops and
    unselected contacts; global endpoints ug, vg [E] of contact c at entry c, for c < C; edges of contact c [E]; C, a
    device count)."""
    e = gs.shape[0]
    # global node ids run in (sample, local row) order, so the key lo * N + hi orders contacts by (sample, u, v)
    lo, hi = torch.minimum(gs, gd), torch.maximum(gs, gd)
    sentinel = n * n
    valid = (gs != gd) & (sel[gs] | sel[gd])
    ks, order = torch.sort(torch.where(valid, lo * n + hi, sentinel), stable=True)
    live = ks < sentinel
    first = live & torch.cat([torch.ones(1, dtype=torch.bool, device=ks.device), ks[1:] != ks[:-1]])
    cid = first.cumsum(0) - 1
    edge_contact = torch.empty_like(cid).scatter_(0, order, torch.where(live, cid, -1))
    mult = torch.zeros(e + 1, dtype=torch.int64, device=ks.device).scatter_add_(0, torch.where(live, cid, e),
                                                                                torch.ones_like(cid))[:e]
    key = ks[_first_selected(first)]                              # the contacts' keys first, in order
    return edge_contact, (key // n).clamp_max(n - 1), key % n, mult, first.sum()


def _contact_tables(graph, nodes, max_graphs):
    """Contact variants in (sample, u, v) order: (tables, edge_contact [ΣE])."""
    variant_passes(1, max_graphs)
    gs, gd, touch = _degrees(graph)
    sel = _selection(graph, nodes, touch)
    n, e = graph.n_nodes, graph.n_edges
    if e == 0:
        raise ValueError("the selection holds no contact: nothing to occlude")
    edge_contact, ug, vg, mult, c = _contacts(gs, gd, sel, n)
    smp = graph.batch[ug]
    off = graph.node_off[smp]
    kept = graph.batch_num_edges().to(ug.device)[smp] - mult
    tables = _finish_tables(graph, smp, ug - off, vg - off, kept, c, -(-e // max_graphs), max_graphs, "contact")
    return tables, edge_contact


def _occlude(model, scorer, graph, tables):
    """Every variant in gathered passes -> (logits [C,K], prob_mean [C], prob_std [C]).  The sequence branch is not
    touched: a pass gathers the base's encoded tensors and draws by sample instead of re-encoding."""
    smp, na, nb, nv, kept, ncs, ecs, passes, node_totals, edge_totals, _ = tables
    mu, logvar, z_vae, e = scorer.item[1:]
    flag = torch.zeros(1, dtype=torch.int32, device=smp.device)

    def expand(j, r, inputs, outputs):
        IF._C.occlusion_expand(*inputs, smp[j:j + r], na[j:j + r], nb[j:j + r], *outputs, flag)

    def pass_item(g, sp, _):
        return model.structure_embedding(g, project=False)[0].contiguous(), mu[sp], logvar[sp], z_vae[sp], e[:, sp]

    out = score_gathered(scorer, graph, smp, nv, kept, ncs, ecs, passes, node_totals, edge_totals, expand, pass_item)
    if flag.item():
        raise RuntimeError("is_occlusion_expand rejected a variant: its indices or offsets disagree with the batch")
    return out


def _residue_result(graph, rows, out, base):
    n, k = graph.n_nodes, out[0].shape[1]
    full = lambda t, shape: torch.full(shape, float("nan"), dtype=t.dtype, device=t.device).index_put_((rows,), t)
    return ResidueOcclusion(full(out[0], (n, k)), full(out[1], (n,)), full(out[2], (n,)), base)


def _contact_result(tables, edge_contact, out, base):
    smp, na, nb = tables[:3]
    return ContactOcclusion(smp, na, nb, edge_contact, *out, base)


def occlude_residues(model, graph, seq, prop, *, nodes: Optional[Tensor] = None, eps: Optional[Tensor] = None,
                     samples: int = 1, max_graphs: int = 4096) -> ResidueOcclusion:
    """Scores of ``model(graph, seq, prop)[3]`` (the logit) with each selected residue occluded: its 23 floats set to 0.0
    and every edge touching it dropped, as an absent (padded) residue.

    ``nodes`` bool [ΣN] selects node rows in ``graph.ndata['x']`` order; by default every row that is not already absent
    (all-zero with no edge).  An explicitly selected absent row is scored and equals ``base`` up to rounding.  ``eps``
    [K, B, latent] gives the draws, or one ``model.sample_eps`` call of [K*B, latent] (K = ``samples``) makes them; a
    variant uses the draws of its sample.  Variants run in row order, in passes of at most ``max_graphs``.  Follows
    ``model.forward`` for the eight classes ``predictive`` supports; the model must be in eval mode; no_grad, and every
    ``.grad`` is left untouched.  The result is aligned with the rows; rows not scanned are NaN."""
    _check(model, samples, (_Hybrid, _Comparative), "occlude_residues", _CLASSES)
    tables, rows = _residue_tables(graph, nodes, max_graphs)
    with torch.no_grad():
        scorer = _scorer(model, graph, seq, prop, eps, samples)
        return _residue_result(graph, rows, _occlude(model, scorer, graph, tables), scorer.base)


def occlude_contacts(model, graph, seq, prop, *, nodes: Optional[Tensor] = None, eps: Optional[Tensor] = None,
                     samples: int = 1, max_graphs: int = 4096) -> ContactOcclusion:
    """Scores of ``model(graph, seq, prop)[3]`` (the logit) with each selected contact occluded: every edge between its
    two residues, in either direction, dropped; rows unchanged.

    The contacts of a graph are the distinct unordered pairs of its non-self-loop edges; ``nodes`` bool [ΣN] selects the
    contacts with at least one selected endpoint (e.g. the peptide rows: the peptide-HLA interface and the peptide's own
    contacts), by default every contact.  Entries are ordered by (sample, u, v); ``edge_contact`` maps each edge of the
    batch to its contact.  Draws, passes, classes, eval mode, no_grad and ``.grad`` as in ``occlude_residues``."""
    _check(model, samples, (_Hybrid, _Comparative), "occlude_contacts", _CLASSES)
    tables, edge_contact = _contact_tables(graph, nodes, max_graphs)
    with torch.no_grad():
        scorer = _scorer(model, graph, seq, prop, eps, samples)
        return _contact_result(tables, edge_contact, _occlude(model, scorer, graph, tables), scorer.base)


def occlude_residues_pair(model, graph_pair, seq_pair, prop_pair, *, nodes: Optional[Tensor] = None, eps=None,
                          samples: int = 1, max_graphs: int = 4096) -> ResidueOcclusion:
    """``occlude_residues`` of the cancer item of ``model.forward_comparative(graph_pair, seq_pair, prop_pair)`` against
    its fixed wild type, for the four comparative classes; ``nodes`` indexes the cancer graph's rows.

    The wild type is encoded once, at batch B; each pass gathers its encoded tensors and its draws by sample.  ``eps`` =
    (eps_c, eps_w), each [K, B, latent], or one ``model.sample_eps`` call of [K*B, latent] per item, cancer first.
    Without ``use_wt_for_downstream`` the wild type is neither run nor drawn for.  ``base`` equals ``predictive_pair`` on
    the same draws."""
    _check(model, samples, _Comparative, "occlude_residues_pair", _PAIR_CLASSES)
    tables, rows = _residue_tables(graph_pair[0], nodes, max_graphs)
    with torch.no_grad():
        scorer = _scorer_pair(model, graph_pair, seq_pair, prop_pair, eps, samples)
        return _residue_result(graph_pair[0], rows, _occlude(model, scorer, graph_pair[0], tables), scorer.base)


def occlude_contacts_pair(model, graph_pair, seq_pair, prop_pair, *, nodes: Optional[Tensor] = None, eps=None,
                          samples: int = 1, max_graphs: int = 4096) -> ContactOcclusion:
    """``occlude_contacts`` of the cancer item of ``model.forward_comparative`` against its fixed wild type; the wild
    type as in ``occlude_residues_pair``."""
    _check(model, samples, _Comparative, "occlude_contacts_pair", _PAIR_CLASSES)
    tables, edge_contact = _contact_tables(graph_pair[0], nodes, max_graphs)
    with torch.no_grad():
        scorer = _scorer_pair(model, graph_pair, seq_pair, prop_pair, eps, samples)
        return _contact_result(tables, edge_contact, _occlude(model, scorer, graph_pair[0], tables), scorer.base)
