"""In-silico saturation mutagenesis: the score of every single-residue substitution at chosen sites of each sample.

For each sample b and site p, each of the 20 residue types c replaces the native residue at two places: the residue columns
of one node row of the graph (``node_index[b, p]``, graph-local) and one row of the sequence one-hot
(``seq_index[b, p]``, written as column ``seq_columns[c]``).  Coordinates and contacts stay those of the input structure:
nothing is re-folded.  Neither the repository nor the reference pins where the peptide sits in the graph or how the
graph's 20 residue columns map onto the sequence alphabet, so the caller names the sites and the map; a device check
rejects a site row that is not exactly one-hot (a padded or masked row) or that contradicts ``seq_columns``.

The P x 20 variants of the batch run in passes of r = min(remaining, max_graphs // B) copies of the whole batch: one
kernel writes a pass's mutant features from the resident batch (``is_mutscan_expand``, csrc/mutscan.cu), the copies'
topology is collated once per distinct r before the first pass (``resident``'s replica passes), the trunk and the VAE
encoder run once per pass and the multi-draw head (``is_head_mc_infer``) scores every draw.  The reparameterisation
noise is common to all variants of a sample (common random numbers), so the difference between two variants is the
effect of the substitution alone.

An entry agrees with the fused eval forward of the B-sample mutant batch on the same draw to rounding, not bit for bit:
where a graph sits in the batch changes two summation orders, the edge kernel's per-tile segment-sum MMA (a node's
in-edges land at other positions of a 128-edge tile) and the K-slice count of the vae_fc1 GEMM (it follows the row count).

``score_variants`` scores a caller's library instead: each variant is one sample of the batch with any list of
substitutions (neoantigen candidates, anchor-modified designs, threaded peptides or HLA alleles).  A pass is a run of up to
``max_graphs`` variants in the caller's order; ``is_variant_expand`` gathers their graphs, edges and sequences from the
resident batch and applies the substitutions, the gathered topology is collated once per pass (``resident``'s gathered
passes), and the trunk and the multi-draw head run as for the scan, each variant on the draws of its base sample.
"""
from __future__ import annotations

from dataclasses import dataclass
from typing import Optional

import torch

from . import functional as IF
from .comparative_models import _Comparative
from .hybrid_models import _Hybrid
from .predictive import _CLASSES, _PAIR_CLASSES, Predictive, _check, _encode, _scorer, _scorer_pair
from .resident import (N_RESIDUES, check_one_hot, native_residues, pass_totals, replicas, scan_passes, score_gathered,
                       score_replicas, sequence_replica, variant_passes)

Tensor = torch.Tensor


@dataclass
class Scan:
    """Scores of the single-residue variants; entries of absent sites are NaN."""
    logits: Tensor        # [B, P, 20, K]  logit of sample b with residue column c at site p, draw k
    prob_mean: Tensor     # [B, P, 20]     mean of sigmoid(logit) over the draws
    prob_std: Tensor      # [B, P, 20]     population standard deviation of sigmoid(logit) over the draws
    native: Tensor        # [B, P]         residue column of the input at the site, -1 = absent site
    base: Predictive      # the unmutated batch on the same draws


def scan_sites(n_sites: int, device=None) -> Tensor:
    """The copies of a scan in order, int32 [P*20, 2] = (site p, residue column c), site-major."""
    p = torch.arange(n_sites, dtype=torch.int32).repeat_interleave(N_RESIDUES)
    c = torch.arange(N_RESIDUES, dtype=torch.int32).repeat(n_sites)
    return torch.stack([p, c], 1).to(device)


def _seq_columns(seq_columns, dev):
    """seq_columns as int64 [20] on ``dev``, after the host checks of its type and shape."""
    cols = torch.as_tensor(seq_columns)
    if cols.dtype.is_floating_point or cols.dtype == torch.bool or cols.shape != (N_RESIDUES,):
        raise ValueError("seq_columns must hold 20 integers: the sequence column of each residue-feature column")
    return cols.to(dev, torch.int64).contiguous()


def _columns_bad(cols, V):
    """Device bool: seq_columns does not map the 20 residue columns to distinct sequence columns in [0, V)."""
    s = cols.sort().values
    return ((s < 0) | (s >= V)).any() | (s[1:] == s[:-1]).any()


def _site_tables(graph, seq, node_index, seq_index, seq_columns):
    """Checked (node_index, seq_index, seq_columns) on the batch's device, int64.  One host read for all checks."""
    b = graph.n_graphs
    for name, t in (("node_index", node_index), ("seq_index", seq_index)):
        if not isinstance(t, Tensor) or t.dtype != torch.int64 or t.dim() != 2 or t.shape[0] != b or t.shape[1] < 1:
            raise ValueError(f"{name} must be an int64 tensor [B={b}, P >= 1]")
    if node_index.shape != seq_index.shape:
        raise ValueError("node_index and seq_index must have the same shape [B, P]")
    if not isinstance(seq, Tensor) or seq.dim() != 3 or seq.shape[0] != b:
        raise ValueError(f"sequence_data must be [B={b}, L, V]")
    dev = graph.ndata["x"].device
    cols = _seq_columns(seq_columns, dev)
    ni, si = node_index.to(dev), seq_index.to(dev)
    L, V = seq.shape[1], seq.shape[2]
    counts = graph.batch_num_nodes().to(dev)
    bad = torch.stack([((ni == -1) != (si == -1)).any(), ((ni < -1) | (si < -1)).any(),
                       (ni >= counts.unsqueeze(1)).any(), (si >= L).any(), _columns_bad(cols, V)]).tolist()
    if bad[0]:
        raise ValueError("a site is absent (-1) in node_index but not in seq_index, or the other way round")
    if bad[1]:
        raise ValueError("site indices must be >= -1 (-1 = absent site)")
    if bad[2]:
        raise ValueError("node_index points past its graph's node count (it is graph-local)")
    if bad[3]:
        raise ValueError(f"seq_index points past the sequence length L={L}")
    if bad[4]:
        raise ValueError(f"seq_columns must map the 20 residue columns to distinct sequence columns in [0, V={V})")
    return ni.contiguous(), si.contiguous(), cols.contiguous()


def _scan(model, scorer, graph, seq, prop, ni, si, cols, max_graphs):
    """Every variant of ``graph`` in replica passes -> (logits [B,P,20,K], prob_mean, prob_std, native)."""
    b, n_sites = ni.shape
    x = graph.ndata["x"].detach().contiguous()
    seq = seq.detach().contiguous()
    sites = scan_sites(n_sites, x.device)
    passes = scan_passes(sites.shape[0], b, max_graphs)
    flag = torch.zeros(1, dtype=torch.int32, device=x.device)

    def run_pass(j, r, g, seq_r, prop_r, e_r):
        IF._C.mutscan_expand(x, graph.node_off, ni, seq, si, cols, sites[j:j + r], g.ndata["x"], seq_r, flag)
        return scorer.score(_encode(model, g, seq_r, prop_r) + (e_r,), r=r)

    reps = replicas(passes, sequence_replica(graph, seq, prop, scorer.item[4]))
    logits, mean, std = score_replicas(scorer, passes, reps, run_pass)
    check_one_hot(flag, "a site row")
    absent = ni < 0
    shape = (n_sites, N_RESIDUES, b)
    logits = logits.reshape(*shape, logits.shape[2]).permute(2, 0, 1, 3).contiguous()
    mean = mean.reshape(shape).permute(2, 0, 1).contiguous()
    std = std.reshape(shape).permute(2, 0, 1).contiguous()
    for t in (logits, mean, std):
        t[absent] = float("nan")
    return logits, mean, std, native_residues(graph, ni)


def mutational_scan(model, graph_data, sequence_data, peptide_property, node_index: Tensor, seq_index: Tensor, *,
                    seq_columns, eps: Optional[Tensor] = None, samples: int = 1, max_graphs: int = 4096) -> Scan:
    """Scores of ``model(graph_data, sequence_data, peptide_property)[3]`` (the logit) for every single-residue variant:
    each of the 20 residue types at each site p of each sample b.

    ``node_index`` / ``seq_index`` int64 [B, P]: the site's node row in its graph (graph-local) and its row of
    ``sequence_data``; -1 in both marks an absent site (a shorter peptide).  ``seq_columns`` [20]: the sequence column of
    each residue-feature column.  ``eps`` [K, B, latent] gives the draws, or one ``model.sample_eps`` call of [K*B, latent]
    (K = ``samples``) makes them; every variant of sample b uses sample b's draws.  Runs in passes of at most
    ``max_graphs`` graphs.  Follows ``model.forward`` for the eight classes ``predictive`` supports; the model must be in
    eval mode; no_grad, and every ``.grad`` is left untouched.  The native residue's column is scored like any other and
    equals ``base`` up to rounding."""
    _check(model, samples, (_Hybrid, _Comparative), "mutational_scan", _CLASSES)
    ni, si, cols = _site_tables(graph_data, sequence_data, node_index, seq_index, seq_columns)
    scan_passes(1, graph_data.n_graphs, max_graphs)
    with torch.no_grad():
        scorer = _scorer(model, graph_data, sequence_data, peptide_property, eps, samples)
        out = _scan(model, scorer, graph_data, sequence_data, peptide_property, ni, si, cols, max_graphs)
    return Scan(*out, scorer.base)


def mutational_scan_pair(model, graph_pair, sequence_pair, property_pair, node_index: Tensor, seq_index: Tensor, *,
                         seq_columns, eps=None, samples: int = 1, max_graphs: int = 4096) -> Scan:
    """``mutational_scan`` of the cancer item of ``model.forward_comparative(graph_pair, sequence_pair, property_pair)``
    against its fixed wild type, for the four comparative classes.  The sites index the cancer item.

    The wild type is encoded once, at batch B, and its encoded tensors are repeated for every pass.  ``eps`` = (eps_c,
    eps_w), each [K, B, latent], or one ``model.sample_eps`` call of [K*B, latent] per item, cancer first.  Without
    ``use_wt_for_downstream`` the wild type is neither run nor drawn for.  ``base`` equals ``predictive_pair`` on the same
    draws."""
    _check(model, samples, _Comparative, "mutational_scan_pair", _PAIR_CLASSES)
    gc = graph_pair[0]
    ni, si, cols = _site_tables(gc, sequence_pair[0], node_index, seq_index, seq_columns)
    scan_passes(1, gc.n_graphs, max_graphs)
    with torch.no_grad():
        scorer = _scorer_pair(model, graph_pair, sequence_pair, property_pair, eps, samples)
        out = _scan(model, scorer, gc, sequence_pair[0], property_pair[0], ni, si, cols, max_graphs)
    return Scan(*out, scorer.base)


# ---- variant libraries: any substitution list on any sample -----------------------------------------------------------
@dataclass
class VariantScores:
    """Scores of a library of multi-site residue variants, in the caller's order."""
    logits: Tensor        # [V, K]  logit of variant v on draw k of its base sample
    prob_mean: Tensor     # [V]     mean of sigmoid(logit) over the draws
    prob_std: Tensor      # [V]     population standard deviation of sigmoid(logit) over the draws
    base: Predictive      # the unmutated batch on the same draws


def _variant_tables(graph, seq, sample, offsets, node_index, seq_index, residue, seq_columns, max_graphs):
    """The checked library on the batch's device: (sample, offsets, node_index, seq_index, residue, seq_columns, node and
    edge count of each variant, their running sums [V+1], the passes, every pass's node and edge totals).  One host read
    for all checks and totals."""
    b = graph.n_graphs
    for name, t in (("sample", sample), ("offsets", offsets), ("node_index", node_index), ("seq_index", seq_index),
                    ("residue", residue)):
        if not isinstance(t, Tensor) or t.dtype != torch.int64 or t.dim() != 1:
            raise ValueError(f"{name} must be a one-dimensional int64 tensor")
    n_var, n_sub = sample.shape[0], node_index.shape[0]
    if n_var < 1:
        raise ValueError("the library needs at least one variant")
    if offsets.shape[0] != n_var + 1:
        raise ValueError(f"offsets must hold V + 1 = {n_var + 1} entries (the substitution CSR of the V variants)")
    if seq_index.shape[0] != n_sub or residue.shape[0] != n_sub:
        raise ValueError("node_index, seq_index and residue must hold one entry per substitution")
    if not isinstance(seq, Tensor) or seq.dim() != 3 or seq.shape[0] != b:
        raise ValueError(f"sequence_data must be [B={b}, L, V]")
    passes = variant_passes(n_var, max_graphs)
    dev = graph.ndata["x"].device
    cols = _seq_columns(seq_columns, dev)
    smp, off, ni, si, res = (t.to(dev).contiguous() for t in (sample, offsets, node_index, seq_index, residue))
    L, V = seq.shape[1], seq.shape[2]
    sb = smp.clamp(0, b - 1)
    nv, ev = graph.batch_num_nodes().to(dev)[sb].contiguous(), graph.batch_num_edges().to(dev)[sb].contiguous()
    ncs, ecs, node_tot, edge_tot = pass_totals(nv, ev, n_var, len(passes), max_graphs)
    owner = (torch.searchsorted(off, torch.arange(n_sub, device=dev), right=True) - 1).clamp(0, n_var - 1)
    last = torch.arange(n_sub, device=dev)
    twice = lambda key: (key.sort().values.diff() == 0).any()
    node_key = torch.where(ni >= 0, owner * (int(graph.max_nodes) + 1) + ni, -1 - last)
    seq_key = owner * L + si
    bad = torch.stack([((smp < 0) | (smp >= b)).any(), (off[0] != 0) | (off.diff() < 0).any() | (off[-1] != n_sub),
                       ((ni < -1) | (ni >= nv[owner])).any(), ((si < 0) | (si >= L)).any(),
                       ((res < 0) | (res >= N_RESIDUES)).any(), _columns_bad(cols, V), twice(node_key),
                       twice(seq_key)]).long()
    vals = torch.cat([bad, node_tot, edge_tot]).tolist()
    if vals[0]:
        raise ValueError(f"sample must index the batch: every entry in [0, B={b})")
    if vals[1]:
        raise ValueError(f"offsets must start at 0, never decrease and end at S={n_sub}")
    if vals[2]:
        raise ValueError("node_index must lie in [-1, n_b) of its variant's base graph (graph-local, -1 = not in the graph)")
    if vals[3]:
        raise ValueError(f"seq_index points outside the sequence length L={L}")
    if vals[4]:
        raise ValueError("residue must be a residue-feature column in [0, 20)")
    if vals[5]:
        raise ValueError(f"seq_columns must map the 20 residue columns to distinct sequence columns in [0, V={V})")
    if vals[6]:
        raise ValueError("a variant substitutes the same node row twice")
    if vals[7]:
        raise ValueError("a variant substitutes the same sequence row twice")
    n_pass = len(passes)
    return (smp, off, ni, si, res, cols, nv, ev, ncs, ecs, passes, vals[8:8 + n_pass], vals[8 + n_pass:])


def _score_variants(model, scorer, graph, seq, prop, tables):
    """Every variant of the library in gathered passes -> (logits [V,K], prob_mean [V], prob_std [V])."""
    smp, off, ni, si, res, cols, nv, ev, ncs, ecs, passes, node_totals, edge_totals = tables
    seq = seq.detach().contiguous()
    prop = prop.detach().contiguous()
    e = scorer.item[4]
    flag = torch.zeros(1, dtype=torch.int32, device=smp.device)

    def expand(j, r, inputs, outputs):
        seq_p = torch.empty(r, *seq.shape[1:], dtype=torch.float32, device=smp.device)
        IF._C.variant_expand(*inputs, seq, smp[j:j + r], off[j:j + r + 1], ni, si, res, cols, *outputs, seq_p, flag)
        return seq_p

    out = score_gathered(scorer, graph, smp, nv, ev, ncs, ecs, passes, node_totals, edge_totals, expand,
                         lambda g, sp, seq_p: _encode(model, g, seq_p, prop[sp]) + (e[:, sp],))
    check_one_hot(flag, "a substituted row")
    return out


def score_variants(model, graph_data, sequence_data, peptide_property, sample: Tensor, offsets: Tensor,
                   node_index: Tensor, seq_index: Tensor, residue: Tensor, *, seq_columns, eps: Optional[Tensor] = None,
                   samples: int = 1, max_graphs: int = 4096) -> VariantScores:
    """Scores of ``model(graph_data, sequence_data, peptide_property)[3]`` (the logit) for a library of V multi-site residue
    variants of the batch's samples.

    Variant v is sample ``sample[v]`` (int64 [V], any order, any number of times) with the substitutions
    ``offsets[v]`` .. ``offsets[v+1] - 1`` (int64 [V+1], from 0 to S) of the int64 [S] tables: residue-feature column
    ``residue[s]`` replaces the residue at graph-local node row ``node_index[s]`` (-1 when the graph does not hold that
    residue, e.g. an HLA position present only in the sequence) and at sequence row ``seq_index[s]`` (always required),
    written as column ``seq_columns[residue[s]]``.  A variant with no substitution is its base sample.  Coordinates and
    contacts stay those of the base structure: nothing is re-folded.  No row may be substituted twice within a variant.

    ``eps`` [K, B, latent] gives the draws, or one ``model.sample_eps`` call of [K*B, latent] (K = ``samples``) makes
    them; variant v uses the draws of sample ``sample[v]``, so variants of one sample differ by their substitutions only.
    The variants run in passes of at most ``max_graphs``, in the caller's order.  Classes, eval mode, no_grad and
    ``.grad`` as in ``mutational_scan``."""
    _check(model, samples, (_Hybrid, _Comparative), "score_variants", _CLASSES)
    tables = _variant_tables(graph_data, sequence_data, sample, offsets, node_index, seq_index, residue, seq_columns,
                             max_graphs)
    with torch.no_grad():
        scorer = _scorer(model, graph_data, sequence_data, peptide_property, eps, samples)
        out = _score_variants(model, scorer, graph_data, sequence_data, peptide_property, tables)
    return VariantScores(*out, scorer.base)


def score_variants_pair(model, graph_pair, sequence_pair, property_pair, sample: Tensor, offsets: Tensor,
                        node_index: Tensor, seq_index: Tensor, residue: Tensor, *, seq_columns, eps=None, samples: int = 1,
                        max_graphs: int = 4096) -> VariantScores:
    """``score_variants`` of the cancer item of ``model.forward_comparative(graph_pair, sequence_pair, property_pair)``
    against its fixed wild type, for the four comparative classes.  The library indexes the cancer item.

    The wild type is encoded once, at batch B; each pass gathers its four encoded tensors and its draws by ``sample``.
    ``eps`` = (eps_c, eps_w), each [K, B, latent], or one ``model.sample_eps`` call of [K*B, latent] per item, cancer
    first.  Without ``use_wt_for_downstream`` the wild type is neither run nor drawn for.  ``base`` equals
    ``predictive_pair`` on the same draws."""
    _check(model, samples, _Comparative, "score_variants_pair", _PAIR_CLASSES)
    gc = graph_pair[0]
    tables = _variant_tables(gc, sequence_pair[0], sample, offsets, node_index, seq_index, residue, seq_columns, max_graphs)
    with torch.no_grad():
        scorer = _scorer_pair(model, graph_pair, sequence_pair, property_pair, eps, samples)
        out = _score_variants(model, scorer, gc, sequence_pair[0], property_pair[0], tables)
    return VariantScores(*out, scorer.base)
