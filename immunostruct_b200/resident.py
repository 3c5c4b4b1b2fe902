"""Pass plans and pass loops of the analyses that score many variants of a batch already on the device
(``mutagenesis``, ``design``, ``occlusion``, ``coordnoise``).

Each analysis makes a ``predictive._scorer`` (or ``_scorer_pair``) of the base batch and runs its variants in passes of
one of two layouts:

* replica passes: r copies of the whole batch in the layout of ``GraphBatch.replicate(r)``, r = min(remaining,
  ``max_graphs`` // B) (``scan_passes``).  The topology of every distinct r is collated once, before the first pass, and
  a pass only rewrites features.
* gathered passes: runs of up to ``max_graphs`` variants in order (``variant_passes``), each variant a graph gathered
  from its base sample with its own node and edge counts.  A pass's topology is collated per pass; its buffers are sized
  by node and edge totals returned by the call's one validation read (``pass_totals``).

Nothing is read back between passes: an expansion kernel's flag is read once, after the last pass.
"""
from __future__ import annotations

import torch

from .graph import GraphBatch
from .predictive import _repeat

N_RESIDUES = 20


def scan_passes(n_copies: int, b: int, max_graphs: int):
    """(first copy, number of copies) of each pass: r = min(remaining, max_graphs // B) copies of the B-graph batch."""
    if b > max_graphs:
        raise ValueError(f"the batch has {b} graphs, more than max_graphs={max_graphs}")
    per = max_graphs // b
    return [(j, min(per, n_copies - j)) for j in range(0, n_copies, per)]


def variant_passes(n_variants: int, max_graphs: int):
    """(first variant, number of variants) of each pass: consecutive runs of at most ``max_graphs`` variants."""
    if max_graphs < 1:
        raise ValueError(f"max_graphs must be >= 1, got {max_graphs}")
    return [(j, min(max_graphs, n_variants - j)) for j in range(0, n_variants, max_graphs)]


def pass_totals(nv, ev, n_var, n_slots, max_graphs):
    """Device tensors (ncs, ecs, node totals, edge totals): the running sums [V+1] of the variants' node counts ``nv``
    and edge counts ``ev``, and the totals [n_slots] of the first n_slots runs of ``max_graphs`` variants.  ``n_var``
    (an int, or a device count when only the device knows it) ends the last run; runs past it total 0."""
    zero = torch.zeros(1, dtype=torch.int64, device=nv.device)
    ncs, ecs = torch.cat([zero, nv.cumsum(0)]), torch.cat([zero, ev.cumsum(0)])
    first = torch.arange(n_slots, device=nv.device) * max_graphs
    end = (first + max_graphs).clamp_max(n_var)
    first = first.clamp_max(n_var)
    return ncs, ecs, ncs[end] - ncs[first], ecs[end] - ecs[first]


def replicas(passes, build):
    """``build(r)`` for every distinct r of ``passes``, in increasing r: what a pass of r copies of the batch needs (the
    replica, collated by ``GraphBatch.replicate``, and any repeated tensors).  Called before the first pass."""
    return {r: build(r) for r in sorted({r for _, r in passes})}


def sequence_replica(graph, seq, prop, eps):
    """``build`` of the replica passes that rewrite node rows and sequence rows: r -> (the r-copy replica of ``graph``, a
    sequence buffer [rB, L, V], ``prop`` and ``eps`` repeated for the r copies)."""
    dev = graph.ndata["x"].device
    return lambda r: (graph.replicate(r), torch.empty(r * seq.shape[0], *seq.shape[1:], dtype=torch.float32, device=dev),
                      _repeat(prop, r), _repeat(eps, r))


def score_replicas(scorer, passes, reps, run_pass):
    """Every replica pass (j, r) of ``passes``: ``run_pass(j, r, *reps[r])`` writes copies j .. j+r-1 of the batch into
    the replicas of r and returns their ``scorer.score`` -> (logits [n, B, K], prob_mean [n, B], prob_std [n, B]) of the
    n copies."""
    k, b, _ = scorer.item[4].shape
    n = passes[-1][0] + passes[-1][1]
    f32 = dict(dtype=torch.float32, device=scorer.item[4].device)
    logits, mean, std = torch.empty(n, b, k, **f32), torch.empty(n, b, **f32), torch.empty(n, b, **f32)
    for j, r in passes:
        lg, m, s = run_pass(j, r, *reps[r])
        logits[j:j + r], mean[j:j + r], std[j:j + r] = lg.reshape(r, b, k), m.reshape(r, b), s.reshape(r, b)
    return logits, mean, std


def score_gathered(scorer, graph, sample, nv, ev, ncs, ecs, passes, node_totals, edge_totals, expand, pass_item):
    """Every gathered pass -> (logits [V, K], prob_mean [V], prob_std [V]).  Variant v has ``nv[v]`` rows and ``ev[v]``
    edges (running sums ``ncs``, ``ecs``) and base sample ``sample[v]``; pass i of ``passes`` holds ``node_totals[i]``
    rows and ``edge_totals[i]`` edges.

    Per pass (j, r): ``expand(j, r, inputs, outputs)`` launches the expansion of variants j .. j+r-1 with ``inputs`` =
    (x, node_off, edge_off, src_local, dst_local, edge_attr) of ``graph`` and ``outputs`` = (node_out, edge_out, x_p,
    src_p, dst_p, edge_attr_p), and returns anything its item needs; the pass's topology is collated; ``pass_item(g,
    sample_p, expanded)`` returns the item of the collated pass ``g``, whose variants have base samples ``sample_p``.  The
    head reads the fixed wild type gathered by ``sample_p``."""
    x = graph.ndata["x"].detach().contiguous()
    ea = graph.edata["edge_attr"].detach().contiguous()
    inputs = (x, graph.node_off, graph.edge_off, graph._src_local.contiguous(), graph._dst_local.contiguous(), ea)
    k, n_var = scorer.item[4].shape[0], sample.shape[0]
    f32, i64 = dict(dtype=torch.float32, device=x.device), dict(dtype=torch.int64, device=x.device)
    logits, mean, std = torch.empty(n_var, k, **f32), torch.empty(n_var, **f32), torch.empty(n_var, **f32)
    for (j, r), n_p, e_p in zip(passes, node_totals, edge_totals):
        outputs = (ncs[j:j + r + 1] - ncs[j], ecs[j:j + r + 1] - ecs[j], torch.empty(n_p, 23, **f32),
                   torch.empty(e_p, **i64), torch.empty(e_p, **i64), torch.empty(e_p, *ea.shape[1:], **f32))
        expanded = expand(j, r, inputs, outputs)
        # the pass's topology is gathered, not a replica of the batch: collated per pass
        g = GraphBatch(*outputs[2:], nv[j:j + r], ev[j:j + r], max_nodes=graph.max_nodes, collate_now=False)
        g._collate()
        sp = sample[j:j + r]
        logits[j:j + r], mean[j:j + r], std[j:j + r] = scorer.score(pass_item(g, sp, expanded), sample=sp)
    return logits, mean, std


def native_residues(graph, node_index):
    """The residue column of each site row, int64 [B, P]: row ``node_index[b, p]`` of graph b (graph-local), -1 at an
    absent site (node_index -1)."""
    rows = graph.node_off[:-1].unsqueeze(1) + node_index.clamp_min(0)
    x = graph.ndata["x"].detach()
    return torch.where(node_index < 0, -1, x[rows.reshape(-1), :N_RESIDUES].argmax(1).reshape(node_index.shape))


def check_one_hot(flag, rows):
    """The substitution kernels' device flag, read once after the last pass: raised for ``rows`` (e.g. "a site row")
    that were not exactly one-hot or did not follow ``seq_columns``."""
    if flag.item():
        raise ValueError(f"{rows} is not exactly one-hot in the graph's residue columns or in the sequence, or its "
                         "sequence column is not seq_columns[residue column] (a padded or masked row, or a wrong map)")
