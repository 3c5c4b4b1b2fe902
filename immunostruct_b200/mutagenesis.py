"""In-silico saturation mutagenesis: the score of every single-residue substitution at chosen sites of each sample.

For each sample b and site p, each of the 20 residue types c replaces the native residue at two places: the residue columns
of one node row of the graph (``node_index[b, p]``, graph-local) and one row of the sequence one-hot
(``seq_index[b, p]``, written as column ``seq_columns[c]``).  Coordinates and contacts stay those of the input structure:
nothing is re-folded.  Neither the repository nor the reference pins where the peptide sits in the graph or how the
graph's 20 residue columns map onto the sequence alphabet, so the caller names the sites and the map; a device check
rejects a site row that is not exactly one-hot (a padded or masked row) or that contradicts ``seq_columns``.

The P x 20 variants of the batch run in passes of r = min(remaining, max_graphs // B) copies of the whole batch: one
kernel writes a pass's mutant features from the resident batch (``is_mutscan_expand``, csrc/mutscan.cu), the copies'
topology is collated once per distinct r, the trunk and the VAE encoder run once per pass and the multi-draw head
(``is_head_mc_infer``) scores every draw.  The reparameterisation noise is common to all variants of a sample (common
random numbers), so the difference between two variants is the effect of the substitution alone.

An entry agrees with the fused eval forward of the B-sample mutant batch on the same draw to rounding, not bit for bit:
where a graph sits in the batch changes two summation orders, the edge kernel's per-tile segment-sum MMA (a node's
in-edges land at other positions of a 128-edge tile) and the K-slice count of the vae_fc1 GEMM (it follows the row count).
"""
from __future__ import annotations

from dataclasses import dataclass
from typing import Optional

import torch

from . import functional as IF
from .comparative_models import _Comparative
from .hybrid_models import _Hybrid
from .predictive import _CLASSES, _PAIR_CLASSES, Predictive, _check, _draws, _encode, _head_params, _pair_items

Tensor = torch.Tensor
N_RESIDUES = 20


@dataclass
class Scan:
    """Scores of the single-residue variants; entries of absent sites are NaN."""
    logits: Tensor        # [B, P, 20, K]  logit of sample b with residue column c at site p, draw k
    prob_mean: Tensor     # [B, P, 20]     mean of sigmoid(logit) over the draws
    prob_std: Tensor      # [B, P, 20]     population standard deviation of sigmoid(logit) over the draws
    native: Tensor        # [B, P]         residue column of the input at the site, -1 = absent site
    base: Predictive      # the unmutated batch on the same draws


def scan_passes(n_copies: int, b: int, max_graphs: int):
    """(first copy, number of copies) of each pass: r = min(remaining, max_graphs // B) copies of the B-graph batch."""
    if b > max_graphs:
        raise ValueError(f"the batch has {b} graphs, more than max_graphs={max_graphs}")
    per = max_graphs // b
    return [(j, min(per, n_copies - j)) for j in range(0, n_copies, per)]


def scan_sites(n_sites: int, device=None) -> Tensor:
    """The copies of a scan in order, int32 [P*20, 2] = (site p, residue column c), site-major."""
    p = torch.arange(n_sites, dtype=torch.int32).repeat_interleave(N_RESIDUES)
    c = torch.arange(N_RESIDUES, dtype=torch.int32).repeat(n_sites)
    return torch.stack([p, c], 1).to(device)


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
    cols = torch.as_tensor(seq_columns)
    if cols.dtype.is_floating_point or cols.dtype == torch.bool or cols.shape != (N_RESIDUES,):
        raise ValueError("seq_columns must hold 20 integers: the sequence column of each residue-feature column")
    dev = graph.ndata["x"].device
    ni, si, cols = node_index.to(dev), seq_index.to(dev), cols.to(dev, torch.int64)
    L, V = seq.shape[1], seq.shape[2]
    counts = graph.batch_num_nodes().to(dev)
    bad = torch.stack([((ni == -1) != (si == -1)).any(), ((ni < -1) | (si < -1)).any(),
                       (ni >= counts.unsqueeze(1)).any(), (si >= L).any(),
                       ((cols < 0) | (cols >= V)).any() | (cols.unique().numel() != N_RESIDUES)]).tolist()
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


def _check_scan(model, samples, kinds, what, names):
    _check(model, samples, kinds, what, names)
    if model.training:
        raise RuntimeError(f"{what} needs model.eval(): dropout would change the function between variants")


def _run(model, graph, seq, prop, ni, si, cols, e, items_of, max_graphs):
    """Every variant of ``graph`` in passes -> (logits [B,P,20,K], prob_mean, prob_std, native).  ``items_of(item, r)``
    turns the mutant item of an r-copy pass into the head's item list."""
    params = _head_params(model)
    b, n_sites = ni.shape
    x = graph.ndata["x"].detach().contiguous()
    seq = seq.detach().contiguous()
    prop = prop.detach().contiguous()
    L, V, k = seq.shape[1], seq.shape[2], e.shape[0]
    sites = scan_sites(n_sites, x.device)
    n_copies = sites.shape[0]
    logits = torch.empty(n_copies, b, k, dtype=torch.float32, device=x.device)
    mean = torch.empty(n_copies, b, dtype=torch.float32, device=x.device)
    std = torch.empty_like(mean)
    flag = torch.zeros(1, dtype=torch.int32, device=x.device)
    passes = {}
    for j, r in scan_passes(n_copies, b, max_graphs):
        if r not in passes:                     # topology of r copies, collated once; only the features change per pass
            passes[r] = (graph.replicate(r), torch.empty(r * b, L, V, dtype=torch.float32, device=x.device),
                         prop.repeat(r, 1))
        g, seq_r, prop_r = passes[r]
        IF._C.mutscan_expand(x, graph.node_off, ni, seq, si, cols, sites[j:j + r], g.ndata["x"], seq_r, flag)
        item = _encode(model, g, seq_r, prop_r) + (e.repeat(1, r, 1),)
        lg, m, s = IF._C.head_mc_infer(items_of(item, r), *params)
        logits[j:j + r], mean[j:j + r], std[j:j + r] = lg.reshape(r, b, k), m.reshape(r, b), s.reshape(r, b)
    if flag.item():
        raise ValueError("a site row is not exactly one-hot in the graph's residue columns or in the sequence, or its "
                         "sequence column is not seq_columns[residue column] (a padded or masked row, or a wrong map)")
    absent = ni < 0
    shape = (n_sites, N_RESIDUES, b)
    logits = logits.reshape(*shape, k).permute(2, 0, 1, 3).contiguous()
    mean = mean.reshape(shape).permute(2, 0, 1).contiguous()
    std = std.reshape(shape).permute(2, 0, 1).contiguous()
    for t in (logits, mean, std):
        t[absent] = float("nan")
    rows = graph.node_off[:-1].unsqueeze(1) + ni.clamp_min(0)
    native = torch.where(absent, -1, x[rows.reshape(-1), :N_RESIDUES].argmax(1).reshape(b, n_sites))
    return logits, mean, std, native


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
    _check_scan(model, samples, (_Hybrid, _Comparative), "mutational_scan", _CLASSES)
    ni, si, cols = _site_tables(graph_data, sequence_data, node_index, seq_index, seq_columns)
    scan_passes(1, graph_data.n_graphs, max_graphs)
    pair = isinstance(model, _Comparative) and model.use_wt_for_downstream
    with torch.no_grad():
        base_item = _encode(model, graph_data, sequence_data, peptide_property)
        e = _draws(model, eps, samples, graph_data.n_graphs, base_item[1])
        base_item += (e,)
        base = Predictive(*IF._C.head_mc_infer([base_item, base_item] if pair else [base_item], *_head_params(model)))
        out = _run(model, graph_data, sequence_data, peptide_property, ni, si, cols, e,
                   lambda item, r: [item, item] if pair else [item], max_graphs)
    return Scan(*out, base)


def mutational_scan_pair(model, graph_pair, sequence_pair, property_pair, node_index: Tensor, seq_index: Tensor, *,
                         seq_columns, eps=None, samples: int = 1, max_graphs: int = 4096) -> Scan:
    """``mutational_scan`` of the cancer item of ``model.forward_comparative(graph_pair, sequence_pair, property_pair)``
    against its fixed wild type, for the four comparative classes.  The sites index the cancer item.

    The wild type is encoded once, at batch B, and its encoded tensors are repeated for every pass.  ``eps`` = (eps_c,
    eps_w), each [K, B, latent], or one ``model.sample_eps`` call of [K*B, latent] per item, cancer first.  Without
    ``use_wt_for_downstream`` the wild type is neither run nor drawn for.  ``base`` equals ``predictive_pair`` on the same
    draws."""
    _check_scan(model, samples, _Comparative, "mutational_scan_pair", _PAIR_CLASSES)
    n = _pair_items(model, eps)
    gc = graph_pair[0]
    ni, si, cols = _site_tables(gc, sequence_pair[0], node_index, seq_index, seq_columns)
    scan_passes(1, gc.n_graphs, max_graphs)
    with torch.no_grad():
        items = []
        for i in range(n):
            item = _encode(model, graph_pair[i], sequence_pair[i], property_pair[i])
            k = samples if eps is None else eps[0].shape[0]
            items.append(item + (_draws(model, None if eps is None else eps[i], k, item[1].shape[0], item[1]),))
        base = Predictive(*IF._C.head_mc_infer(items, *_head_params(model)))
        wt = items[1] if n == 2 else None

        def items_of(item, r):
            if wt is None:
                return [item]
            return [item, tuple(t.repeat(1, r, 1) if t.dim() == 3 else t.repeat(r, 1) for t in wt)]

        out = _run(model, gc, sequence_pair[0], property_pair[0], ni, si, cols, items[0][4], items_of, max_graphs)
    return Scan(*out, base)
