"""Structural uncertainty: the score of every sample over seeded perturbations of its coordinates.

The inputs are predicted structures, and the EGNN stack reads the coordinates in every layer (``||x_i - x_j||^2`` in the
edge MLP, the coordinate update of the first layers).  ``coordinate_ensemble`` carries a per-residue positional error
into the score: structure draw m of sample b is sample b with the coordinates (x23 columns 20..22) of every node row i
replaced by ``x + sigma_i z``, z three standard normals of a counter-based stream keyed on (seed, item, m, b, local row
a).  Residue columns, edges, edge attributes, the sequence and the properties are unchanged, and contacts are not
re-derived: the graph's edges stay the interaction graph of the input structure (nothing is re-folded).  A row with
sigma 0 is copied bit-exact, so a per-row ``sigma`` is also the selection (e.g. the peptide rows only).

The stream depends on the key alone: a given (seed, m, b) is the same structure whatever ``max_graphs`` is and on every
run.  The K latent draws ``eps [K, B, latent]`` are shared by all M structures of a sample (common random numbers), so
the spread over m is the structural effect alone, and the law of total variance splits the spread of the probability
into a structural and a latent part.

The M structures run in passes of r = min(remaining, max_graphs // B) copies of the batch, on the topology of r copies
collated once per distinct r before the first pass.  Per pass ``is_coord_noise_expand`` (csrc/coordnoise.cu) writes the
r perturbed copies, the structure trunk runs on them, and ``is_head_mc_infer`` scores every draw on the sample's encoded
sequence; the VAE encoder runs once per call, at batch B.  Every argument is checked before the first launch, with at
most one host read (sigma), and nothing is read back between passes.

An entry agrees with the fused eval forward of the host-built perturbed batch on the same draw to rounding, not bit for
bit: where a graph sits in a batch changes two summation orders (mutagenesis module docstring, DESIGN 4.4c).
"""
from __future__ import annotations

import math
from dataclasses import dataclass
from typing import Optional

import torch

from . import functional as IF
from .comparative_models import _Comparative
from .hybrid_models import _Hybrid
from .predictive import _CLASSES, _PAIR_CLASSES, Predictive, _check, _repeat, _scorer, _scorer_pair
from .resident import replicas, scan_passes, score_replicas

Tensor = torch.Tensor


@dataclass
class CoordinateEnsemble:
    """Scores of M seeded coordinate perturbations of every sample on K latent draws, and the split of their spread."""
    logits: Tensor          # [B, M, K]  logit of structure draw m of sample b on latent draw k
    prob_mean: Tensor       # [B]  mean of sigmoid(logit) over the M K entries
    prob_std: Tensor        # [B]  population standard deviation of sigmoid(logit) over the M K entries
    std_structure: Tensor   # [B]  population standard deviation over m of the mean over k
    std_latent: Tensor      # [B]  square root of the mean over m of the population variance over k
    seed: int               # the seed of the coordinate stream
    base: Predictive        # the unperturbed batch on the same latent draws


def _sigma(sigma, graph, what):
    """sigma as fp32 [ΣN] on the batch's device, and the device bool "not finite or negative" (None for a number)."""
    n, dev = graph.n_nodes, graph.ndata["x"].device
    if isinstance(sigma, (int, float)) and not isinstance(sigma, bool):
        if not (math.isfinite(sigma) and sigma >= 0):
            raise ValueError(f"{what} must be finite and >= 0, got {sigma}")
        return torch.full((n,), float(sigma), dtype=torch.float32, device=dev), None
    if not isinstance(sigma, Tensor) or sigma.dtype != torch.float32 or tuple(sigma.shape) != (n,):
        raise ValueError(f"{what} must be a float or a float32 tensor [ΣN={n}] over the batch's node rows")
    s = sigma.detach().to(dev).contiguous()
    return s, ~(torch.isfinite(s) & (s >= 0)).all()


def _seed(seed):
    if seed is None:        # from torch's default CPU generator, so torch.manual_seed makes a call reproducible
        return int(torch.randint(0, 2 ** 63 - 1, (1,), dtype=torch.int64)[0])
    if not isinstance(seed, int) or isinstance(seed, bool) or not 0 <= seed < 2 ** 64:
        raise ValueError(f"seed must be an integer in [0, 2^64), got {seed!r}")
    return seed


def _checked(structures, seed, b, max_graphs, sigmas):
    """Host checks of the call -> (seed, passes).  ``sigmas``: (name, device bool or None) of each perturbed item; their
    flags are read together, the call's one host read."""
    if not isinstance(structures, int) or isinstance(structures, bool) or structures < 1:
        raise ValueError(f"structures must be an integer >= 1, got {structures!r}")
    if structures > 2 ** 32:
        raise ValueError("structures must be <= 2^32 (the stream's draw counter is 32-bit)")
    seed = _seed(seed)
    passes = scan_passes(structures, b, max_graphs)
    flags = [(name, bad) for name, bad in sigmas if bad is not None]
    if flags:
        read = torch.stack([bad for _, bad in flags]).tolist()
        for (name, _), bad in zip(flags, read):
            if bad:
                raise ValueError(f"{name} must be finite and >= 0 in every row")
    return seed, passes


def _statistics(logits):
    """(prob_mean, prob_std, std_structure, std_latent) [B] of logits [B, M, K], in fp64 and rounded to fp32."""
    p = torch.sigmoid(logits.double())
    mean = p.mean((1, 2))
    std = (p - mean[:, None, None]).square().mean((1, 2)).sqrt()
    pm = p.mean(2)
    std_s = (pm - mean[:, None]).square().mean(1).sqrt()
    std_l = (p - pm[:, :, None]).square().mean(2).mean(1).sqrt()
    return tuple(t.float() for t in (mean, std, std_s, std_l))


def _ensemble(model, scorer, perturbed, passes, seed):
    """Every structure draw in replica passes -> logits [B, M, K].  ``perturbed``: (graph, sigma) of the scored item and,
    when the wild type is perturbed too, of the wild type; item i draws from stream item i.  A wild type that is not
    perturbed stays the scorer's fixed one."""
    encoded = [scorer.item[1:], None if scorer.wt is None else scorer.wt[1:]]
    reps = replicas(passes, lambda r: [(g.replicate(r), tuple(_repeat(t, r) for t in enc))
                                       for (g, _), enc in zip(perturbed, encoded)])
    bases = [(g.ndata["x"].detach().contiguous(), g.node_off, s) for g, s in perturbed]

    def run_pass(j, r, *copies):
        for item, ((x, node_off, s), (g, _)) in enumerate(zip(bases, copies)):
            IF._C.coord_noise_expand(x, node_off, s, seed, item, j, g.ndata["x"])
        items = [(model.structure_embedding(g, project=False)[0].contiguous(),) + enc for g, enc in copies]
        return scorer.score(items[0], r=r, wt=items[1] if len(items) == 2 else None)

    return score_replicas(scorer, passes, reps, run_pass)[0].permute(1, 0, 2).contiguous()


def _result(logits, seed, base):
    return CoordinateEnsemble(logits, *_statistics(logits), seed, base)


def coordinate_ensemble(model, graph, seq, prop, *, sigma, structures: int = 16, seed: Optional[int] = None,
                        eps: Optional[Tensor] = None, samples: int = 1, max_graphs: int = 4096) -> CoordinateEnsemble:
    """Scores of ``model(graph, seq, prop)[3]`` (the logit) over ``structures`` = M seeded perturbations of each
    sample's coordinates: structure draw m moves node row i's coordinates (x23 columns 20..22) by ``sigma_i z``, z three
    standard normals of the stream keyed on (seed, item 0, m, b, graph-local row).  Contacts are not re-derived.

    ``sigma`` is in the coordinates' units (Å for the reference's graphs): a float, or a float32 tensor [ΣN] per row in
    ``graph.ndata['x']`` order, finite and >= 0; a row with sigma 0 stays bit-exact.  ``seed`` in [0, 2^64), by default
    one 63-bit integer from torch's default CPU generator (the seed used is returned).  ``eps`` [K, B, latent] gives
    the latent draws, or one ``model.sample_eps`` call of [K*B, latent] (K = ``samples``) makes them; all M structures
    of a sample share its draws.  Structures run in passes of at most ``max_graphs`` graphs.  Follows ``model.forward``
    for the eight classes ``predictive`` supports; the model must be in eval mode; no_grad, and every ``.grad`` is left
    untouched.  ``prob_std^2 = std_structure^2 + std_latent^2`` (the law of total variance, computed in fp64)."""
    _check(model, samples, (_Hybrid, _Comparative), "coordinate_ensemble", _CLASSES)
    s, bad = _sigma(sigma, graph, "sigma")
    seed, passes = _checked(structures, seed, graph.n_graphs, max_graphs, [("sigma", bad)])
    with torch.no_grad():
        scorer = _scorer(model, graph, seq, prop, eps, samples)
        logits = _ensemble(model, scorer, [(graph, s)], passes, seed)
    return _result(logits, seed, scorer.base)


def coordinate_ensemble_pair(model, graph_pair, seq_pair, prop_pair, *, sigma, structures: int = 16,
                             seed: Optional[int] = None, eps=None, samples: int = 1,
                             max_graphs: int = 4096) -> CoordinateEnsemble:
    """``coordinate_ensemble`` of ``model.forward_comparative(graph_pair, seq_pair, prop_pair)`` for the four comparative
    classes.  ``sigma`` = (sigma_c, sigma_w), each a float or a float32 tensor over its own batch's node rows: the
    cancer item is perturbed from the stream of item 0 with sigma_c.

    With ``use_wt_for_downstream`` and sigma_w given, the wild type is perturbed too, from its own stream (item 1) and on
    its own replica, and its trunk runs per pass; with sigma_w None it stays fixed, encoded once and repeated per pass.
    Without ``use_wt_for_downstream`` the wild type is neither run nor drawn for, and sigma_w must be None.  ``eps`` =
    (eps_c, eps_w), each [K, B, latent], or one ``model.sample_eps`` call of [K*B, latent] per item, cancer first.
    ``base`` equals ``predictive_pair`` on the same draws."""
    _check(model, samples, _Comparative, "coordinate_ensemble_pair", _PAIR_CLASSES)
    if not isinstance(sigma, (tuple, list)) or len(sigma) != 2 or sigma[0] is None:
        raise ValueError("sigma must be a pair (sigma_c, sigma_w); sigma_w may be None")
    if not model.use_wt_for_downstream and sigma[1] is not None:
        raise ValueError("sigma_w needs use_wt_for_downstream: without it the wild type does not enter the score")
    gc = graph_pair[0]
    b = gc.n_graphs
    if model.use_wt_for_downstream and graph_pair[1].n_graphs != b:
        raise ValueError("the cancer and wild-type batches must hold the same number of graphs")
    s_c, bad_c = _sigma(sigma[0], gc, "sigma_c")
    s_w, bad_w = (None, None) if sigma[1] is None else _sigma(sigma[1], graph_pair[1], "sigma_w")
    seed, passes = _checked(structures, seed, b, max_graphs, [("sigma_c", bad_c), ("sigma_w", bad_w)])
    with torch.no_grad():
        scorer = _scorer_pair(model, graph_pair, seq_pair, prop_pair, eps, samples)
        logits = _ensemble(model, scorer, [(gc, s_c)] + ([] if s_w is None else [(graph_pair[1], s_w)]), passes, seed)
    return _result(logits, seed, scorer.base)
