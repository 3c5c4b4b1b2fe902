"""Beam search over residue substitutions: the combination of residues at chosen sites of each sample that maximises (or
minimises) the score, found in device-resident rounds.

A state of sample b holds one residue-feature column for each of its P named sites (``node_index`` / ``seq_index`` and
``seq_columns`` as in ``mutagenesis.mutational_scan``, -1 in both for an absent site).  The native state is read from
the site rows; applying a state writes its residue into every present site's node row and sequence row (the native
residue is a bit-exact no-op), and coordinates and contacts stay those of the input structure.  A state's key is
sum_p state[p] 20^p (digit 0 at absent sites); keys only deduplicate and break ties, and they cap P at 14.

Round t extends each of the W_t beam states (W_1 = 1: the native state; later W_t = W) at one site: slot (w, p, c) is
state w with site p set to residue c, k = (w P + p) 20 + c.  Every slot is one copy of the whole batch, so a round runs
in passes of r = ``max_graphs`` // B copies, on topology collated once per distinct r before the first round.  A slot is
valid when its parent is, site p is present, c is allowed there and differs from the parent's residue, the new state
lies within ``max_mutations`` of the native state, and it is canonical: no earlier parent yields the same state and no
beam state equals it.  An invalid slot is written as its parent state and its score is ignored.  The next beam is the
top W of the carried beam (with the scores it has) and the round's valid slots by objective
``fmaf(kappa, prob_std, prob_mean)`` (one fp32 rounding), descending with ``maximize``, ties to the smaller key, NaN never
taken; the best objective therefore never gets worse from one round to the next.

Per pass one ``is_design_expand`` writes the slot copies from the resident batch, the trunk and the VAE encoder run once
and ``is_head_mc_infer`` scores every draw; per round one ``is_design_select`` (one CTA per sample) writes the next beam
into the other of two buffers (csrc/mutscan.cu).  Nothing is read back between rounds: the arguments are checked with one
host read before the first launch and the device flag once after the last round.  One ``eps [K, B, latent]`` serves the
base, every round and every candidate of a sample, so rankings compare substitution effects, not draws.
"""
from __future__ import annotations

import math
from dataclasses import dataclass
from typing import Optional

import torch

from . import functional as IF
from .comparative_models import _Comparative
from .hybrid_models import _Hybrid
from .mutagenesis import _site_tables
from .predictive import _CLASSES, _PAIR_CLASSES, Predictive, _check, _encode, _scorer, _scorer_pair
from .resident import (N_RESIDUES, check_one_hot, native_residues, replicas, scan_passes, score_replicas,
                       sequence_replica)

Tensor = torch.Tensor
MAX_SITES = 14            # keys sum_p state[p] 20^p must fit int64
MAX_BEAM = 32             # the slot rule compares a slot with every beam state in one warp ballot


@dataclass
class Design:
    """The final beam of each sample, best first; entries past the number found are invalid (NaN scores)."""
    states: Tensor        # [B, W, P]  int64 residue columns, -1 at absent sites
    n_mutations: Tensor   # [B, W]     Hamming distance to the native state
    valid: Tensor         # [B, W]     bool
    logits: Tensor        # [B, W, K]
    prob_mean: Tensor     # [B, W]
    prob_std: Tensor      # [B, W]
    objective: Tensor     # [B, W]     fmaf(kappa, prob_std, prob_mean)
    history: Tensor       # [B, T+1]   best objective after each round; column 0 is the native state
    base: Predictive      # the native batch on the same draws


def round_slots(n_sites: int, beam: int, rounds: int):
    """Slots (= batch copies) of each round: P 20 for round 1 (the native state alone), W P 20 after."""
    return [(1 if t == 0 else beam) * n_sites * N_RESIDUES for t in range(rounds)]


def _design_args(b, n_sites, allowed, max_mutations, beam, rounds, kappa, dev):
    """Host checks of the search arguments -> (allowed bool [B, P, 20] on ``dev``, max_mutations, rounds, kappa)."""
    if n_sites > MAX_SITES:
        raise ValueError(f"beam search supports at most {MAX_SITES} sites (keys are base-20 int64), got P={n_sites}")
    if not isinstance(beam, int) or not 1 <= beam <= MAX_BEAM:
        raise ValueError(f"beam must be an integer in [1, {MAX_BEAM}], got {beam}")
    m = n_sites if max_mutations is None else max_mutations
    if not isinstance(m, int) or not 1 <= m <= n_sites:
        raise ValueError(f"max_mutations must be an integer in [1, P={n_sites}], got {max_mutations}")
    t = m if rounds is None else rounds
    if not isinstance(t, int) or t < 1:
        raise ValueError(f"rounds must be a positive integer, got {rounds}")
    if not isinstance(kappa, (int, float)) or not math.isfinite(kappa):
        raise ValueError(f"kappa must be a finite number, got {kappa}")
    if allowed is None:
        allowed = torch.ones(b, n_sites, N_RESIDUES, dtype=torch.bool, device=dev)
    if not isinstance(allowed, Tensor) or allowed.dtype != torch.bool or tuple(allowed.shape[-2:]) != (n_sites, N_RESIDUES) \
            or allowed.dim() not in (2, 3) or (allowed.dim() == 3 and allowed.shape[0] != b):
        raise ValueError(f"allowed must be a bool tensor [P={n_sites}, 20] or [B={b}, P, 20]")
    # the kernel computes in fp32: the host's reference objective uses the same kappa
    return allowed.to(dev).expand(b, n_sites, N_RESIDUES), m, t, float(torch.tensor(float(kappa), dtype=torch.float32))


def _search(model, scorer, graph, seq, prop, ni, si, cols, allowed, max_mut, beam, rounds, maximize, kappa, max_graphs):
    """The rounds of one search -> Design fields without ``base``."""
    base = scorer.base
    b, n_sites = ni.shape
    x = graph.ndata["x"].detach().contiguous()
    seq = seq.detach().contiguous()
    k, dev = scorer.item[4].shape[0], x.device
    f32, i64 = dict(dtype=torch.float32, device=dev), dict(dtype=torch.int64, device=dev)
    native = native_residues(graph, ni)
    allowed = allowed.clone()
    allowed.scatter_(2, native.clamp_min(0).unsqueeze(2), torch.ones(b, n_sites, 1, dtype=torch.bool, device=dev))
    nan = float("nan")

    def new_beam():
        return (torch.empty(b, beam, n_sites, **i64), torch.empty(b, beam, **i64), torch.empty(b, beam, **i64),
                torch.zeros(b, beam, dtype=torch.bool, device=dev), torch.full((b, beam, k), nan, **f32),
                torch.full((b, beam), nan, **f32), torch.full((b, beam), nan, **f32), torch.full((b, beam), nan, **f32))

    cur, nxt = new_beam(), new_beam()
    cur[0].copy_(native.unsqueeze(1).expand(b, beam, n_sites))
    cur[1].copy_((native.clamp_min(0) * 20 ** torch.arange(n_sites, **i64)).sum(1, keepdim=True).expand(b, beam))
    cur[2].zero_()
    cur[3][:, 0] = True
    cur[4][:, 0], cur[5][:, 0], cur[6][:, 0] = base.logits, base.prob_mean, base.prob_std
    obj0 = (kappa * base.prob_std.double() + base.prob_mean.double()).float()     # one rounding, as fmaf
    cur[7][:, 0] = obj0
    history = torch.empty(b, rounds + 1, **f32)
    history[:, 0] = obj0
    sizes = round_slots(n_sites, beam, rounds)
    plans = {s: scan_passes(s, b, max_graphs) for s in set(sizes)}
    # topology of r copies, collated before round 1
    reps = replicas([p for plan in plans.values() for p in plan], sequence_replica(graph, seq, prop, scorer.item[4]))
    flag = torch.zeros(1, dtype=torch.int32, device=dev)

    def run_pass(j, r, g, seq_r, prop_r, e_r):             # slots j .. j+r-1 of the current round
        IF._C.design_expand(x, graph.node_off, ni, seq, si, cols, cur, native, allowed, n_states, max_mut, j,
                            g.ndata["x"], seq_r, flag)
        return scorer.score(_encode(model, g, seq_r, prop_r) + (e_r,), r=r)

    for t, n_slots in enumerate(sizes, 1):
        n_states = 1 if t == 1 else beam
        r_logits, r_mean, r_std = score_replicas(scorer, plans[n_slots], reps, run_pass)
        IF._C.design_select(cur, r_logits, r_mean, r_std, native, allowed, ni, n_states, max_mut, kappa, maximize, nxt,
                            history[:, t])
        cur, nxt = nxt, cur
    check_one_hot(flag, "a site row")
    states, _, n_mut, valid, logits, mean, std, obj = cur
    return states, n_mut, valid, logits, mean, std, obj, history


def _prepare(graph, seq, node_index, seq_index, seq_columns, allowed, max_mutations, beam, rounds, kappa, max_graphs):
    ni, si, cols = _site_tables(graph, seq, node_index, seq_index, seq_columns)
    scan_passes(1, graph.n_graphs, max_graphs)
    return (ni, si, cols) + _design_args(graph.n_graphs, ni.shape[1], allowed, max_mutations, beam, rounds, kappa,
                                         ni.device)


def beam_search(model, graph_data, sequence_data, peptide_property, node_index: Tensor, seq_index: Tensor, *, seq_columns,
                allowed: Optional[Tensor] = None, max_mutations: Optional[int] = None, beam: int = 8,
                rounds: Optional[int] = None, maximize: bool = True, kappa: float = 0.0, eps: Optional[Tensor] = None,
                samples: int = 1, max_graphs: int = 4096) -> Design:
    """Beam search for the residues at the named sites of each sample that maximise (``maximize=False``: minimise) the
    objective ``prob_mean + kappa * prob_std`` of ``model(graph_data, sequence_data, peptide_property)[3]`` over the draws.

    ``node_index`` / ``seq_index`` int64 [B, P] (P <= 14) and ``seq_columns`` as in ``mutational_scan``.  ``allowed``
    bool [P, 20] or [B, P, 20] (default all True; the native residue is always allowed) restricts the residues of each
    site; ``max_mutations`` in [1, P] (default P) bounds the Hamming distance to the native state.  ``beam`` = W in
    [1, 32] states are kept per sample for ``rounds`` rounds (default ``max_mutations``); each round changes one site of
    each kept state.  ``eps`` [K, B, latent] gives the draws, or one ``model.sample_eps`` call of [K*B, latent]
    (K = ``samples``) makes them; every candidate of sample b uses sample b's draws.  Rounds run in passes of at most
    ``max_graphs`` graphs.  Follows ``model.forward`` for the eight classes ``predictive`` supports; the model must be in
    eval mode; no_grad, and every ``.grad`` is left untouched."""
    _check(model, samples, (_Hybrid, _Comparative), "beam_search", _CLASSES)
    ni, si, cols, allowed, max_mut, rounds, kappa = _prepare(graph_data, sequence_data, node_index, seq_index, seq_columns,
                                                             allowed, max_mutations, beam, rounds, kappa, max_graphs)
    with torch.no_grad():
        scorer = _scorer(model, graph_data, sequence_data, peptide_property, eps, samples)
        out = _search(model, scorer, graph_data, sequence_data, peptide_property, ni, si, cols, allowed, max_mut, beam,
                      rounds, maximize, kappa, max_graphs)
    return Design(*out, scorer.base)


def beam_search_pair(model, graph_pair, sequence_pair, property_pair, node_index: Tensor, seq_index: Tensor, *,
                     seq_columns, allowed: Optional[Tensor] = None, max_mutations: Optional[int] = None, beam: int = 8,
                     rounds: Optional[int] = None, maximize: bool = True, kappa: float = 0.0, eps=None, samples: int = 1,
                     max_graphs: int = 4096) -> Design:
    """``beam_search`` of the cancer item of ``model.forward_comparative(graph_pair, sequence_pair, property_pair)``
    against its fixed wild type, for the four comparative classes.  The sites index the cancer item.

    The wild type is encoded once, at batch B, and its encoded tensors are repeated for every pass.  ``eps`` = (eps_c,
    eps_w), each [K, B, latent], or one ``model.sample_eps`` call of [K*B, latent] per item, cancer first.  Without
    ``use_wt_for_downstream`` the wild type is neither run nor drawn for.  ``base`` equals ``predictive_pair`` on the same
    draws."""
    _check(model, samples, _Comparative, "beam_search_pair", _PAIR_CLASSES)
    gc = graph_pair[0]
    ni, si, cols, allowed, max_mut, rounds, kappa = _prepare(gc, sequence_pair[0], node_index, seq_index, seq_columns,
                                                             allowed, max_mutations, beam, rounds, kappa, max_graphs)
    with torch.no_grad():
        scorer = _scorer_pair(model, graph_pair, sequence_pair, property_pair, eps, samples)
        out = _search(model, scorer, gc, sequence_pair[0], property_pair[0], ni, si, cols, allowed, max_mut, beam, rounds,
                      maximize, kappa, max_graphs)
    return Design(*out, scorer.base)
