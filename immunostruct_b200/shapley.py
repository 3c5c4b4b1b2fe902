"""Shapley values of residues and residue groups: how much of the score each part of the structure carries, with credit
shared fairly between parts that back each other up.

Single-residue occlusion (``occlusion``) misses redundancy: when two pocket residues both make the contact that anchors
a peptide position, removing either one alone changes nothing and both score near zero.  The Shapley value of player i
is its marginal effect averaged over every removal order, so redundant players share the effect, and the values of a
sample add up exactly to ``v(full structure) - v(every player removed)``.

Players.  ``players`` int64 [ΣN] gives a graph-local player id per node row (-1: never removed), the ids of graph b
exactly 0 .. P_b - 1; a bool [ΣN] makes every selected row its own player, numbered in row order within its graph; by
default every row that is not already absent (all-zero with no edge, occlusion's rule) is a player.  P_b <= 256.
Removing a set of players is occlusion's removal of every row they hold: the 23 floats become 0.0 and every edge touching
such a row is dropped, the kept edges in base order.  Sequence, properties and draws are untouched.

Estimator.  T permutations per sample (T even), in antithetic pairs: permutation 2u orders the players by the key v0 of
Philox4x32-10 with counter (p, b, u, 2) and key ``seed``, ties to the smaller id, and 2u + 1 is its reverse.  The ranks
depend on (seed, b, u, p) alone, not on ``max_graphs``.  Coalition (t, j) removes the players of rank < j; j = 0 is the
base batch and j = P_b the one "every player removed" variant shared by all permutations, so a sample has
1 + T (P_b - 1) variants.  The value of a coalition is the mean over the K draws of the logit (``logit``) or of
sigmoid(logit) (``prob``).  The player at position j - 1 of permutation t gets Δ = v(t, j - 1) - v(t, j); d_u is the
mean of its two Δ of pair u, φ the mean of d_u over the T/2 pairs and ``se`` the standard error of that mean (NaN at
T = 2).  Every permutation telescopes, so ``gap = (v(base) - v(empty)) - Σ φ`` is at fp64 rounding.

Device flow.  Every argument check that needs no device data (the draws' shapes included) raises before anything
runs on the device.  One host read checks the players and sizes the call, the base batch is encoded and scored,
``is_shapley_plan`` (csrc/shapley.cu) draws and ranks every permutation and counts the kept edges of every variant, and
a second read sizes the passes.  A pass is a run of up to ``max_graphs`` variants: ``is_shapley_expand`` writes their
rows and compacted edges from the resident batch, the pass's topology is collated, the structure trunk runs, and
``is_head_mc_infer`` scores every draw on the sample's encoded sequence (the VAE encoder runs once per call).  The
logits of all variants stay on the device (V K 4 bytes) for ``is_shapley_reduce``, which writes φ, se and gap in fp64
in a fixed order; its flag and the expansion's are read once, after it.  An entry agrees with the fused eval forward of the host-built coalition batch to rounding, not bit for bit
(mutagenesis module docstring, DESIGN 4.4c).
"""
from __future__ import annotations

from dataclasses import dataclass
from typing import Optional

import torch

from . import functional as IF
from .comparative_models import _Comparative
from .coordnoise import _seed
from .graph import MAX_GRAPH_NODES
from .hybrid_models import _Hybrid
from .occlusion import _degrees, _selection
from .predictive import _CLASSES, _PAIR_CLASSES, Predictive, _check, _pair_items, _scorer, _scorer_pair
from .resident import pass_totals, score_gathered, variant_passes

Tensor = torch.Tensor


@dataclass
class ResidueShapley:
    """Shapley values of the players of every sample; sample b's players are entries offsets[b] .. offsets[b+1]-1, in id
    order."""
    players: Tensor       # [ΣN]  int64, graph-local player id of each node row, -1 for rows never removed
    offsets: Tensor       # [B+1] int64
    logit: Tensor         # [Q]   φ of v_logit (mean logit over the draws)
    prob: Tensor          # [Q]   φ of v_prob (mean sigmoid(logit) over the draws)
    logit_se: Tensor      # [Q]   standard error of the mean over the antithetic pairs; NaN for T = 2
    prob_se: Tensor       # [Q]
    empty: Predictive     # every player removed (base for a sample without players)
    gap_logit: Tensor     # [B]   (v(base) - v(empty)) - Σ φ, of v_logit
    gap_prob: Tensor      # [B]
    base: Predictive      # the unmodified batch on the same draws
    seed: int             # the seed of the permutation keys
    permutations: int     # T


def _checked(model, permutations, seed, max_graphs, eps, graphs):
    """Checks that need no device data, before any launch -> seed.  ``eps``: the draws of the items of ``graphs``
    (one item, or the pair's (eps_c, eps_w)), checked as ``predictive._scorer`` / ``_scorer_pair`` will read them."""
    if not isinstance(permutations, int) or isinstance(permutations, bool) or not 2 <= permutations <= 2 ** 16 \
            or permutations % 2:
        raise ValueError(f"permutations must be an even integer in [2, 2^16], got {permutations!r}")
    variant_passes(1, max_graphs)
    if len(graphs) == 2:
        items = [] if eps is None else list(zip(eps[:_pair_items(model, eps)], graphs))
    else:
        items = [] if eps is None else [(eps, graphs[0])]
    for e, g in items:
        if not isinstance(e, Tensor) or e.dim() != 3 or e.shape[0] < 1 or \
                tuple(e.shape[1:]) != (g.n_graphs, model.vae_latent_dim):
            raise ValueError(f"eps must have shape [K, {g.n_graphs}, {model.vae_latent_dim}], "
                             f"got {tuple(e.shape) if isinstance(e, Tensor) else type(e).__name__}")
    return _seed(seed)


def _players(graph, players):
    """(graph-local ids int64 [ΣN], P_b int64 [B], device bools (ids not exactly 0 .. P_b - 1, P_b > 256)) on the
    batch's device."""
    n, b, dev = graph.n_nodes, graph.n_graphs, graph.ndata["x"].device
    if players is None:
        players = _selection(graph, None, _degrees(graph)[2])
    elif not isinstance(players, Tensor) or players.dtype not in (torch.bool, torch.int64) or tuple(players.shape) != (n,):
        raise ValueError(f"players must be a bool or int64 tensor [ΣN={n}] over the batch's node rows")
    players = players.to(dev)
    batch, first = graph.batch.to(dev), graph.node_off[:-1].to(dev)
    if players.dtype == torch.bool:
        c = torch.cat([torch.zeros(1, dtype=torch.int64, device=dev), players.long().cumsum(0)])
        ids = torch.where(players, c[1:] - 1 - c[first][batch], -1)
        count = c[graph.node_off[1:].to(dev)] - c[first]
        return ids, count, torch.zeros((), dtype=torch.bool, device=dev), (count > MAX_GRAPH_NODES).any()
    ids = players
    live = ids >= 0
    count = torch.zeros(b, dtype=torch.int64, device=dev).scatter_reduce_(0, batch, ids + 1, "amax")
    held = torch.zeros(b * MAX_GRAPH_NODES + 1, dtype=torch.int64, device=dev)
    slot = torch.where(live & (ids < MAX_GRAPH_NODES), batch * MAX_GRAPH_NODES + ids, b * MAX_GRAPH_NODES)
    held.index_fill_(0, slot, 1)
    distinct = held[:-1].view(b, MAX_GRAPH_NODES).sum(1)
    too_many = (count > MAX_GRAPH_NODES).any()
    return ids, count, (ids < -1).any() | (~too_many & (distinct != count).any()), too_many


def _sizes(graph, players, permutations):
    """The checked players and the call's sizes, with its first host read -> (ids, P_b [B], variants per sample [B],
    Pmax, V, Q)."""
    ids, count, bad, too_many = _players(graph, players)
    nvar = torch.where(count > 0, 1 + permutations * (count - 1), 0)
    bad_ids, many, pmax, v, q = torch.stack([bad.long(), too_many.long(), count.max(), nvar.sum(), count.sum()]).tolist()
    if many:
        raise ValueError(f"a sample has more than {MAX_GRAPH_NODES} players")
    if bad_ids:
        raise ValueError("the player ids of each graph must be exactly 0 .. P_b - 1, each held by at least one row, "
                         "and -1 for rows that are never removed")
    if q == 0:
        raise ValueError("the players hold no residue: nothing to attribute")
    return ids, count, nvar, pmax, v, q


def _plan(graph, sizes, permutations, seed, max_graphs):
    """The plan launch and the pass tables, with the call's second host read -> dict of device tables and pass sizes."""
    ids, count, nvar, pmax, v, q = sizes
    t = permutations
    dev = ids.device
    zero = torch.zeros(1, dtype=torch.int64, device=dev)
    voff, poff = torch.cat([zero, nvar.cumsum(0)]), torch.cat([zero, count.cumsum(0)])
    b = count.shape[0]
    smp = torch.repeat_interleave(torch.arange(b, device=dev), nvar, output_size=v)
    local = torch.arange(v, device=dev) - voff[smp]
    p = count[smp]
    step = (local - 1).clamp_min(0)
    width = (p - 1).clamp_min(1)
    row = smp * t + torch.where(local == 0, 0, step // width)               # the empty variant reads any row: all removed
    thr = torch.where(local == 0, p, step % width + 1)
    ranks = torch.empty(b, t, pmax, dtype=torch.int32, device=dev)
    kept = torch.zeros(v, dtype=torch.int64, device=dev)                      # sizes the passes even if the plan fails
    flag = torch.zeros(1, dtype=torch.int32, device=dev)
    ids32 = ids.to(torch.int32)
    IF._C.shapley_plan(graph.node_off, graph.edge_off, graph._src_local.contiguous(), graph._dst_local.contiguous(),
                       ids32, poff, voff, seed, ranks, kept, flag)
    nv = graph.batch_num_nodes().to(dev)[smp]
    passes = variant_passes(v, max_graphs)
    ncs, ecs, node_tot, edge_tot = pass_totals(nv, kept, v, len(passes), max_graphs)
    totals = torch.cat([node_tot, edge_tot]).tolist()
    return dict(ids=ids, ids32=ids32, count=count, voff=voff, poff=poff, smp=smp, row=row, thr=thr, ranks=ranks,
                kept=kept, nv=nv, ncs=ncs, ecs=ecs, passes=passes, node_tot=totals[:len(passes)],
                edge_tot=totals[len(passes):], flag=flag, q=q)


def _shapley(model, scorer, graph, plan, seed, permutations):
    """Every chain variant in gathered passes, then the reduction -> ResidueShapley."""
    mu, logvar, z_vae, e = scorer.item[1:]
    smp, row, thr, ranks, flag = plan["smp"], plan["row"], plan["thr"], plan["ranks"], plan["flag"]

    def expand(j, r, inputs, outputs):
        IF._C.shapley_expand(*inputs, plan["ids32"], ranks, smp[j:j + r], row[j:j + r], thr[j:j + r], *outputs, flag)

    def pass_item(g, sp, _):
        return model.structure_embedding(g, project=False)[0].contiguous(), mu[sp], logvar[sp], z_vae[sp], e[:, sp]

    logits, mean, std = score_gathered(scorer, graph, smp, plan["nv"], plan["kept"], plan["ncs"], plan["ecs"],
                                       plan["passes"], plan["node_tot"], plan["edge_tot"], expand, pass_item)
    base, q, b = scorer.base, plan["q"], plan["count"].shape[0]
    f32 = dict(dtype=torch.float32, device=logits.device)
    phi, se, gap = torch.empty(2, q, **f32), torch.empty(2, q, **f32), torch.empty(2, b, **f32)
    IF._C.shapley_reduce(logits, base.logits.contiguous(), ranks, plan["poff"], plan["voff"], phi, se, gap, flag)
    if flag.item():
        raise RuntimeError("a Shapley kernel rejected its tables: player ids, ranks or offsets disagree with the batch")
    has = plan["count"] > 0
    first = plan["voff"][:-1].clamp_max(logits.shape[0] - 1)
    empty = Predictive(torch.where(has[:, None], logits[first], base.logits), torch.where(has, mean[first], base.prob_mean),
                       torch.where(has, std[first], base.prob_std))
    return ResidueShapley(plan["ids"], plan["poff"], phi[0], phi[1], se[0], se[1], empty, gap[0], gap[1], base, seed,
                          permutations)


def residue_shapley(model, graph, seq, prop, *, players: Optional[Tensor] = None, permutations: int = 32,
                    seed: Optional[int] = None, eps: Optional[Tensor] = None, samples: int = 1,
                    max_graphs: int = 4096) -> ResidueShapley:
    """Shapley values of the players of every sample for ``model(graph, seq, prop)[3]`` (the logit), removing players
    as occlusion removes a residue (zeroed rows, every edge touching them dropped).

    ``players``: int64 [ΣN] graph-local player ids (-1: never removed; the ids of graph b exactly 0 .. P_b - 1), or bool
    [ΣN] (each selected row its own player, in row order), by default every row that is not already absent; P_b <= 256,
    a sample may have none.  ``permutations`` = T, even, in [2, 2^16], in antithetic pairs keyed on (``seed``, sample,
    pair, player); ``seed`` in [0, 2^64), by default one 63-bit integer from torch's default CPU generator (returned).
    ``eps`` [K, B, latent] gives the draws, or one ``model.sample_eps`` call of [K*B, latent] (K = ``samples``) makes
    them; every coalition of a sample uses its draws.  A sample has 1 + T (P_b - 1) variants, run in passes of at most
    ``max_graphs``; their logits stay on the device until the reduction (V K 4 bytes).  Follows ``model.forward`` for
    the eight classes ``predictive`` supports; the model must be in eval mode; no_grad, and every ``.grad`` is left
    untouched."""
    _check(model, samples, (_Hybrid, _Comparative), "residue_shapley", _CLASSES)
    seed = _checked(model, permutations, seed, max_graphs, eps, [graph])
    with torch.no_grad():
        sizes = _sizes(graph, players, permutations)
        scorer = _scorer(model, graph, seq, prop, eps, samples)
        plan = _plan(graph, sizes, permutations, seed, max_graphs)
        return _shapley(model, scorer, graph, plan, seed, permutations)


def residue_shapley_pair(model, graph_pair, seq_pair, prop_pair, *, players: Optional[Tensor] = None,
                         permutations: int = 32, seed: Optional[int] = None, eps=None, samples: int = 1,
                         max_graphs: int = 4096) -> ResidueShapley:
    """``residue_shapley`` of the cancer item of ``model.forward_comparative(graph_pair, seq_pair, prop_pair)`` against
    its fixed wild type, for the four comparative classes; ``players`` indexes the cancer graph's rows.

    The wild type is encoded once, at batch B; each pass gathers its encoded tensors and its draws by sample.  ``eps`` =
    (eps_c, eps_w), each [K, B, latent], or one ``model.sample_eps`` call of [K*B, latent] per item, cancer first.
    Without ``use_wt_for_downstream`` the wild type is neither run nor drawn for.  ``base`` equals ``predictive_pair`` on
    the same draws."""
    _check(model, samples, _Comparative, "residue_shapley_pair", _PAIR_CLASSES)
    seed = _checked(model, permutations, seed, max_graphs, eps, graph_pair)
    with torch.no_grad():
        sizes = _sizes(graph_pair[0], players, permutations)
        scorer = _scorer_pair(model, graph_pair, seq_pair, prop_pair, eps, samples)
        plan = _plan(graph_pair[0], sizes, permutations, seed, max_graphs)
        return _shapley(model, scorer, graph_pair[0], plan, seed, permutations)
