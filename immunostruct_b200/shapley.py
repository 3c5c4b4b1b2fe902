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

Contacts.  ``contact_shapley`` plays the same game with sets of edges as the players, answering which contacts carry
the call where residue removal cannot separate a residue's contacts.  Removing players drops their edges and nothing
else: every row stays, and the kept edges keep their attributes and base order, so a coalition is exactly the graph a
boolean edge mask builds.  Players are explicit edge groups (int64 [ΣE]) or every contact with a selected endpoint (bool
[ΣN], numbered as ``occlusion.occlude_contacts`` numbers contacts).  The keys use counter word 3 = 3 instead of 2, so a
contact game's permutations are independent of a residue game's on the same seed.  ``is_shapley_edge_plan`` and
``is_shapley_edge_expand`` replace the plan and the expansion; variants, passes and the reduction are shared.
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
from .occlusion import _contacts, _degrees, _selection
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


@dataclass
class ContactShapley:
    """Shapley values of the contact players of every sample; sample b's players are entries offsets[b] ..
    offsets[b+1]-1, in id order."""
    edge_player: Tensor   # [ΣE]  int64, graph-local player id of each edge, -1 for edges never removed
    offsets: Tensor       # [B+1] int64
    u: Tensor             # [Q]   int64, graph-local endpoints of a bool-selected contact, u < v; -1 for explicit groups
    v: Tensor             # [Q]
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


def _counted(ids, owner, b):
    """P_b of explicit graph-local ids [M] whose entries belong to graphs ``owner`` [M] -> (P_b int64 [B], device bools
    (ids not exactly 0 .. P_b - 1, P_b > 256))."""
    dev = ids.device
    live = ids >= 0
    count = torch.zeros(b, dtype=torch.int64, device=dev).scatter_reduce_(0, owner, ids + 1, "amax")
    held = torch.zeros(b * MAX_GRAPH_NODES + 1, dtype=torch.int64, device=dev)
    slot = torch.where(live & (ids < MAX_GRAPH_NODES), owner * MAX_GRAPH_NODES + ids, b * MAX_GRAPH_NODES)
    held.index_fill_(0, slot, 1)
    distinct = held[:-1].view(b, MAX_GRAPH_NODES).sum(1)
    too_many = (count > MAX_GRAPH_NODES).any()
    return count, (ids < -1).any() | (~too_many & (distinct != count).any()), too_many


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
    return (players, *_counted(players, batch, b))


def _edge_players(graph, players):
    """(graph-local ids int64 [ΣE], P_b int64 [B], device bools (ids not exactly 0 .. P_b - 1, P_b > 256), graph-local
    endpoints (u, v) [ΣE] of player q of sample b at entry offsets[b] + q, or None for explicit ids) on the batch's
    device."""
    n, e, b, dev = graph.n_nodes, graph.n_edges, graph.n_graphs, graph.ndata["x"].device
    if not isinstance(players, Tensor) or not ((players.dtype == torch.bool and tuple(players.shape) == (n,)) or
                                               (players.dtype == torch.int64 and tuple(players.shape) == (e,))):
        raise ValueError(f"players must be an int64 tensor [ΣE={e}] of graph-local player ids over the batch's edges, "
                         f"or a bool tensor [ΣN={n}] selecting node rows")
    players = players.to(dev)
    owner = torch.repeat_interleave(torch.arange(b, device=dev), graph.batch_num_edges().to(dev), output_size=e)
    if players.dtype == torch.int64:
        return (players, *_counted(players, owner, b), None)
    no = torch.zeros((), dtype=torch.bool, device=dev)
    if e == 0:
        return torch.zeros(0, dtype=torch.int64, device=dev), torch.zeros(b, dtype=torch.int64, device=dev), no, no, None
    # every contact with a selected endpoint is its own player, numbered as occlusion numbers contacts
    gs, gd = graph.edge_index
    edge_contact, ug, vg, _, c = _contacts(gs, gd, players, n)
    smp = graph.batch[ug]
    count = torch.zeros(b, dtype=torch.int64, device=dev).scatter_add_(0, smp, (torch.arange(e, device=dev) < c).long())
    first = torch.cat([torch.zeros(1, dtype=torch.int64, device=dev), count.cumsum(0)[:-1]])
    ids = torch.where(edge_contact >= 0, edge_contact - first[owner], -1)
    off = graph.node_off[smp]
    return ids, count, no, (count > MAX_GRAPH_NODES).any(), (ug - off, vg - off)


def _sized(checked, permutations, holder, too_many_message):
    """The checked players and the call's sizes, with its first host read -> (ids, P_b [B], variants per sample [B],
    Pmax, V, Q).  ``holder`` names what holds a player; ``too_many_message(Pmax)`` is the error for more than 256."""
    ids, count, bad, too_many = checked
    nvar = torch.where(count > 0, 1 + permutations * (count - 1), 0)
    bad_ids, many, pmax, v, q = torch.stack([bad.long(), too_many.long(), count.max(), nvar.sum(), count.sum()]).tolist()
    if many:
        raise ValueError(too_many_message(pmax))
    if bad_ids:
        raise ValueError(f"the player ids of each graph must be exactly 0 .. P_b - 1, each held by at least one "
                         f"{holder}, and -1 for {holder}s that are never removed")
    if q == 0:
        raise ValueError(f"the players hold no {'residue' if holder == 'row' else holder}: nothing to attribute")
    return ids, count, nvar, pmax, v, q


def _sizes(graph, players, permutations):
    """Residue players: ``_sized`` of the node-row ids."""
    return _sized(_players(graph, players), permutations, "row",
                  lambda pmax: f"a sample has more than {MAX_GRAPH_NODES} players")


def _edge_sizes(graph, players, permutations):
    """Contact players: (``_sized`` of the edge ids, graph-local endpoints (u, v) [Q] of the players, -1 for explicit
    groups)."""
    *checked, uv = _edge_players(graph, players)
    sizes = _sized(checked, permutations, "edge",
                   lambda pmax: f"a sample has {pmax} players, more than {MAX_GRAPH_NODES}: group its edges into "
                                f"at most {MAX_GRAPH_NODES} players")
    q = sizes[-1]
    if uv is None:
        uv = (torch.full((q,), -1, dtype=torch.int64, device=sizes[0].device),) * 2
    return sizes, tuple(x[:q].contiguous() for x in uv)


def _row_plan(graph, ids32, poff, voff, seed, ranks, kept, flag):
    IF._C.shapley_plan(graph.node_off, graph.edge_off, graph._src_local.contiguous(), graph._dst_local.contiguous(),
                       ids32, poff, voff, seed, ranks, kept, flag)


def _edge_plan(graph, ids32, poff, voff, seed, ranks, kept, flag):
    IF._C.shapley_edge_plan(graph.edge_off, ids32, poff, voff, seed, ranks, kept, flag)


def _plan(graph, sizes, permutations, seed, max_graphs, launch=_row_plan):
    """The plan launch (``launch``: ``_row_plan`` or ``_edge_plan``) and the pass tables, with the call's second host
    read -> dict of device tables and pass sizes."""
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
    launch(graph, ids32, poff, voff, seed, ranks, kept, flag)
    nv = graph.batch_num_nodes().to(dev)[smp]
    passes = variant_passes(v, max_graphs)
    ncs, ecs, node_tot, edge_tot = pass_totals(nv, kept, v, len(passes), max_graphs)
    totals = torch.cat([node_tot, edge_tot]).tolist()
    return dict(ids=ids, ids32=ids32, count=count, voff=voff, poff=poff, smp=smp, row=row, thr=thr, ranks=ranks,
                kept=kept, nv=nv, ncs=ncs, ecs=ecs, passes=passes, node_tot=totals[:len(passes)],
                edge_tot=totals[len(passes):], flag=flag, q=q)


def _shapley(model, scorer, graph, plan, expand):
    """Every chain variant in gathered passes, each expanded by ``expand`` (``_C.shapley_expand`` or
    ``_C.shapley_edge_expand``), then the reduction -> (φ [2, Q], se [2, Q], gap [2, B], empty)."""
    mu, logvar, z_vae, e = scorer.item[1:]
    smp, row, thr, ranks, flag = plan["smp"], plan["row"], plan["thr"], plan["ranks"], plan["flag"]

    def expand_pass(j, r, inputs, outputs):
        expand(*inputs, plan["ids32"], ranks, smp[j:j + r], row[j:j + r], thr[j:j + r], *outputs, flag)

    def pass_item(g, sp, _):
        return model.structure_embedding(g, project=False)[0].contiguous(), mu[sp], logvar[sp], z_vae[sp], e[:, sp]

    logits, mean, std = score_gathered(scorer, graph, smp, plan["nv"], plan["kept"], plan["ncs"], plan["ecs"],
                                       plan["passes"], plan["node_tot"], plan["edge_tot"], expand_pass, pass_item)
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
    return phi, se, gap, empty


def _residue_result(scorer, plan, out, seed, permutations):
    phi, se, gap, empty = out
    return ResidueShapley(plan["ids"], plan["poff"], phi[0], phi[1], se[0], se[1], empty, gap[0], gap[1], scorer.base,
                          seed, permutations)


def _contact_result(scorer, plan, uv, out, seed, permutations):
    phi, se, gap, empty = out
    return ContactShapley(plan["ids"], plan["poff"], *uv, phi[0], phi[1], se[0], se[1], empty, gap[0], gap[1],
                          scorer.base, seed, permutations)


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
        return _residue_result(scorer, plan, _shapley(model, scorer, graph, plan, IF._C.shapley_expand), seed,
                               permutations)


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
        return _residue_result(scorer, plan, _shapley(model, scorer, graph_pair[0], plan, IF._C.shapley_expand), seed,
                               permutations)


def contact_shapley(model, graph, seq, prop, players: Tensor, *, permutations: int = 32, seed: Optional[int] = None,
                    eps: Optional[Tensor] = None, samples: int = 1, max_graphs: int = 4096) -> ContactShapley:
    """Shapley values of contacts, or of contact groups, of every sample for ``model(graph, seq, prop)[3]`` (the
    logit).  A player is a set of edges of one graph; removing players drops their edges and nothing else (rows, the
    attributes and base order of the kept edges, sequence, properties and draws are unchanged).

    ``players``: int64 [ΣE] aligned with ``graph.edata['edge_attr']``, the graph-local player id of each edge (-1: never
    removed; the ids of graph b exactly 0 .. P_b - 1, each held by at least one edge; any edge may be grouped, a
    self-loop included), or bool [ΣN] selecting node rows: every contact (an unordered pair u != v joined by at least one
    edge, both directions and multi-edges included) with a selected endpoint is its own player, numbered in (u, v) order
    within its graph as ``occlusion.occlude_contacts`` numbers them; a self-loop is never a player.  P_b <= 256 (group
    edges to cover more); a sample may have none.  Permutations, seed, draws, passes, classes, eval mode, no_grad and
    ``.grad`` as in ``residue_shapley``; the keys are drawn on their own Philox stream, so a contact game's permutations
    are independent of a residue game's on the same seed."""
    _check(model, samples, (_Hybrid, _Comparative), "contact_shapley", _CLASSES)
    seed = _checked(model, permutations, seed, max_graphs, eps, [graph])
    with torch.no_grad():
        sizes, uv = _edge_sizes(graph, players, permutations)
        scorer = _scorer(model, graph, seq, prop, eps, samples)
        plan = _plan(graph, sizes, permutations, seed, max_graphs, _edge_plan)
        return _contact_result(scorer, plan, uv, _shapley(model, scorer, graph, plan, IF._C.shapley_edge_expand), seed,
                               permutations)


def contact_shapley_pair(model, graph_pair, seq_pair, prop_pair, players: Tensor, *, permutations: int = 32,
                         seed: Optional[int] = None, eps=None, samples: int = 1,
                         max_graphs: int = 4096) -> ContactShapley:
    """``contact_shapley`` of the cancer item of ``model.forward_comparative(graph_pair, seq_pair, prop_pair)`` against
    its fixed wild type, for the four comparative classes; ``players`` indexes the cancer graph's edges (or rows).  The
    wild type and the draws as in ``residue_shapley_pair``."""
    _check(model, samples, _Comparative, "contact_shapley_pair", _PAIR_CLASSES)
    seed = _checked(model, permutations, seed, max_graphs, eps, graph_pair)
    with torch.no_grad():
        sizes, uv = _edge_sizes(graph_pair[0], players, permutations)
        scorer = _scorer_pair(model, graph_pair, seq_pair, prop_pair, eps, samples)
        plan = _plan(graph_pair[0], sizes, permutations, seed, max_graphs, _edge_plan)
        return _contact_result(scorer, plan, uv,
                               _shapley(model, scorer, graph_pair[0], plan, IF._C.shapley_edge_expand), seed,
                               permutations)
