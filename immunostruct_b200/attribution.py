"""Integrated-gradients attribution (Sundararajan, Taly & Yan 2017) of a model's logit to its inputs: which residues,
which contacts (edges), which sequence positions and which peptide properties drove an immunogenicity call.

    IG_i(x) = (x_i - x'_i) * mean over k of  dF/dx_i (x' + a_k (x - x')),   a_k = (k + 1/2) / steps

with the all-zero baseline x' (an all-zero residue row is how the reference's ``pad_graph`` writes an absent residue).
Coordinates are not interpolated: with every residue on one point, ``diff / (sqrt(r) + 1e-30)`` has no usable derivative;
the plain input gradient (``x23.requires_grad_()`` and backward) is the coordinate answer.

The path points run through the model's own training kernels (the EGNN stack's input gradients, csrc/egnn_node_bwd_tc.cu,
csrc/egnn_edge_attr.cu): the batch is replicated on the device, several alpha values per pass, at most ``max_graphs``
graphs per pass.
"""
from __future__ import annotations

from dataclasses import dataclass
from typing import Optional

import torch

from . import functional as IF
from .graph import GraphBatch

Tensor = torch.Tensor


@dataclass
class Attribution:
    """Integrated gradients of the logit (index 3 of the forward tuple) for one batch.  An attribution is None where the
    model does not consume that input.  ``completeness_gap`` = logit - baseline_logit - (sum of the sample's
    attributions): the path-integral discretisation error, which shrinks as ``steps`` grows."""
    residue_features: Optional[Tensor]     # [sum N, 20]
    edge_attr: Optional[Tensor]            # [sum E]
    sequence: Optional[Tensor]             # shape of sequence_data ([B, L, 21])
    peptide_property: Optional[Tensor]     # [B, 2]
    logit: Tensor                          # [B]
    baseline_logit: Tensor                 # [B]
    completeness_gap: Tensor               # [B]


def integrated_gradients(model, graph_data: GraphBatch, sequence_data: Optional[Tensor], peptide_property: Optional[Tensor],
                         *, steps: int = 32, eps: Optional[Tensor] = None, max_graphs: int = 4096) -> Attribution:
    """Integrated-gradients attribution of ``model(graph_data, sequence_data, peptide_property)[3]`` (the logit) to the 20
    residue-feature columns of ``graph_data.ndata['x']``, to ``edge_attr``, to ``sequence_data`` and to
    ``peptide_property``, against the all-zero baseline, over ``steps`` midpoint alpha values.

    ``model`` must be in eval mode (dropout would change the function along the path).  The reparameterisation noise is
    drawn once per sample (``eps`` [B, latent], or one ``model.sample_eps`` call) and reused at every alpha.  Runs under
    ``torch.enable_grad()`` (so it works inside a ``no_grad`` scan) and leaves every parameter's ``.grad`` untouched."""
    if model.training:
        raise RuntimeError("integrated_gradients needs model.eval(): dropout would change the function along the path")
    if steps < 1:
        raise ValueError("steps must be >= 1")
    b = graph_data.n_graphs
    if b > max_graphs:
        raise ValueError(f"the batch has {b} graphs, more than max_graphs={max_graphs}")
    x = graph_data.ndata["x"]
    dev, n = x.device, graph_data.n_nodes
    per_pass = max(1, min(steps, max_graphs // b))
    has_eps = hasattr(model, "sample_eps") and hasattr(model, "vae_latent_dim")
    injected = model.__dict__.get("sample_eps")
    graphs = {}

    def run(alphas, want_grad):
        """Logits [len(alphas), B] at the given path points and, with ``want_grad``, the gradients of their sum with respect
        to (x23, edge_attr, sequence, property) summed over the points (None where unused)."""
        r = len(alphas)
        if r not in graphs:
            g = graph_data.replicate(r)
            graphs[r] = (g, g.ndata["x"])
        g, x_rep = graphs[r]
        a = torch.tensor(alphas, dtype=x.dtype, device=dev)

        def scaled(t, rows):                    # r stacked copies of t, copy k scaled by alphas[k]
            if t is None:
                return None
            ones = [1] * (t.dim() - 1)
            return t.detach().repeat(r, *ones) * a.repeat_interleave(rows).reshape(-1, *ones)

        xp = x_rep.clone()
        xp[:, :20] *= a.repeat_interleave(n).unsqueeze(1)
        ea = graph_data.edata["edge_attr"]
        eap, sp, pp = scaled(ea, ea.shape[0]), scaled(sequence_data, b), scaled(peptide_property, b)
        leaves = [t for t in (xp, eap, sp, pp) if t is not None]
        if want_grad:
            for t in leaves:
                t.requires_grad_(True)
        g.ndata["x"], g.edata["edge_attr"] = xp, eap
        out = model(g, sp, pp)[3].reshape(-1)
        if out.numel() != r * b:
            raise ValueError(f"the model's output 3 has {out.numel() // r} values per pass copy, expected one logit per graph")
        logits = out.detach().reshape(r, b)
        if not want_grad:
            return logits, None
        got = iter(torch.autograd.grad(out.sum(), leaves, allow_unused=True))
        grads = [None if t is None else next(got) for t in (xp, eap, sp, pp)]
        sums = [None if gr is None else gr.reshape(r, -1, *gr.shape[1:]).sum(0) for gr in grads]
        return logits, sums

    try:
        with torch.enable_grad():
            if has_eps:
                if eps is None:
                    eps = model.sample_eps(torch.empty(b, model.vae_latent_dim, dtype=x.dtype, device=dev))
                eps = eps.detach().to(dev, x.dtype)
                model.sample_eps = lambda like: eps.repeat(like.shape[0] // b, 1)
            if per_pass >= 2:
                logit, baseline_logit = run([1.0, 0.0], False)[0]
            else:
                logit, baseline_logit = run([1.0], False)[0][0], run([0.0], False)[0][0]
            alphas = [(k + 0.5) / steps for k in range(steps)]
            total = None
            for k0 in range(0, steps, per_pass):
                _, sums = run(alphas[k0:k0 + per_pass], True)
                total = sums if total is None else [None if t is None else t + s for t, s in zip(total, sums)]
    finally:
        if has_eps:
            if injected is None:
                model.__dict__.pop("sample_eps", None)
            else:
                model.sample_eps = injected

    gx, gea, gs, gp = (None if t is None else t / steps for t in total)
    with torch.no_grad():
        a_res = None if gx is None else x[:, :20] * gx[:, :20]
        a_edge = None if gea is None else (graph_data.edata["edge_attr"] * gea).reshape(-1)
        a_seq = None if gs is None else sequence_data * gs
        a_prop = None if gp is None else peptide_property * gp
        total_attr = torch.zeros(b, dtype=logit.dtype, device=dev)
        if a_res is not None:
            total_attr += IF.segment_pool(graph_data, a_res.contiguous(), "sum").sum(1)
        if a_edge is not None:
            total_attr += IF.segment_pool(graph_data.edge_off, a_edge.unsqueeze(1).contiguous(), "sum")[:, 0]
        if a_seq is not None:
            total_attr += a_seq.reshape(b, -1).sum(1)
        if a_prop is not None:
            total_attr += a_prop.reshape(b, -1).sum(1)
        gap = logit - baseline_logit - total_attr
    return Attribution(a_res, a_edge, a_seq, a_prop, logit, baseline_logit, gap)
