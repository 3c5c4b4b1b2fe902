"""Predictive mean and spread of the immunogenicity score over the VAE's reparameterisation draw.

The reference samples ``z = mu + eps * exp(0.5 logvar)`` in eval mode too (``reparameterize``, hybrid_models.py:301-304),
so one forward returns one random draw of the score.  ``predictive`` returns K draws of the logit together with the mean
and the population standard deviation of sigmoid(logit) over them.

Only the 32 latent tokens of the fused head depend on the draw.  The structure trunk (EGNN stack, attention, pooling)
and the VAE encoder run once per item; the head runs once for all K draws (``is_head_mc_infer``, csrc/head.cu), with
the arithmetic of the fused eval forward: draw k of a non-SSL hybrid model is bit-identical to ``model(...)[3]`` run on
``eps[k]``.  The VAE decoder does not enter the score: ``vae_fc4`` and the reconstruction are not computed (the fc3
output of the shared ``vae_mid_infer`` kernel is discarded).
"""
from __future__ import annotations

from dataclasses import dataclass, field
from typing import Optional

import torch

from . import functional as IF
from .comparative_models import _Comparative
from .hybrid_models import _Hybrid
from .trunk import _tc_linear

Tensor = torch.Tensor

_PAIR_CLASSES = "HybridModel_Comparative, HybridModel_Comparative_SSL, HybridModelv2_Comparative, HybridModelv2_Comparative_SSL"
_CLASSES = "HybridModel, HybridModelv2, HybridModel_SSL, HybridModelv2_SSL, " + _PAIR_CLASSES


@dataclass
class Predictive:
    """K draws of the logit of each sample and the statistics of the probability sigmoid(logit) over them
    (procedures/infer.py:22 applies the sigmoid)."""
    logits: Tensor        # [B, K]
    prob_mean: Tensor     # [B]  mean of sigmoid(logit) over the draws
    prob_std: Tensor      # [B]  population standard deviation of sigmoid(logit) over the draws


def _head_params(model):
    """Weights of the fused head, after checking that the model has one: (Wc, bc, coef, n_head, W1, b1, W2, b2)."""
    if model.gat_hidden_channels != 64 or model.mlp_features != 32:
        raise NotImplementedError("the fused head needs gat_hidden_channels = 64 and mlp_features = 32")
    fus = model.combined_attention if model._fusion_dim else None
    if fus is not None and fus.n_head > 8:
        raise NotImplementedError("the fused head supports at most 8 fusion-attention heads")
    cls1 = model.classifier[1]
    if cls1.in_features > 256:
        raise NotImplementedError(f"the fused head supports at most 256 fused tokens, the classifier takes {cls1.in_features}")
    out = model.classifier_head if model._ssl else model.classifier[4]
    wc = model.self_attention.out_projection
    d = lambda t: None if t is None else t.detach()
    return (d(None if wc is None else wc.weight), d(None if wc is None else wc.bias),
            None if fus is None else d(fus.fusion_coefficients()), 0 if fus is None else fus.n_head,
            d(cls1.weight), d(cls1.bias), d(out.weight), d(out.bias))


def _encode(model, graph_data, sequence_data, peptide_property):
    """The draw-independent part of one item: (pooled [B,64] before w_concat, mu, logvar, z_vae [B,LD+PD]).  z_vae's
    latent columns are mu (zero noise); only its property columns are read by the head."""
    pooled = model.structure_embedding(graph_data, project=False)[0].contiguous()
    h1 = _tc_linear(model.vae_fc1, sequence_data.reshape(-1, model.vae_input_dim), relu=True)
    zero = torch.zeros(h1.shape[0], model.vae_latent_dim, dtype=h1.dtype, device=h1.device)
    mu, logvar, z_vae, _ = model.vae_mid_eval(h1, model.property_embedding, peptide_property, zero)
    return pooled, mu, logvar, z_vae


def _draws(model, eps, k, b, like):
    """eps [K,B,LD] as given (checked) or drawn by one ``model.sample_eps`` call of [K*B, LD]."""
    ld = model.vae_latent_dim
    if eps is None:
        return model.sample_eps(torch.empty(k * b, ld, dtype=like.dtype, device=like.device)).reshape(k, b, ld).contiguous()
    if eps.dim() != 3 or eps.shape[0] < 1 or tuple(eps.shape[1:]) != (b, ld):
        raise ValueError(f"eps must have shape [K, {b}, {ld}], got {tuple(eps.shape)}")
    return eps.detach().to(like.device, like.dtype).contiguous()


def _check(model, samples, kinds, what, names):
    if not isinstance(model, kinds):
        raise NotImplementedError(f"{what} supports {names}; {type(model).__name__} is not one of them")
    if samples < 1:
        raise ValueError("samples must be >= 1")
    if model.training:
        raise RuntimeError(f"{what} needs model.eval(): dropout would change the function between draws and variants")


def _pair_items(model, eps):
    """Number of items the pair head reads (2 with ``use_wt_for_downstream``, else 1), after checking eps = (eps_c, eps_w)."""
    if eps is not None and (not isinstance(eps, (tuple, list)) or len(eps) != 2):
        raise ValueError("eps must be a pair (eps_c, eps_w)")
    n = 2 if model.use_wt_for_downstream else 1
    if eps is not None and any(e is None for e in eps[:n]):
        raise ValueError("eps needs eps_c, and eps_w when use_wt_for_downstream is set")
    if eps is not None and n == 2 and eps[0].shape[:1] != eps[1].shape[:1]:
        raise ValueError("eps_c and eps_w must hold the same number of draws")
    return n


def _repeat(t, r):
    """A tensor of an item or of the batch, [B, ...] or draws-first [K, B, latent], repeated for r copies of the batch."""
    return t.repeat(1, r, 1) if t.dim() == 3 else t.repeat(r, 1)


@dataclass
class _Scorer:
    """The base of a batch on the device and the head that scores its variants.  ``item`` = (pooled, mu, logvar, z_vae,
    eps) of the scored item at batch B; ``wt`` the fixed wild-type item at batch B, or None; ``repeat``: the single form
    of a pair-wide head, which reads its one item twice; ``params`` the head's weights; ``base`` the item's scores."""
    item: tuple
    wt: Optional[tuple]
    repeat: bool
    params: tuple
    base: Predictive
    _wt_r: dict = field(default_factory=dict, repr=False)

    def score(self, item, *, r=None, sample=None, wt=None):
        """(logits, prob_mean, prob_std) of a pass item.  The head reads it against ``wt`` when given, else against the
        fixed wild type repeated for a pass of r copies of the batch (built once per r) or gathered by ``sample``."""
        if self.repeat:
            items = [item, item]
        elif wt is not None:
            items = [item, wt]
        elif self.wt is None:
            items = [item]
        elif sample is not None:
            items = [item, tuple(t[:, sample] if t.dim() == 3 else t[sample] for t in self.wt)]
        else:
            if r not in self._wt_r:
                self._wt_r[r] = tuple(_repeat(t, r) for t in self.wt)
            items = [item, self._wt_r[r]]
        return IF._C.head_mc_infer(items, *self.params)


def _scorer(model, graph_data, sequence_data, peptide_property, eps, samples) -> _Scorer:
    """The scorer of ``model.forward``'s one item (``predictive``): drawn, then encoded and scored.  Under no_grad."""
    params = _head_params(model)
    e = _draws(model, eps, samples, graph_data.n_graphs, graph_data.ndata["x"])
    item = _encode(model, graph_data, sequence_data, peptide_property) + (e,)
    repeat = isinstance(model, _Comparative) and model.use_wt_for_downstream
    base = Predictive(*IF._C.head_mc_infer([item, item] if repeat else [item], *params))
    return _Scorer(item, None, repeat, params, base)


def _scorer_pair(model, graph_pair, sequence_pair, property_pair, eps, samples) -> _Scorer:
    """The scorer of ``model.forward_comparative``'s cancer item against its wild type (``predictive_pair``): both items
    drawn, cancer first, then encoded and scored; the wild type is neither drawn nor run without
    ``use_wt_for_downstream``.  Under no_grad."""
    n = _pair_items(model, eps)
    params = _head_params(model)
    k = samples if eps is None else eps[0].shape[0]
    draws = [_draws(model, None if eps is None else eps[i], k, graph_pair[i].n_graphs, graph_pair[i].ndata["x"])
             for i in range(n)]
    items = [_encode(model, graph_pair[i], sequence_pair[i], property_pair[i]) + (draws[i],) for i in range(n)]
    base = Predictive(*IF._C.head_mc_infer(items, *params))
    return _Scorer(items[0], items[1] if n == 2 else None, False, params, base)


def predictive(model, graph_data, sequence_data, peptide_property, *, samples: int = 32,
               eps: Optional[Tensor] = None) -> Predictive:
    """K draws of ``model(graph_data, sequence_data, peptide_property)[3]`` (the logit), with K = ``samples`` or
    ``eps.shape[0]``.  Follows ``model.forward``: for the comparative classes that is the single-graph forward, which
    repeats one item's features (and its one draw) across the pair-wide classifier when ``use_wt_for_downstream``.

    ``eps`` [K, B, latent] gives the standard-normal draws (then ``samples`` is not used).  By default they come from one
    ``model.sample_eps`` call of [K*B, latent] (an injected sampler is honoured).  These are not the random numbers that
    K sequential forwards would consume, only numbers of the same distribution.

    The model must be in eval mode.  Runs under ``torch.no_grad()`` and leaves every ``.grad`` untouched; the structure
    trunk and the VAE encoder run once, the head runs once for all draws."""
    _check(model, samples, (_Hybrid, _Comparative), "predictive", _CLASSES)
    with torch.no_grad():
        return _scorer(model, graph_data, sequence_data, peptide_property, eps, samples).base


def predictive_pair(model, graph_pair, sequence_pair, property_pair, *, samples: int = 32,
                    eps=None) -> Predictive:
    """K draws of the logit of ``model.forward_comparative(graph_pair, sequence_pair, property_pair)`` for the four
    comparative classes: the cancer item and the wild-type item each take their own draw.

    ``eps`` = (eps_c, eps_w), each [K, B, latent].  By default they come from ``model.sample_eps``, one call of
    [K*B, latent] per item, cancer first.  Without ``use_wt_for_downstream`` the logit depends on the cancer item only:
    the wild-type item is not run, no wild-type noise is drawn, and eps_w may be None.  The draws are not the random
    numbers that K sequential forwards would consume, only numbers of the same distribution.  Eval mode, no_grad and
    ``.grad`` as in ``predictive``."""
    _check(model, samples, _Comparative, "predictive_pair", _PAIR_CLASSES)
    with torch.no_grad():
        return _scorer_pair(model, graph_pair, sequence_pair, property_pair, eps, samples).base
