"""Nearest neighbours in the classifier's feature space.

``embed`` / ``embed_pair`` return the classifier's hidden layer, ReLU(classifier[1](combined)): the 32 features that the
output layer (``classifier[4]``, or ``classifier_head`` / ``node_predictor_head`` of the SSL classes) reads, taken after
the fusion attention in v2 models.  The latent is fixed at its mean (z = mu, no noise), so the features are
deterministic.  The structure trunk and the VAE encoder run as in ``predictive``; one head kernel
(``is_head_features_infer``, csrc/head.cu) writes the hidden layer with the arithmetic of the fused eval forward.

``nearest`` is an exact k-nearest-neighbour search of query rows in a bank of rows (``is_knn``, csrc/knn.cu), in
squared Euclidean distance with a fixed fp32 rounding sequence per pair and the total order (distance, bank index).
With a bank of labelled training features it gives explanations by example; the distance to the k-th neighbour,
leave-self-out on the training set, is the deep k-NN out-of-distribution score.
"""
from __future__ import annotations

from dataclasses import dataclass
from typing import Optional

import torch

from . import functional as IF
from .comparative_models import _Comparative
from .hybrid_models import _Hybrid
from .predictive import _CLASSES, _PAIR_CLASSES, _check, _encode, _head_params

Tensor = torch.Tensor


@dataclass
class Neighbors:
    """The k nearest bank rows of every query, ascending by (distance, index).  Unfilled slots (fewer than k eligible
    rows) hold index -1 and distance +inf."""
    index: Tensor         # [Q, k] int64 rows of the bank
    distance: Tensor      # [Q, k] float32 squared Euclidean distance


def _features(model, items):
    wc, bc, coef, n_head, w1, b1, _, _ = _head_params(model)
    return IF._C.head_features_infer([it[:2] + it[3:] for it in items], wc, bc, coef, n_head, w1, b1)


def embed(model, graph_data, sequence_data, peptide_property) -> Tensor:
    """Features [B, 32] float32 of ``model(graph_data, sequence_data, peptide_property)`` at z = mu: the classifier's
    hidden layer.  Follows ``model.forward``: for the comparative classes with ``use_wt_for_downstream`` the single
    form repeats the item across the pair-wide classifier.

    Deterministic: one call is bit-reproducible run to run, and a graph's features in another batch agree to the 1e-6
    batch-position bound of the fused forward.  The model must be in eval mode; runs under ``torch.no_grad()`` and
    leaves every ``.grad`` untouched.  ``vae_fc4`` (the decoder) is not run."""
    _check(model, 1, (_Hybrid, _Comparative), "embed", _CLASSES)
    with torch.no_grad():
        item = _encode(model, graph_data, sequence_data, peptide_property)
        repeat = isinstance(model, _Comparative) and model.use_wt_for_downstream
        return _features(model, [item, item] if repeat else [item])


def embed_pair(model, graph_pair, sequence_pair, property_pair) -> Tensor:
    """Features [B, 32] float32 of ``model.forward_comparative(graph_pair, sequence_pair, property_pair)`` at z = mu
    for the four comparative classes: the cancer item against its wild type.  Without ``use_wt_for_downstream`` the
    classifier reads the cancer item only, and the wild type is neither run nor read.  Eval mode, no_grad and
    ``.grad`` as in ``embed``."""
    _check(model, 1, _Comparative, "embed_pair", _PAIR_CLASSES)
    n = 2 if model.use_wt_for_downstream else 1
    with torch.no_grad():
        items = [_encode(model, graph_pair[i], sequence_pair[i], property_pair[i]) for i in range(n)]
        return _features(model, items)


def _slices(n_query: int, n_bank: int) -> int:
    """Bank slice count of ``nearest``: enough (query tile, slice) CTAs to occupy every SM of the current device when
    the queries alone are too few, and never a slice without a full 128-row tile."""
    tiles = -(-n_query // IF._C.KNN_QUERY_TILE)
    return max(1, min(IF._C.knn_max_slices(n_bank), -(-IF._C.num_sms() // tiles)))


def nearest(query: Tensor, bank: Tensor, k: int, *, exclude: Optional[Tensor] = None) -> Neighbors:
    """The exact k nearest rows of ``bank`` [R, D] for every row of ``query`` [Q, D] (float32 CUDA, contiguous;
    1 <= k <= 64, 1 <= D <= 256, R < 2^31).

    Distance: squared Euclidean in fp32, each pair summed in ascending feature order as t = q_d - r_d,
    acc = fmaf(t, t, acc); the value does not depend on how the search is tiled, sliced or batched.  For cosine order
    pass L2-normalised rows (|a - b|^2 = 2 - 2 cos).  Order: ascending (distance, index), ties to the smaller index, so
    the result is bit-identical whatever the launch configuration.  A bank row with a NaN feature is never returned and
    a query with a NaN feature gets no neighbours; unfilled slots hold index -1 and distance +inf.

    ``exclude`` int64 [Q]: the bank row query q must not return (-1 = none); ``torch.arange(Q)`` searches a bank
    against itself leaving each row out.  Every argument is checked before the launch (the range of ``exclude`` with
    one host read)."""
    if not isinstance(query, Tensor) or not isinstance(bank, Tensor) or query.dim() != 2 or bank.dim() != 2:
        raise ValueError("nearest: query [Q, D] and bank [R, D] tensors expected")
    slices = 1
    if query.is_cuda and 1 <= bank.shape[0] < 2 ** 31 and query.shape[0] >= 1:
        slices = _slices(query.shape[0], bank.shape[0])
    index, distance = IF._C.knn(query, bank, k, exclude, slices=slices)
    return Neighbors(index, distance)
