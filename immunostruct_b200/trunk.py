"""Shared pieces of the reference's model zoo, factored once (the reference repeats them per class).

``StructureTrunk``: EGNN stack -> per-graph attention -> global mean pool
(models/hybrid_models.py:82-97 / :316-331, identical in every structure-bearing model).
``SequenceVAE``: encode_vae / reparameterize / decode_vae (hybrid_models.py:63-74).
Attribute names equal the reference's so that ``state_dict`` keys and shapes match exactly.
"""
from __future__ import annotations

import torch
import torch.nn as nn
import torch.nn.functional as F

from . import functional as IF
from .graph import GraphBatch
from .layers import EGNNConv, MultiHeadAttention, SelfAttention


def _require_device_batch(graph_data):
    if not isinstance(graph_data, GraphBatch):
        raise TypeError("graph_data must be an immunostruct_b200.GraphBatch (see immunostruct_b200.batch)")
    if not graph_data.ndata["x"].is_cuda:
        raise RuntimeError("immunostruct_b200 models run on CUDA only; call graph_data.to(device) first "
                           "(there is no CPU fallback)")


class StructureTrunk:
    """Mixin: builds ``GCN_layers`` + ``self_attention`` and runs them."""

    def _build_trunk(self, gcn_layers, hidden, attention, heads=1):
        self.gat_hidden_channels = hidden
        self.GCN_layers = nn.ModuleList([EGNNConv(20, hidden, hidden, 1)])
        for _ in range(gcn_layers):
            self.GCN_layers.append(EGNNConv(hidden, hidden, hidden, 1))
        self.self_attention = SelfAttention(hidden) if attention == "sa" else MultiHeadAttention(hidden, heads)

    def structure_embedding(self, graph_data, want_attn=False, want_nodes=False, project=True):
        """-> (pooled [B,64], attention weights or None, per-node attention output or None).
        ``project=False`` leaves the attention's output projection (w_concat) to the caller.

        The per-graph ``batch_tensor`` of the reference (B host syncs per forward,
        hybrid_models.py:86-87) is replaced by the segment offsets cached on the GraphBatch."""
        _require_device_batch(graph_data)
        xin = graph_data.ndata["x"]
        node_feat, coord_feat, edge_feat = xin[:, :20], xin[:, 20:], graph_data.edata["edge_attr"]
        if not torch.is_grad_enabled():
            # inference: the whole stack through the fused kernels, nothing saved for a backward pass
            # (the attention projections ride in the last node kernel when it runs on the tensor cores)
            fuse_qkv = getattr(self.self_attention, "feature_dim", self.gat_hidden_channels) == 64 and self.gat_hidden_channels == 64
            out = IF.egnn_stack_infer(graph_data, xin, edge_feat, [l.kernel_params() for l in self.GCN_layers],
                                      qkv=self.self_attention.qkv_params() if fuse_qkv else None)
            node_feat, qkv = out if fuse_qkv else (out, None)
            return self.self_attention.pooled(graph_data, node_feat, want_attn=want_attn, want_nodes=want_nodes, qkv=qkv,
                                              project=project)
        # training: one autograd node for the whole stack (the last layer's coordinates are never consumed,
        # hybrid_models.py:323-326, so its coordinate branch is skipped and coord_mlp gets no gradient)
        # (the attention projections ride in the last node kernel here too; their backward runs inside the same node)
        fuse_qkv = getattr(self.self_attention, "feature_dim", self.gat_hidden_channels) == 64 and self.gat_hidden_channels == 64
        out = IF.egnn_stack(graph_data, xin, edge_feat, [l.kernel_params() for l in self.GCN_layers],
                            qkv=self.self_attention.qkv_params() if fuse_qkv else None)
        node_feat, qkv = out if fuse_qkv else (out, None)
        return self.self_attention.pooled(graph_data, node_feat, want_attn=want_attn, want_nodes=want_nodes, qkv=qkv,
                                          project=project)


def _tc_linear(layer, x, relu=False):
    """``layer(x)`` (+ ReLU) for the two large Linear layers.  On CUDA, in every tensor-core precision mode, forward AND
    backward run on the TMA-fed tcgen05 GEMM (csrc/gemm_tma.cu: pre-split bf16 planes, weights split once per
    parameter version); the "fp32" mode keeps torch's fp32 GEMM (a plain library GEMM)."""
    prec = IF._PRECISIONS[IF.get_precision()]
    if prec is None or x.dim() != 2 or not (x.is_cuda or IF._C.lib_is_patched()):
        y = layer(x)
        return F.relu(y) if relu else y
    if x.stride(-1) != 1:
        x = x.contiguous()
    if IF._linear_impl == "fused" and not torch.is_grad_enabled():
        # the round-1 kernel (csrc/linear_tc.cu: operands split on the fly by SIMT threads); kept for A/B timing
        node_prec = IF._C.PREC_BF16 if prec == IF._C.PREC_BF16 else IF._C.PREC_BF16X3
        return IF._C.linear_tc(x, layer.weight.detach(), None if layer.bias is None else layer.bias.detach(), relu=relu,
                               precision=node_prec)
    return IF.linear_tc(x, layer.weight, layer.bias, relu)


class SequenceVAE:
    """Mixin: the sequence VAE branch.  The two large Linear layers (vae_fc1, vae_fc4: the model's only big dense
    contractions) run on the tensor cores in the no-grad path; the tiny ones stay torch / cuBLAS."""

    def _build_vae(self, vae_input_dim, vae_hidden_dim, vae_latent_dim, cond_dim):
        self.vae_input_dim, self.vae_hidden_dim, self.vae_latent_dim = vae_input_dim, vae_hidden_dim, vae_latent_dim
        self.vae_fc1 = nn.Linear(vae_input_dim, vae_hidden_dim)
        self.vae_fc21 = nn.Linear(vae_hidden_dim, vae_latent_dim)
        self.vae_fc22 = nn.Linear(vae_hidden_dim, vae_latent_dim)
        self.vae_fc3 = nn.Linear(vae_latent_dim + cond_dim, vae_hidden_dim)
        self.vae_fc4 = nn.Linear(vae_hidden_dim, vae_input_dim)

    def encode_vae(self, x):
        h1 = _tc_linear(self.vae_fc1, x, relu=True)
        return self.vae_fc21(h1), self.vae_fc22(h1)

    def sample_eps(self, like):
        """The standard-normal draw of ``reparameterize`` (``torch.randn_like(std)``, hybrid_models.py:303) -- one
        place for both the torch path and the fused eval kernel, so tests can inject a fixed noise tensor."""
        return torch.randn_like(like)

    def reparameterize(self, mu, logvar):
        # sampled in eval mode too, exactly like the reference (hybrid_models.py:301-304)
        std = torch.exp(0.5 * logvar)
        eps = self.sample_eps(std)
        return mu + eps * std

    def decode_vae(self, z):
        return _tc_linear(self.vae_fc4, F.relu(self.vae_fc3(z)))

    def vae_branch_eval(self, sequence_data, prop_mlp, peptide_property):
        """Eval-mode, no-grad sequence branch with the small layers fused (csrc/head.cu): vae_fc1 and vae_fc4 on the
        tensor cores, property MLP + vae_fc21 / fc22 + reparameterisation + vae_fc3 in one kernel.  Same RNG draw as
        ``reparameterize`` (one standard-normal [B, latent] tensor).  -> (recon, mu, logvar, z_vae)."""
        h1 = _tc_linear(self.vae_fc1, sequence_data.reshape(-1, self.vae_input_dim), relu=True)
        eps = self.sample_eps(torch.empty(h1.shape[0], self.vae_latent_dim, dtype=h1.dtype, device=h1.device)).contiguous()
        mu, logvar, z_vae, h3 = self.vae_mid_eval(h1, prop_mlp, peptide_property, eps)
        return _tc_linear(self.vae_fc4, h3), mu, logvar, z_vae

    def vae_mid_eval(self, h1, prop_mlp, peptide_property, eps):
        """Property MLP, vae_fc21 / fc22, reparameterisation with ``eps`` [B, latent] and vae_fc3 + ReLU in one kernel
        (csrc/head.cu, no autograd).  -> (mu, logvar, z_vae, h3)."""
        d = lambda t: t.detach()
        return IF._C.vae_mid_infer(
            h1, peptide_property.contiguous(), eps, d(prop_mlp[0].weight), d(prop_mlp[0].bias), d(prop_mlp[3].weight),
            d(prop_mlp[3].bias), d(self.vae_fc21.weight), d(self.vae_fc21.bias), d(self.vae_fc22.weight),
            d(self.vae_fc22.bias), d(self.vae_fc3.weight), d(self.vae_fc3.bias))

    def vae_branch(self, sequence_data, cond=None):
        mu, logvar = self.encode_vae(sequence_data.reshape(-1, self.vae_input_dim))
        z = self.reparameterize(mu, logvar)
        if cond is not None:
            z = torch.cat([z, cond], dim=1)
        return self.decode_vae(z), mu, logvar, z


def property_mlp(out_dim):
    return nn.Sequential(nn.Linear(2, 32), nn.ReLU(True), nn.Dropout(0.1), nn.Linear(32, out_dim), nn.ReLU(True))


def classifier_mlp(in_dim, with_out=True):
    layers = [nn.Flatten(1), nn.Linear(in_dim, 32), nn.ReLU(True), nn.Dropout(0.1)]
    if with_out:
        layers.append(nn.Linear(32, 1))
    return nn.Sequential(*layers)


class LoadTrained:
    """``load_trained(path, new_head, map_location)`` (hybrid_models.py:310-313, :197-200 for SSL).  Also the cache
    hygiene of every model class: ``train()`` / ``eval()``, ``load_state_dict()`` and ``to()`` / ``cuda()`` drop the
    parameter-derived caches (fused projection weights, fusion coefficients, pre-split weight planes)."""

    _head_attr = "classifier"

    def train(self, mode: bool = True):
        IF.invalidate_caches()
        return super().train(mode)

    def load_state_dict(self, *args, **kwargs):
        IF.invalidate_caches()
        return super().load_state_dict(*args, **kwargs)

    def _apply(self, fn, *args, **kwargs):
        IF.invalidate_caches()
        return super()._apply(fn, *args, **kwargs)

    def load_trained(self, path, new_head=False, map_location=None):
        self.load_state_dict(torch.load(path, map_location=map_location))
        if new_head:
            if self._head_attr == "classifier":
                self.classifier = self.get_classifier().to(self.device)
            else:
                self.classifier_head = nn.Linear(self.mlp_features, 1).to(self.device)
