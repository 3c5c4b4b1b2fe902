"""Shared test helpers: build product inputs from golden groups, inject eps, collect grads, compare per segment,
run the full-model oracle in chunks."""
import contextlib
import types

import torch

import immunostruct_b200 as I
from immunostruct_b200.graph import GraphBatch
from immunostruct_b200.synthetic import split_graphs

def graph_batch(arrays, device="cpu"):
    """golden/synthetic 'graph' group (graph-local endpoints) -> GraphBatch on ``device``."""
    gb = GraphBatch.from_arrays(arrays["x"].float(), arrays["src"], arrays["dst"], arrays["edge_attr"].float(),
                                arrays["node_counts"], arrays["edge_counts"],
                                max_nodes=int(arrays["node_counts"].max()))
    if torch.device(device).type == "cpu":
        gb._collate()          # CPU: only reachable with the kernel contracts patched in (tests)
        return gb
    return gb.to(device)


def inject_eps(model, *eps_list):
    """Make the model's reparameterisation consume the given noise tensors in order (instead of randn_like);
    ``sample_eps`` feeds both ``reparameterize`` and the fused eval-mode kernel."""
    it = iter(eps_list)

    def sample_eps(self, like):
        return next(it).to(like.device, like.dtype)

    model.sample_eps = types.MethodType(sample_eps, model)
    return model


def named_grads(model):
    return {k: p.grad for k, p in model.named_parameters()}


def build_model(name, golden, device="cpu", **kw):
    meta = golden["meta"]
    model = I.model_map[name](vae_input_dim=231, device=device, gcn_layers=int(meta["gcn_layers"]) - 1,
                              vae_hidden_dim=int(meta.get("vae_hidden_dim", torch.tensor(32))), **kw)
    missing = model.load_state_dict(golden["weights"], strict=True)
    assert not missing.missing_keys and not missing.unexpected_keys
    return model.to(device).eval()


def log_error(msg):
    """One line of the margin log the kernel tests keep (test_kernels_gpu._log)."""
    from test_kernels_gpu import _log          # imported here: test_kernels_gpu imports this module
    _log(msg)


# ---- fp64 runs of the kernel contracts ----------------------------------------------------------------------------
@contextlib.contextmanager
def fp64_default():
    """torch's default dtype is float64 inside the block: the contracts of oracle/kernel_contracts.py allocate their
    intermediates with the default dtype, so with double inputs they compute in fp64.  The previous default comes back
    however the block ends."""
    old = torch.get_default_dtype()
    torch.set_default_dtype(torch.float64)
    try:
        yield
    finally:
        torch.set_default_dtype(old)


# ---- per-segment comparison ---------------------------------------------------------------------------------------
def tile_segments(n_rows, rows=128):
    """Segment id of each row: one segment per ``rows``-row tile."""
    return torch.arange(n_rows) // rows


def graph_segments(node_off):
    """Segment id of each node row: one segment per graph."""
    off = node_off.detach().cpu().long()
    return torch.repeat_interleave(torch.arange(off.numel() - 1), off[1:] - off[:-1])


def close_per_segment(got, ref, seg, tol, what="", floor=1e-3):
    """Rows grouped into segments (``seg[i]`` = segment of row i): within each segment, max |got - ref| must stay within
    ``tol`` times that segment's own max |ref|, floored at ``floor`` times the max |ref| of the whole tensor (so that
    near-zero segments are not judged on noise).  A whole-tensor scale would let an error in a small-valued segment --
    a 150-node graph's gradient next to a 1-node graph's -- pass at a fraction of its own size.  Every value of ``got``
    must be finite: outputs are NaN-filled before the kernel runs, so a row no CTA wrote fails here."""
    got, ref = got.detach().double().cpu(), ref.detach().double().cpu()
    assert got.shape == ref.shape, (what, got.shape, ref.shape)
    g2, r2 = got.reshape(got.shape[0], -1), ref.reshape(ref.shape[0], -1)
    bad = int((~torch.isfinite(g2)).any(1).sum())
    assert bad == 0, f"{what}: {bad} rows with non-finite values"
    seg = seg.long()
    assert seg.numel() == g2.shape[0], (what, seg.numel(), g2.shape[0])
    nseg = int(seg.max()) + 1 if seg.numel() else 0
    err = torch.zeros(nseg, dtype=torch.float64).scatter_reduce(0, seg, (g2 - r2).abs().amax(1), "amax")
    scale = torch.zeros(nseg, dtype=torch.float64).scatter_reduce(0, seg, r2.abs().amax(1), "amax")
    gscale = float(r2.abs().max()) if r2.numel() else 0.0
    ratio = err / scale.clamp_min(floor * gscale).clamp_min(1e-30)
    worst = int(ratio.argmax()) if nseg else 0
    wr = float(ratio[worst]) if nseg else 0.0
    log_error(f"{what}: worst segment {worst}/{nseg} err {float(err[worst]) if nseg else 0.0:.3e} "
              f"scale {float(scale[worst]) if nseg else 0.0:.3e} err/bound {wr / tol:.3f}")
    assert wr <= tol, (f"{what}: segment {worst} of {nseg}: max abs err {float(err[worst]):.3e} vs segment scale "
                       f"{float(scale[worst]):.3e} (rel {wr:.2e} > {tol:.0e})")


# ---- batches of graphs --------------------------------------------------------------------------------------------
def slice_graphs(arrays, lo, hi):
    """Graphs [lo, hi) of a batch of graph-local arrays (synthetic_graph_arrays / random_multigraph_arrays layout)."""
    nc, ec = arrays["node_counts"].cpu(), arrays["edge_counts"].cpu()
    n0, n1 = int(nc[:lo].sum()), int(nc[:hi].sum())
    e0, e1 = int(ec[:lo].sum()), int(ec[:hi].sum())
    return {"x": arrays["x"][n0:n1], "src": arrays["src"][e0:e1], "dst": arrays["dst"][e0:e1],
            "edge_attr": arrays["edge_attr"][e0:e1], "node_counts": arrays["node_counts"][lo:hi],
            "edge_counts": arrays["edge_counts"][lo:hi]}


def concat_graphs(*batches):
    """One batch holding the graphs of every argument in turn (endpoints are graph-local, so nothing is renumbered)."""
    return {k: torch.cat([b[k] for b in batches]) for k in ("x", "src", "dst", "edge_attr", "node_counts", "edge_counts")}


def oracle_training_step(state, arr, dense, eps, dtype, chunk=None, pos_weight=4.25):
    """HybridModelv2's eval-mode training step on the full-model oracle (oracle/reference_ops.py) in ``dtype``:
    forward, ``bce_loss``, backward.  With ``chunk`` the batch is run ``chunk`` graphs at a time: every term of
    ``bce_loss`` is a mean over rows, so the loss of the batch and its gradients are the sum over chunks of the chunk's
    loss weighted by (graphs in the chunk) / (graphs in the batch); nothing in the eval-mode forward couples samples.
    Returns (logits [B, 1], loss, {name: grad})."""
    from oracle import reference_ops as R
    b = int(arr["node_counts"].numel())
    chunk = chunk or b
    p = {k: v.detach().clone().cpu().to(dtype).requires_grad_(True) for k, v in state.items()}
    outs, loss = [], torch.zeros((), dtype=dtype)
    for lo in range(0, b, chunk):
        hi = min(lo + chunk, b)
        g = R.dgl_batch(split_graphs(slice_graphs(arr, lo, hi)))
        g = dict(g, x=g["x"].to(dtype), edge_attr=g["edge_attr"].to(dtype))
        seq = dense["seq"][lo:hi].to(dtype)
        recon, mu, logvar, out = R.hybrid_forward(p, g, seq, dense["prop"][lo:hi].to(dtype), eps[lo:hi].to(dtype))
        part = R.bce_loss(recon, seq, mu, logvar, out, dense["target"][lo:hi].to(dtype), pos_weight) * ((hi - lo) / b)
        part.backward()
        outs.append(out.detach())
        loss = loss + part.detach()
    return torch.cat(outs), loss, {k: v.grad for k, v in p.items()}
