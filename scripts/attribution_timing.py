"""Cost of input gradients and integrated gradients at batch 512 (HybridModelv2, 200-node 10-NN graphs), on one GPU.

Times, as the fastest of three CUDA-event windows of --steps calls each (after --warmup calls):
  (i)   forward + backward of the BCE loss with parameter gradients only (the training step without the optimiser);
  (ii)  the same with x23 and edge_attr requiring grad (the input gradients of the whole EGNN stack);
  (iii) integrated_gradients(steps=32) of the logit;
and the edge-feature gradient kernel alone (is_egnn_edge_attr_grad, accumulate = 1, one layer's gz1 of the batch) with
its achieved bandwidth against a device-to-device copy measured in the same run.  The card's name and power limit are
read in the same run.  Prints one JSON line (and, with --out FILE, writes it there too).

    python scripts/attribution_timing.py [--batch 512] [--steps 5] [--warmup 2] [--out FILE]
"""
import argparse
import json
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import immunostruct_b200 as I  # noqa: E402
from immunostruct_b200 import _C  # noqa: E402
from immunostruct_b200.attribution import integrated_gradients  # noqa: E402
from immunostruct_b200.graph import GraphBatch  # noqa: E402
from immunostruct_b200.synthetic import synthetic_dense, synthetic_graph_arrays  # noqa: E402


def fastest_ms(fn, steps, warmup, windows=3):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    best = float("inf")
    for _ in range(windows):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            fn()
        e1.record()
        e1.synchronize()
        best = min(best, e0.elapsed_time(e1) / steps)
    return best


def card():
    name = torch.cuda.get_device_name(0)
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        q = "unknown"
    return {"name": name, "power_limit_and_max_sm_clock": q}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=512)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--ig-steps", type=int, default=32)
    ap.add_argument("--out", default=None, help="also write the JSON line to this file")
    args = ap.parse_args()
    assert torch.cuda.is_available(), "needs a CUDA device"
    dev = torch.device("cuda:0")
    b = args.batch
    arr = synthetic_graph_arrays(b, 200, 10, seed=1, n_pad=10)
    dense = synthetic_dense(b, seed=1)
    torch.manual_seed(1)
    model = I.model_map["HybridModelv2"](vae_input_dim=5943, device=dev).to(dev).eval()
    keys = ("x", "src", "dst", "edge_attr", "node_counts", "edge_counts")
    gb = GraphBatch.from_arrays(*(arr[k] for k in keys), max_nodes=200).to(dev).validate()
    seq, prop, y = dense["seq"].to(dev), dense["prop"].to(dev), dense["target"].to(dev)
    losses = I.Losses(5943, [4.25, 1.0], sequence=True)
    x0, ea0 = gb.ndata["x"], gb.edata["edge_attr"]

    def train_bwd(inputs):
        def fn():
            x, ea = x0.detach().requires_grad_(inputs), ea0.detach().requires_grad_(inputs)
            gb.ndata["x"], gb.edata["edge_attr"] = x, ea
            model.zero_grad(set_to_none=True)
            r, mu, lv, out = model(gb, seq, prop)
            losses.BCE_loss(r, seq, mu, lv, out, y).backward()
        return fn

    out = {"workload": f"HybridModelv2, batch {b}, 200-node 10-NN graphs, precision {I.get_precision()} (training kernels bf16x3)",
           "card": card()}
    out["ms_fwd_bwd_param_grads"] = fastest_ms(train_bwd(False), args.steps, args.warmup)
    out["ms_fwd_bwd_param_and_input_grads"] = fastest_ms(train_bwd(True), args.steps, args.warmup)
    gb.ndata["x"], gb.edata["edge_attr"] = x0, ea0
    eps = torch.randn(b, 32, device=dev)
    out["ms_integrated_gradients"] = fastest_ms(
        lambda: integrated_gradients(model, gb, seq, prop, steps=args.ig_steps, eps=eps), 1, 1)
    out["integrated_gradients_steps"] = args.ig_steps

    # the edge-feature gradient kernel alone: gz1 [E, 64] read once, csr_eid read, g_a read and written (accumulate)
    e = gb.n_edges
    gz1 = torch.randn(e, 64, device=dev)
    W1 = model.GCN_layers[1].edge_mlp[0].weight.detach().contiguous()
    g_a = torch.zeros(e, device=dev)
    kernel_ms = fastest_ms(lambda: _C.egnn_edge_attr_grad(gz1, gb, W1, 64, g_a, True), 50, 5)
    kernel_bytes = e * (64 * 4 + 4 + 4 + 4)
    big = torch.empty(1 << 29, dtype=torch.uint8, device=dev)          # 512 MB, well beyond the 126 MB L2
    dst = torch.empty_like(big)
    copy_ms = fastest_ms(lambda: dst.copy_(big), 20, 3)
    copy_gbs = 2 * big.numel() / copy_ms / 1e6
    out["edge_attr_grad_kernel"] = {"n_edges": e, "ms": kernel_ms, "bytes": kernel_bytes,
                                    "GB_per_s": kernel_bytes / kernel_ms / 1e6,
                                    "measured_copy_GB_per_s": copy_gbs,
                                    "fraction_of_measured_copy": kernel_bytes / kernel_ms / 1e6 / copy_gbs}
    line = json.dumps(out)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
