"""Cost of the predictive mean and spread over the reparameterisation draw (immunostruct_b200/predictive.py), on one GPU.

Workloads, in the default precision mode with the inputs resident on the device (200-node 10-NN graphs):
  HybridModelv2 at batch 512, and HybridModelv2_Comparative at 256 cancer / wild-type pairs.
Times, as the fastest of three CUDA-event windows of --steps calls each (after --warmup calls):
  one eval forward; 16 sequential eval forwards; predictive (predictive_pair) at K in {1, 16, 64, 256};
  the multi-draw head kernel alone (is_head_mc_infer at K = 64, per draw); the single-draw head kernel alone
  (is_head_infer, hybrid only).
The card's name and power limit are read in the same run.  Prints one JSON line (and, with --out FILE, writes it there).

    python scripts/predictive_timing.py [--batch 512] [--pairs 256] [--steps 5] [--warmup 2] [--out FILE]
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
from immunostruct_b200.graph import GraphBatch  # noqa: E402
from immunostruct_b200.predictive import _encode, _head_params, predictive, predictive_pair  # noqa: E402
from immunostruct_b200.synthetic import synthetic_dense, synthetic_graph_arrays  # noqa: E402

DRAWS = (1, 16, 64, 256)


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
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        q = "unknown"
    return {"name": torch.cuda.get_device_name(0), "nvidia_smi_name_and_power_limit": q}


def inputs(b, seed, dev):
    arr = synthetic_graph_arrays(b, 200, 10, seed=seed, n_pad=10)
    dense = synthetic_dense(b, seed=seed)
    keys = ("x", "src", "dst", "edge_attr", "node_counts", "edge_counts")
    gb = GraphBatch.from_arrays(*(arr[k] for k in keys), max_nodes=200).to(dev).validate()
    return gb, dense["seq"].to(dev), dense["prop"].to(dev)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=512)
    ap.add_argument("--pairs", type=int, default=256)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--out", default=None, help="also write the JSON line to this file")
    args = ap.parse_args()
    assert torch.cuda.is_available(), "needs a CUDA device"
    dev = torch.device("cuda:0")
    st, wu = args.steps, args.warmup
    out = {"precision": I.get_precision(), "card": card()}

    # ---- HybridModelv2, batch B ----
    b = args.batch
    torch.manual_seed(1)
    model = I.model_map["HybridModelv2"](vae_input_dim=5943, device=dev).to(dev).eval()
    g, seq, prop = inputs(b, 1, dev)

    def fwd():
        with torch.no_grad():
            model(g, seq, prop)

    def fwd16():
        for _ in range(16):
            fwd()

    h = {"workload": f"HybridModelv2, batch {b}"}
    h["ms_forward"] = fastest_ms(fwd, st, wu)
    h["ms_16_forwards"] = fastest_ms(fwd16, st, wu)
    for k in DRAWS:
        h[f"ms_predictive_K{k}"] = fastest_ms(lambda: predictive(model, g, seq, prop, samples=k), st, wu)
    h["predictive_K64_over_forward"] = h["ms_predictive_K64"] / h["ms_forward"]
    with torch.no_grad():
        params = _head_params(model)
        pooled, mu, logvar, z_vae = _encode(model, g, seq, prop)
        eps = torch.randn(64, b, 32, device=dev)
        item = (pooled, mu, logvar, z_vae, eps)
        h["us_head_mc_infer_per_draw_K64"] = 1e3 * fastest_ms(lambda: _C.head_mc_infer([item], *params), 20, 3) / 64
        Wc, bc, coef, n_head, W1, b1, W2, b2 = params
        h["us_head_infer"] = 1e3 * fastest_ms(lambda: _C.head_infer(pooled, Wc, bc, z_vae, coef, n_head, W1, b1, W2, b2),
                                              200, 10)
    out["hybrid_v2"] = h
    del model, g, seq, prop

    # ---- HybridModelv2_Comparative, P pairs ----
    p = args.pairs
    torch.manual_seed(2)
    model = I.model_map["HybridModelv2_Comparative"](vae_input_dim=5943, device=dev).to(dev).eval()
    gc, sc, pc = inputs(p, 2, dev)
    gw, sw, pw = inputs(p, 3, dev)
    pair = ((gc, gw), (sc, sw), (pc, pw))

    def fwd_pair():
        with torch.no_grad():
            model.forward_comparative(*pair)

    def fwd_pair16():
        for _ in range(16):
            fwd_pair()

    c = {"workload": f"HybridModelv2_Comparative, {p} pairs, use_wt_for_downstream"}
    c["ms_forward_comparative"] = fastest_ms(fwd_pair, st, wu)
    c["ms_16_forwards_comparative"] = fastest_ms(fwd_pair16, st, wu)
    for k in DRAWS:
        c[f"ms_predictive_pair_K{k}"] = fastest_ms(lambda: predictive_pair(model, *pair, samples=k), st, wu)
    c["predictive_pair_K64_over_forward"] = c["ms_predictive_pair_K64"] / c["ms_forward_comparative"]
    with torch.no_grad():
        params = _head_params(model)
        items = [_encode(model, gr, s, pr) + (torch.randn(64, p, 32, device=dev),) for gr, s, pr in zip(*pair)]
        c["us_head_mc_infer_per_draw_K64"] = 1e3 * fastest_ms(lambda: _C.head_mc_infer(items, *params), 20, 3) / 64
    out["comparative_v2"] = c

    line = json.dumps(out)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
