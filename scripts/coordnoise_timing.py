"""Cost of structural-uncertainty ensembles (immunostruct_b200/coordnoise.py), on one GPU.

Workloads, HybridModelv2 in the default precision mode with the inputs resident on the device, batch 512 of 200-node
10-NN graphs with 10 padded rows, sigma 1.0 on the 190 present rows of every graph and 0 on the padded rows:
  ``coordinate_ensemble`` at M = 16 and 64 structures, K = 1 and 16 latent draws.
  The host loop it replaces: M times (clone the node features, add sigma * ``torch.randn`` to columns 20..22, swap them
    into a resident ``GraphBatch`` and call ``predictive`` with the same K).  Its topology is collated once, so the loop
    pays the encoder and the head per structure but no collation.
  is_coord_noise_expand alone on one 4 096-graph pass (8 copies of the batch).  Bytes = the written pass plus one read
    of the base rows and of sigma (the base is read from L2 by the other copies).
Times are the fastest of three CUDA-event windows of --steps calls each, after --warmup calls.  The card's name and
power limit are read in the same run.  Prints one JSON line (and, with --out FILE, writes it there).

    python scripts/coordnoise_timing.py [--batch 512] [--steps 2] [--warmup 1] [--out FILE]
"""
import argparse
import json
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import immunostruct_b200 as I  # noqa: E402
from immunostruct_b200 import _C  # noqa: E402
from immunostruct_b200.coordnoise import coordinate_ensemble  # noqa: E402
from immunostruct_b200.graph import GraphBatch  # noqa: E402
from immunostruct_b200.predictive import predictive  # noqa: E402
from immunostruct_b200.synthetic import synthetic_dense, synthetic_graph_arrays  # noqa: E402

sys.path.insert(0, os.path.join(ROOT, "scripts"))
from variant_timing import HBM_PEAK, KEYS, card, fastest_ms  # noqa: E402

N, PAD = 200, 10
PASS_GRAPHS = 4096


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=512)
    ap.add_argument("--steps", type=int, default=2)
    ap.add_argument("--warmup", type=int, default=1)
    ap.add_argument("--out", default=None, help="also write the JSON line to this file")
    args = ap.parse_args()
    assert torch.cuda.is_available(), "needs a CUDA device"
    dev = torch.device("cuda:0")
    st, wu, b = args.steps, args.warmup, args.batch
    out = {"precision": I.get_precision(), "card": card()}

    torch.manual_seed(1)
    model = I.model_map["HybridModelv2"](vae_input_dim=5943, device=dev).to(dev).eval()
    arr = {k: v.to(dev) for k, v in synthetic_graph_arrays(b, N, 10, seed=1, n_pad=PAD).items()}
    dense = synthetic_dense(b, seed=1)
    g = GraphBatch.from_arrays(*(arr[k] for k in KEYS), max_nodes=N).validate()
    seq, prop = dense["seq"].to(dev), dense["prop"].to(dev)
    sigma = ((torch.arange(b * N, device=dev) % N) < N - PAD).float()      # 1.0 on present rows, 0 on padded rows

    r = {"workload": f"HybridModelv2, batch {b} of {N}-node graphs, sigma 1.0 on the {N - PAD} present rows of each"}
    for m in (16, 64):
        for k in (1, 16):
            ms = fastest_ms(lambda: coordinate_ensemble(model, g, seq, prop, sigma=sigma, structures=m, seed=7,
                                                        samples=k), st, wu)
            r[f"ms_ensemble_M{m}_K{k}"] = ms
            r[f"us_per_graph_M{m}_K{k}"] = 1e3 * ms / (m * b)

    # ---- the host loop: clone, torch.randn coordinate noise, predictive, per structure ----
    gl = GraphBatch.from_arrays(*(arr[k] for k in KEYS), max_nodes=N).validate()
    x0 = arr["x"]
    s3 = sigma[:, None]

    def loop(m, k):
        for _ in range(m):
            x = x0.clone()
            x[:, 20:] += s3 * torch.randn(x.shape[0], 3, device=dev)
            gl.ndata["x"] = x
            predictive(model, gl, seq, prop, samples=k)

    for m in (16, 64):
        for k in (1, 16):
            ms = fastest_ms(lambda: loop(m, k), 1, 1)
            r[f"ms_host_loop_M{m}_K{k}"] = ms
            r[f"speedup_M{m}_K{k}"] = ms / r[f"ms_ensemble_M{m}_K{k}"]

    # ---- is_coord_noise_expand alone, one 4096-graph pass ----
    copies = PASS_GRAPHS // b
    n = x0.shape[0]
    xo = torch.empty(copies * n, 23, device=dev)
    expand = lambda: _C.coord_noise_expand(x0, g.node_off, sigma, 7, 0, 0, xo)
    k_ms = fastest_ms(expand, 50, 5)
    e = {"graphs": copies * b, "us": 1e3 * k_ms, "bytes": 4 * 23 * n * copies + 4 * 23 * n + 4 * n}
    e["bytes_per_s"] = e["bytes"] / (k_ms * 1e-3)
    e["share_of_hbm_peak"] = e["bytes_per_s"] / HBM_PEAK
    pass_ms = r["ms_ensemble_M16_K1"] * copies / 16
    e["share_of_a_pass_M16_K1"] = k_ms / pass_ms
    r["is_coord_noise_expand"] = e
    out["coordnoise"] = r

    line = json.dumps(out)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
