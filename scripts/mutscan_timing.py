"""Cost of the single-residue mutational scan (immunostruct_b200/mutagenesis.py), on one GPU.

Workloads, in the default precision mode with the inputs resident on the device (200-node 10-NN graphs, 10 padded rows),
P = 9 peptide sites per sample (node rows 0..8 and sequence rows 0..8), all 20 residue types: 180 variants per sample.
  HybridModelv2 at batch 512 (92 160 variants): ``mutational_scan`` at K = 1 and K = 16, against the hand-written loop
    (180 mutant batches built with torch indexing on the device, each collated and run through one ``model()`` call);
    one eval forward for scale.
  HybridModelv2_Comparative at 256 pairs: ``mutational_scan_pair`` (K = 1) against the same loop over
    ``forward_comparative``, which re-runs the wild type for every variant.
  is_mutscan_expand alone: one pass of 8 copies of the 512-graph batch.  Bytes = one read of the base features plus the
    write of the 8 copies (x23 and sequence one-hots); share of HBM peak against the data sheet's 7.7 TB/s.
Times are the fastest of three CUDA-event windows of --steps calls each, after --warmup calls.  The card's name and
power limit are read in the same run.  Prints one JSON line (and, with --out FILE, writes it there).

    python scripts/mutscan_timing.py [--batch 512] [--pairs 256] [--steps 2] [--warmup 1] [--out FILE]
"""
import argparse
import json
import os
import subprocess
import sys

import torch
import torch.nn.functional as F

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import immunostruct_b200 as I  # noqa: E402
from immunostruct_b200 import _C  # noqa: E402
from immunostruct_b200.graph import GraphBatch  # noqa: E402
from immunostruct_b200.mutagenesis import mutational_scan, mutational_scan_pair, scan_sites  # noqa: E402
from immunostruct_b200.synthetic import synthetic_dense, synthetic_graph_arrays  # noqa: E402

SITES = 9
HBM_PEAK = 7.7e12          # bytes/s, NVIDIA data sheet (HGX B200, per GPU)
KEYS = ("x", "src", "dst", "edge_attr", "node_counts", "edge_counts")


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
    """Device batch whose sequence rows 0..8 carry the residues of node rows 0..8 (identity column map)."""
    arr = {k: v.to(dev) for k, v in synthetic_graph_arrays(b, 200, 10, seed=seed, n_pad=10).items()}
    dense = synthetic_dense(b, seed=seed)
    seq = dense["seq"].to(dev)
    native = arr["x"].reshape(b, 200, 23)[:, :SITES, :20].argmax(-1)
    seq[:, :SITES] = F.one_hot(native, seq.shape[2]).float()
    gb = GraphBatch.from_arrays(*(arr[k] for k in KEYS), max_nodes=200).validate()
    return arr, gb, seq, dense["prop"].to(dev)


def hand_loop(arr, seq, run):
    """The scan written by hand: per (site, residue) a mutant copy of the batch by torch indexing, collated, then run."""
    b = seq.shape[0]
    rows = torch.arange(b, device=seq.device) * 200
    for p in range(SITES):
        for c in range(20):
            x = arr["x"].clone()
            x[rows + p, :20] = F.one_hot(torch.tensor(c, device=x.device), 20).float()
            s = seq.clone()
            s[:, p] = F.one_hot(torch.tensor(c, device=x.device), s.shape[2]).float()
            run(GraphBatch.from_arrays(x, *(arr[k] for k in KEYS[1:]), max_nodes=200), s)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=512)
    ap.add_argument("--pairs", type=int, default=256)
    ap.add_argument("--steps", type=int, default=2)
    ap.add_argument("--warmup", type=int, default=1)
    ap.add_argument("--out", default=None, help="also write the JSON line to this file")
    args = ap.parse_args()
    assert torch.cuda.is_available(), "needs a CUDA device"
    dev = torch.device("cuda:0")
    st, wu = args.steps, args.warmup
    out = {"precision": I.get_precision(), "sites": SITES, "card": card()}
    cols = torch.arange(20)

    # ---- HybridModelv2, batch B ----
    b = args.batch
    torch.manual_seed(1)
    model = I.model_map["HybridModelv2"](vae_input_dim=5943, device=dev).to(dev).eval()
    arr, g, seq, prop = inputs(b, 1, dev)
    ni = torch.arange(SITES).repeat(b, 1)
    h = {"workload": f"HybridModelv2, batch {b}, {SITES * 20 * b} variants"}
    with torch.no_grad():
        h["ms_forward"] = fastest_ms(lambda: model(g, seq, prop), 5, 2)
    for k in (1, 16):
        h[f"ms_scan_K{k}"] = fastest_ms(lambda: mutational_scan(model, g, seq, prop, ni, ni, seq_columns=cols, samples=k),
                                        st, wu)

    def loop():
        with torch.no_grad():
            hand_loop(arr, seq, lambda gm, s: model(gm, s, prop))

    h["ms_hand_loop_180_forwards"] = fastest_ms(loop, st, wu)
    h["scan_K1_speedup_over_hand_loop"] = h["ms_hand_loop_180_forwards"] / h["ms_scan_K1"]
    h["scan_K1_in_forwards_per_variant_batch"] = h["ms_scan_K1"] / (SITES * 20) / h["ms_forward"]

    # ---- the expansion kernel alone: one pass of r = 8 copies ----
    r = 8
    sites = scan_sites(SITES, dev)[:r].contiguous()
    L, V = seq.shape[1], seq.shape[2]
    xo = torch.empty(r * g.n_nodes, 23, device=dev)
    so = torch.empty(r * b, L, V, device=dev)
    flag = torch.zeros(1, dtype=torch.int32, device=dev)
    nid, cold = ni.to(dev), cols.to(dev)
    base_bytes = 4 * (g.n_nodes * 23 + b * L * V)
    k_ms = fastest_ms(lambda: _C.mutscan_expand(g.ndata["x"], g.node_off, nid, seq, nid, cold, sites, xo, so, flag), 50, 5)
    assert int(flag) == 0
    e = {"copies": r, "graphs_per_copy": b, "us": 1e3 * k_ms, "bytes": (1 + r) * base_bytes}
    e["bytes_per_s"] = e["bytes"] / (k_ms * 1e-3)
    e["share_of_hbm_peak"] = e["bytes_per_s"] / HBM_PEAK
    h["is_mutscan_expand"] = e
    out["hybrid_v2"] = h
    del model, g, seq, prop, arr, xo, so

    # ---- HybridModelv2_Comparative, P pairs ----
    p = args.pairs
    torch.manual_seed(2)
    model = I.model_map["HybridModelv2_Comparative"](vae_input_dim=5943, device=dev).to(dev).eval()
    arr_c, gc, sc, pc = inputs(p, 2, dev)
    _, gw, sw, pw = inputs(p, 3, dev)
    ni = torch.arange(SITES).repeat(p, 1)
    c = {"workload": f"HybridModelv2_Comparative, {p} pairs, use_wt_for_downstream, {SITES * 20 * p} variants"}
    with torch.no_grad():
        c["ms_forward_comparative"] = fastest_ms(lambda: model.forward_comparative((gc, gw), (sc, sw), (pc, pw)), 5, 2)
    c["ms_scan_pair_K1"] = fastest_ms(lambda: mutational_scan_pair(model, (gc, gw), (sc, sw), (pc, pw), ni, ni,
                                                                   seq_columns=cols), st, wu)

    def loop_pair():
        with torch.no_grad():
            hand_loop(arr_c, sc, lambda gm, s: model.forward_comparative((gm, gw), (s, sw), (pc, pw)))

    c["ms_hand_loop_180_forward_comparative"] = fastest_ms(loop_pair, st, wu)
    c["scan_pair_speedup_over_hand_loop"] = c["ms_hand_loop_180_forward_comparative"] / c["ms_scan_pair_K1"]
    out["comparative_v2"] = c

    line = json.dumps(out)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
