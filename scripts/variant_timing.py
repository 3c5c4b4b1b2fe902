"""Cost of scoring variant libraries (immunostruct_b200/mutagenesis.py: score_variants), on one GPU.

Workloads, in the default precision mode with the inputs resident on the device (200-node 10-NN graphs, 10 padded rows):
  HybridModelv2 on 8 templates, a library of 32 768 variants, each a random template with 1 to 9 random substitutions
    at distinct peptide rows 0..8: ``score_variants`` at K = 1 and K = 16, against the same library built by hand
    (per 512 variants: torch indexing on the host templates, ``batch``, ``.to(device)``, one ``model()`` call).
  ``score_variants`` against ``mutational_scan`` on the same single-site set (batch 512, 9 sites, 20 residues, copy-major
    order): the price of the per-pass gather and collation over the scan's replicated topology.
  is_variant_expand and the pass's collation alone, on one pass of 4 096 variants of the library, and their share of
    that pass.  Bytes of the expansion = the written pass (x23, edges, sequences); the base is read from L2.
Times are the fastest of three CUDA-event windows of --steps calls each, after --warmup calls.  The card's name and
power limit are read in the same run.  Prints one JSON line (and, with --out FILE, writes it there).

    python scripts/variant_timing.py [--variants 32768] [--steps 2] [--warmup 1] [--out FILE]
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
from immunostruct_b200.graph import Graph, GraphBatch, batch  # noqa: E402
from immunostruct_b200.mutagenesis import mutational_scan, score_variants  # noqa: E402
from immunostruct_b200.synthetic import synthetic_dense, synthetic_graph_arrays  # noqa: E402

SITES = 9
HAND_CHUNK = 512
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


def inputs(b, seed):
    """Host batch whose sequence rows 0..8 carry the residues of node rows 0..8 (identity column map)."""
    arr = synthetic_graph_arrays(b, 200, 10, seed=seed, n_pad=10)
    dense = synthetic_dense(b, seed=seed)
    seq = dense["seq"]
    seq[:, :SITES] = F.one_hot(arr["x"].reshape(b, 200, 23)[:, :SITES, :20].argmax(-1), seq.shape[2]).float()
    return arr, seq, dense["prop"]


def library(n_var, b, seed):
    """Random library: template, 1..9 distinct peptide rows, random residues -> (sample, offsets, rows, residues)."""
    gen = torch.Generator().manual_seed(seed)
    sample = torch.randint(0, b, (n_var,), generator=gen)
    counts = torch.randint(1, SITES + 1, (n_var,), generator=gen)
    rows = torch.rand(n_var, SITES, generator=gen).argsort(1)
    keep = torch.arange(SITES).unsqueeze(0) < counts.unsqueeze(1)
    rows = rows[keep]
    res = torch.randint(0, 20, (rows.numel(),), generator=gen)
    offsets = torch.cat([torch.zeros(1, dtype=torch.int64), counts.cumsum(0)])
    return sample, offsets, rows, res


def hand_built(arr, seq, sample, offsets, rows, res, lo, hi):
    """Variants lo..hi built on the host: per variant a Graph with substituted rows, then ``batch``."""
    graphs, seqs = [], []
    for v in range(lo, hi):
        b = int(sample[v])
        s0, s1 = int(offsets[v]), int(offsets[v + 1])
        x = arr["x"][b * 200:(b + 1) * 200].clone()
        s = seq[b].clone()
        x[rows[s0:s1], :20] = F.one_hot(res[s0:s1], 20).float()
        s[rows[s0:s1]] = F.one_hot(res[s0:s1], s.shape[1]).float()
        e = arr["edge_counts"][0]
        g = Graph((arr["src"][b * e:(b + 1) * e], arr["dst"][b * e:(b + 1) * e]), num_nodes=200)
        g.ndata["x"], g.edata["edge_attr"] = x, arr["edge_attr"][b * e:(b + 1) * e]
        graphs.append(g)
        seqs.append(s)
    return batch(graphs), torch.stack(seqs)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--variants", type=int, default=32768)
    ap.add_argument("--batch", type=int, default=512)
    ap.add_argument("--steps", type=int, default=2)
    ap.add_argument("--warmup", type=int, default=1)
    ap.add_argument("--out", default=None, help="also write the JSON line to this file")
    args = ap.parse_args()
    assert torch.cuda.is_available(), "needs a CUDA device"
    dev = torch.device("cuda:0")
    st, wu = args.steps, args.warmup
    out = {"precision": I.get_precision(), "card": card()}
    cols = torch.arange(20)

    # ---- HybridModelv2 on 8 templates, a library of --variants variants ----
    torch.manual_seed(1)
    model = I.model_map["HybridModelv2"](vae_input_dim=5943, device=dev).to(dev).eval()
    arr, seq_h, prop_h = inputs(8, 1)
    g = GraphBatch.from_arrays(*(arr[k].to(dev) for k in KEYS), max_nodes=200).validate()
    seq, prop = seq_h.to(dev), prop_h.to(dev)
    sample, offsets, rows, res = library(args.variants, 8, 2)
    tab = [t.to(dev) for t in (sample, offsets, rows, rows, res)]
    h = {"workload": f"HybridModelv2, 8 templates, {args.variants} variants of 1..{SITES} substitutions"}
    for k in (1, 16):
        h[f"ms_score_variants_K{k}"] = fastest_ms(lambda: score_variants(model, g, seq, prop, *tab, seq_columns=cols,
                                                                         samples=k), st, wu)

    def loop():
        with torch.no_grad():
            for lo in range(0, args.variants, HAND_CHUNK):
                hi = min(lo + HAND_CHUNK, args.variants)
                gb, s = hand_built(arr, seq_h, sample, offsets, rows, res, lo, hi)
                model(gb.to(dev), s.to(dev), prop_h[sample[lo:hi]].to(dev))

    h["ms_hand_built"] = fastest_ms(loop, 1, 1)
    h["speedup_over_hand_built"] = h["ms_hand_built"] / h["ms_score_variants_K1"]
    h["us_per_variant_K1"] = 1e3 * h["ms_score_variants_K1"] / args.variants

    # ---- is_variant_expand and the collation alone, one pass of 4096 variants ----
    r = 4096
    sp, op = tab[0][:r].contiguous(), tab[1][:r + 1].contiguous()
    nv, ev = g.batch_num_nodes()[sp], g.batch_num_edges()[sp]
    zero = torch.zeros(1, dtype=torch.int64, device=dev)
    node_out, edge_out = torch.cat([zero, nv.cumsum(0)]), torch.cat([zero, ev.cumsum(0)])
    n_p, e_p = int(node_out[-1]), int(edge_out[-1])
    L, V = seq.shape[1], seq.shape[2]
    xo, eao = torch.empty(n_p, 23, device=dev), torch.empty(e_p, 1, device=dev)
    so, do = torch.empty(e_p, dtype=torch.int64, device=dev), torch.empty(e_p, dtype=torch.int64, device=dev)
    sq = torch.empty(r, L, V, device=dev)
    flag = torch.zeros(1, dtype=torch.int32, device=dev)
    cold = cols.to(dev)
    expand = lambda: _C.variant_expand(g.ndata["x"], g.node_off, g.edge_off, g._src_local, g._dst_local, g.edata["edge_attr"],
                                       seq, sp, op, tab[2], tab[3], tab[4], cold, node_out, edge_out, xo, so, do, eao, sq, flag)
    k_ms = fastest_ms(expand, 50, 5)
    assert int(flag) == 0

    def collate():
        gp = GraphBatch(xo, so, do, eao, nv, ev, max_nodes=200, collate_now=False)
        gp._collate()

    c_ms = fastest_ms(collate, 50, 5)
    pass_ms = h["ms_score_variants_K1"] * r / args.variants
    e = {"variants": r, "us": 1e3 * k_ms, "bytes": 4 * (n_p * 23 + e_p + r * L * V) + 16 * e_p}
    e["bytes_per_s"] = e["bytes"] / (k_ms * 1e-3)
    e["share_of_hbm_peak"] = e["bytes_per_s"] / HBM_PEAK
    h["is_variant_expand"] = e
    h["us_collation_of_a_pass"] = 1e3 * c_ms
    h["expand_plus_collation_share_of_a_pass"] = (k_ms + c_ms) / pass_ms
    out["library"] = h

    # ---- score_variants against mutational_scan on the same single-site set ----
    b = args.batch
    arr, seq_h, prop_h = inputs(b, 3)
    g = GraphBatch.from_arrays(*(arr[k].to(dev) for k in KEYS), max_nodes=200).validate()
    seq, prop = seq_h.to(dev), prop_h.to(dev)
    ni = torch.arange(SITES).repeat(b, 1)
    n_var = SITES * 20 * b
    p = torch.arange(SITES).repeat_interleave(20 * b)
    c = torch.arange(20).repeat_interleave(b).repeat(SITES)
    single = [torch.arange(b).repeat(SITES * 20), torch.arange(n_var + 1), p, p, c]
    single = [t.to(dev) for t in single]
    s = {"workload": f"HybridModelv2, batch {b}, {SITES} sites x 20 residues = {n_var} single-site variants"}
    s["ms_mutational_scan"] = fastest_ms(lambda: mutational_scan(model, g, seq, prop, ni, ni, seq_columns=cols), st, wu)
    s["ms_score_variants"] = fastest_ms(lambda: score_variants(model, g, seq, prop, *single, seq_columns=cols,
                                                               max_graphs=(4096 // b) * b), st, wu)
    s["score_variants_over_scan"] = s["ms_score_variants"] / s["ms_mutational_scan"]
    out["single_site"] = s

    line = json.dumps(out)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
