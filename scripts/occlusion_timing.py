"""Cost of structural occlusion scans (immunostruct_b200/occlusion.py), on one GPU.

Workloads, HybridModelv2 in the default precision mode with the inputs resident on the device, batch 512 of 200-node
10-NN graphs with 10 padded rows (190 present residues per graph):
  ``occlude_residues`` over every present row (97 280 variants) at K = 1 and K = 16.
  ``occlude_contacts`` over the contacts of 9 "peptide" rows (graph-local rows 0..8) of every graph, at K = 1.
  The same residue scan by hand on the device: per 512 variants, torch indexing builds the occluded batch (rows gathered,
    the row zeroed, a boolean edge mask), then a ``GraphBatch`` and one ``model()`` call.
  is_occlusion_expand and the pass's collation alone, on the first 4 096-variant pass of the residue scan, and their
    share of that pass.  Bytes of the expansion = the written pass (x23 rows, kept edges: two int64 endpoints and one fp32
    attribute each); the base batch is read from L2.
Times are the fastest of three CUDA-event windows of --steps calls each, after --warmup calls.  The card's name and
power limit are read in the same run.  Prints one JSON line (and, with --out FILE, writes it there).

    python scripts/occlusion_timing.py [--batch 512] [--steps 2] [--warmup 1] [--out FILE]
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
from immunostruct_b200.graph import GraphBatch  # noqa: E402
from immunostruct_b200.occlusion import _residue_tables, occlude_contacts, occlude_residues  # noqa: E402
from immunostruct_b200.synthetic import synthetic_dense, synthetic_graph_arrays  # noqa: E402

sys.path.insert(0, os.path.join(ROOT, "scripts"))
from variant_timing import HBM_PEAK, KEYS, card, fastest_ms  # noqa: E402

N, PAD, PEPTIDE = 200, 10, 9
HAND_CHUNK = 512


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
    n_res = b * (N - PAD)
    peptide = (torch.arange(b * N, device=dev) % N) < PEPTIDE

    r = {"workload": f"HybridModelv2, batch {b} of {N}-node graphs, {N - PAD} present rows each: {n_res} residue variants"}
    for k in (1, 16):
        r[f"ms_occlude_residues_K{k}"] = fastest_ms(lambda: occlude_residues(model, g, seq, prop, samples=k), st, wu)
    r["us_per_variant_K1"] = 1e3 * r["ms_occlude_residues_K1"] / n_res
    con = occlude_contacts(model, g, seq, prop, nodes=peptide)
    n_con = int(con.sample.numel())
    r["contacts_of_9_peptide_rows"] = n_con
    r["ms_occlude_contacts_K1"] = fastest_ms(lambda: occlude_contacts(model, g, seq, prop, nodes=peptide), st, wu)
    r["us_per_contact_variant_K1"] = 1e3 * r["ms_occlude_contacts_K1"] / n_con

    # ---- the residue scan by hand: torch indexing per 512 variants, GraphBatch, model() ----
    e_per = int(arr["edge_counts"][0])
    x3 = arr["x"].reshape(b, N, 23)
    src2, dst2, ea2 = arr["src"].reshape(b, e_per), arr["dst"].reshape(b, e_per), arr["edge_attr"].reshape(b, e_per)
    sample = torch.arange(b, device=dev).repeat_interleave(N - PAD)
    row = torch.arange(N - PAD, device=dev).repeat(b)

    def loop():
        with torch.no_grad():
            for lo in range(0, n_res, HAND_CHUNK):
                s, a = sample[lo:lo + HAND_CHUNK], row[lo:lo + HAND_CHUNK]
                m = s.numel()
                x = x3[s].clone()
                x[torch.arange(m, device=dev), a] = 0.0
                keep = (src2[s] != a[:, None]) & (dst2[s] != a[:, None])
                gb = GraphBatch(x.reshape(-1, 23), src2[s][keep], dst2[s][keep], ea2[s][keep].unsqueeze(1),
                                torch.full((m,), N, dtype=torch.int64, device=dev), keep.sum(1), max_nodes=N)
                model(gb, seq[s], prop[s])

    r["ms_hand_built"] = fastest_ms(loop, 1, 1)
    r["speedup_over_hand_built"] = r["ms_hand_built"] / r["ms_occlude_residues_K1"]

    # ---- is_occlusion_expand and the collation alone, the first 4096-variant pass ----
    tables = _residue_tables(g, None, 4096)[0]
    smp, na, nb, nv, kept, ncs, ecs, passes, node_tot, edge_tot, _ = tables
    j, rr = passes[0]
    n_p, e_p = node_tot[0], edge_tot[0]
    xo, eao = torch.empty(n_p, 23, device=dev), torch.empty(e_p, 1, device=dev)
    so, do = torch.empty(e_p, dtype=torch.int64, device=dev), torch.empty(e_p, dtype=torch.int64, device=dev)
    flag = torch.zeros(1, dtype=torch.int32, device=dev)
    node_out, edge_out = ncs[:rr + 1].contiguous(), ecs[:rr + 1].contiguous()
    expand = lambda: _C.occlusion_expand(g.ndata["x"], g.node_off, g.edge_off, g._src_local, g._dst_local,
                                         g.edata["edge_attr"], smp[:rr], na[:rr], nb[:rr], node_out, edge_out, xo, so, do,
                                         eao, flag)
    k_ms = fastest_ms(expand, 50, 5)
    assert int(flag) == 0

    def collate():
        gp = GraphBatch(xo, so, do, eao, nv[:rr], kept[:rr], max_nodes=N, collate_now=False)
        gp._collate()

    c_ms = fastest_ms(collate, 50, 5)
    pass_ms = r["ms_occlude_residues_K1"] * rr / n_res
    e = {"variants": rr, "us": 1e3 * k_ms, "bytes": 4 * n_p * 23 + 20 * e_p}
    e["bytes_per_s"] = e["bytes"] / (k_ms * 1e-3)
    e["share_of_hbm_peak"] = e["bytes_per_s"] / HBM_PEAK
    r["is_occlusion_expand"] = e
    r["us_collation_of_a_pass"] = 1e3 * c_ms
    r["expand_plus_collation_share_of_a_pass"] = (k_ms + c_ms) / pass_ms
    out["occlusion"] = r

    line = json.dumps(out)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
