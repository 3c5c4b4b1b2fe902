"""Cost of the beam search over residue substitutions (immunostruct_b200/design.py: beam_search), on one GPU.

Workload, in the default precision mode with the inputs resident on the device (200-node 10-NN graphs, 10 padded rows):
HybridModelv2 on 8 templates, P = 9 sites (peptide rows 0..8), all 20 residues allowed, beam W = 8, T = 9 rounds:
180 + 8 x 1 440 = 11 700 slot copies of the 8-graph batch, 93 600 graphs.
  ``beam_search`` at K = 1 and K = 16; one full-width round (W P 20 = 1 440 copies), as the difference between T = 2
    and T = 1; ``is_design_select`` alone on the batch.
  The same search written as a host loop over ``score_variants``: per round, the candidates of every beam state are
    enumerated and deduplicated on the host, scored as one library on the same draws, read back and ranked on the host.
    The loop's final best objective is compared with the device search's.
Times are the fastest of three CUDA-event windows of --steps calls each, after --warmup calls.  The card's name and
power limit are read in the same run.  Prints one JSON line (and, with --out FILE, writes it there).

    python scripts/design_timing.py [--steps 2] [--warmup 1] [--out FILE]
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
from immunostruct_b200.design import beam_search, round_slots  # noqa: E402
from immunostruct_b200.graph import GraphBatch  # noqa: E402
from immunostruct_b200.mutagenesis import score_variants  # noqa: E402
from immunostruct_b200.predictive import predictive  # noqa: E402
from immunostruct_b200.synthetic import synthetic_dense, synthetic_graph_arrays  # noqa: E402

SITES, BEAM, ROUNDS, TEMPLATES = 9, 8, 9, 8
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


def host_loop(model, g, seq, prop, native, cols, eps):
    """The search as a host loop over score_variants -> best objective per sample after the last round."""
    b, P = native.shape
    base = predictive(model, g, seq, prop, eps=eps).prob_mean.tolist()
    key = lambda s: sum(d * 20 ** p for p, d in enumerate(s))
    beams = [[(tuple(native[i].tolist()), base[i])] for i in range(b)]
    for _ in range(ROUNDS):
        cand, sample, counts, flat = [], [], [], []
        for i in range(b):
            members = {s for s, _ in beams[i]}
            seen = set()
            for s, _ in beams[i]:
                for p in range(P):
                    for c in range(20):
                        if c == s[p]:
                            continue
                        n = s[:p] + (c,) + s[p + 1:]
                        if n not in members and n not in seen:
                            seen.add(n)
                            cand.append((i, n))
                            sample.append(i)
                            counts.append(P)
                            flat += n
        rows = torch.arange(P).repeat(len(cand))
        offsets = torch.cat([torch.zeros(1, dtype=torch.int64), torch.tensor(counts).cumsum(0)])
        tab = [t.to(seq.device) for t in (torch.tensor(sample), offsets, rows, rows, torch.tensor(flat))]
        scores = score_variants(model, g, seq, prop, *tab, seq_columns=cols, eps=eps).prob_mean.tolist()
        pools = [list(bm) for bm in beams]
        for (i, n), o in zip(cand, scores):
            pools[i].append((n, o))
        beams = [sorted(pl, key=lambda e: (-e[1], key(e[0])))[:BEAM] for pl in pools]
    return [bm[0][1] for bm in beams]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=2)
    ap.add_argument("--warmup", type=int, default=1)
    ap.add_argument("--out", default=None, help="also write the JSON line to this file")
    args = ap.parse_args()
    assert torch.cuda.is_available(), "needs a CUDA device"
    dev = torch.device("cuda:0")
    st, wu = args.steps, args.warmup
    out = {"precision": I.get_precision(), "card": card()}
    cols = torch.arange(20)
    torch.manual_seed(1)
    model = I.model_map["HybridModelv2"](vae_input_dim=5943, device=dev).to(dev).eval()
    arr, seq_h, prop_h = inputs(TEMPLATES, 1)
    g = GraphBatch.from_arrays(*(arr[k].to(dev) for k in KEYS), max_nodes=200).validate()
    seq, prop = seq_h.to(dev), prop_h.to(dev)
    ni = torch.arange(SITES).repeat(TEMPLATES, 1)
    graphs = TEMPLATES * sum(round_slots(SITES, BEAM, ROUNDS))
    h = {"workload": f"HybridModelv2, {TEMPLATES} templates, P = {SITES}, W = {BEAM}, T = {ROUNDS}: {graphs} graphs"}
    run = lambda **kw: beam_search(model, g, seq, prop, ni, ni, seq_columns=cols, beam=BEAM, **kw)
    for k in (1, 16):
        eps = torch.randn(k, TEMPLATES, 32, device=dev, generator=torch.Generator(dev).manual_seed(2))
        h[f"ms_beam_search_K{k}"] = fastest_ms(lambda: run(rounds=ROUNDS, eps=eps), st, wu)
    eps = torch.randn(1, TEMPLATES, 32, device=dev, generator=torch.Generator(dev).manual_seed(2))
    t1, t2 = (fastest_ms(lambda: run(rounds=t, eps=eps), st, wu) for t in (1, 2))
    h["ms_one_full_round"] = t2 - t1
    h["us_per_graph_K1"] = 1e3 * h["ms_beam_search_K1"] / graphs

    # is_design_select alone on the batch, one full-width round
    b, n = TEMPLATES, BEAM * SITES * 20
    res = run(rounds=2, eps=eps)
    keys = (res.states.clamp_min(0) * 20 ** torch.arange(SITES, device=dev)).sum(-1)
    beam = (res.states, keys, res.n_mutations, res.valid, res.logits, res.prob_mean, res.prob_std, res.objective)
    out_b = tuple(torch.empty_like(t) for t in beam)
    native = res.states[:, 0].clone()
    allowed = torch.ones(b, SITES, 20, dtype=torch.bool, device=dev)
    rl, rm, rs = torch.randn(n, b, 1, device=dev), torch.rand(n, b, device=dev), torch.zeros(n, b, device=dev)
    best = torch.empty(b, device=dev)
    h["us_design_select"] = 1e3 * fastest_ms(lambda: _C.design_select(beam, rl, rm, rs, native, allowed, ni.to(dev), BEAM,
                                                                       SITES, 0.0, True, out_b, best), 50, 5)

    # the same search as a host loop over score_variants
    native = arr["x"].reshape(TEMPLATES, 200, 23)[:, :SITES, :20].argmax(-1)
    with torch.no_grad():
        h["ms_host_loop_over_score_variants_K1"] = fastest_ms(lambda: host_loop(model, g, seq, prop, native, cols, eps),
                                                              1, 0)
        loop_best = host_loop(model, g, seq, prop, native, cols, eps)
    dev_best = run(rounds=ROUNDS, eps=eps).objective[:, 0].tolist()
    h["max_abs_diff_best_objective_vs_host_loop"] = max(abs(a - b_) for a, b_ in zip(loop_best, dev_best))
    h["speedup_over_host_loop"] = h["ms_host_loop_over_score_variants_K1"] / h["ms_beam_search_K1"]
    out["beam_search"] = h
    line = json.dumps(out)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
