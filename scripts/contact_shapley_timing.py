"""Cost of Shapley values of contacts (immunostruct_b200/shapley.py, ``contact_shapley``), on one GPU.

Workloads, HybridModelv2 in the default precision mode with the inputs resident on the device, batches of 200-node
10-NN graphs with 10 padded rows, every contact of the peptide interface (rows 0..8) a player:
  ``contact_shapley`` on --batch samples at T = 16 and T = 64, K = 1.
  ``occlude_contacts`` over the same selection, for the cost per variant.
  The plan, one 4 096-variant expansion pass and the reduction of the T = 64 call alone, and their share of it.
  A host-written baseline of the T = 16 call: per 512 variants, torch indexing builds the edge-masked coalition batch
    from the same plan (rows gathered, a boolean edge mask), then a ``GraphBatch`` and one ``predictive`` call.
Times are the fastest of three CUDA-event windows of --steps calls each, after --warmup calls.  The card's name and
power limit are read in the same run.  Prints one JSON line (and, with --out FILE, writes it there).

    python scripts/contact_shapley_timing.py [--batch 64] [--steps 2] [--warmup 1] [--out FILE]
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
from immunostruct_b200.occlusion import occlude_contacts  # noqa: E402
from immunostruct_b200.predictive import predictive  # noqa: E402
from immunostruct_b200.shapley import _edge_plan, _edge_sizes, _plan, contact_shapley  # noqa: E402
from immunostruct_b200.synthetic import synthetic_dense, synthetic_graph_arrays  # noqa: E402

sys.path.insert(0, os.path.join(ROOT, "scripts"))
from variant_timing import KEYS, card, fastest_ms  # noqa: E402

N, PAD, PEPTIDE = 200, 10, 9
CHUNK = 512


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=64)
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
    eps = torch.randn(1, b, 32, generator=torch.Generator().manual_seed(2)).to(dev)
    sel = torch.zeros(b, N, dtype=torch.bool, device=dev)
    sel[:, :PEPTIDE] = True
    sel = sel.reshape(-1)

    sizes = _edge_sizes(g, sel, 2)[0]
    count = sizes[1]
    q = int(count.sum())
    r = {"workload": f"HybridModelv2, batch {b} of {N}-node graphs, every contact of rows 0..{PEPTIDE - 1} a player, "
                     f"K = 1", "players": q, "players_per_sample_min_max": [int(count.min()), int(count.max())]}
    for t in (16, 64):
        call = lambda: contact_shapley(model, g, seq, prop, sel, permutations=t, seed=5, eps=eps)
        v = int((1 + t * (count - 1)).sum())
        ms = fastest_ms(call, st, wu)
        res = call()
        r[f"T{t}"] = {"variants": v, "ms": ms, "us_per_variant": 1e3 * ms / v,
                      "max_abs_gap_logit": float(res.gap_logit.abs().max())}
    occ_ms = fastest_ms(lambda: occlude_contacts(model, g, seq, prop, nodes=sel, eps=eps), st, wu)
    r["occlude_contacts"] = {"variants": q, "ms": occ_ms, "us_per_variant": 1e3 * occ_ms / q}

    # ---- the kernels alone, on the T = 64 call's tables ----
    t = 64
    plan = _plan(g, _edge_sizes(g, sel, t)[0], t, 5, 4096, _edge_plan)
    ranks, kept, flag = torch.empty_like(plan["ranks"]), torch.empty_like(plan["kept"]), plan["flag"]
    src, dst = g._src_local.contiguous(), g._dst_local.contiguous()
    plan_ms = fastest_ms(lambda: _C.shapley_edge_plan(g.edge_off, plan["ids32"], plan["poff"], plan["voff"], 5, ranks,
                                                      kept, flag), 50, 5)
    rr = plan["passes"][0][1]
    n_p, e_p = plan["node_tot"][0], plan["edge_tot"][0]
    xo, eao = torch.empty(n_p, 23, device=dev), torch.empty(e_p, 1, device=dev)
    so, do = torch.empty(e_p, dtype=torch.int64, device=dev), torch.empty(e_p, dtype=torch.int64, device=dev)
    node_out, edge_out = plan["ncs"][:rr + 1].contiguous(), plan["ecs"][:rr + 1].contiguous()
    expand_ms = fastest_ms(lambda: _C.shapley_edge_expand(g.ndata["x"], g.node_off, g.edge_off, src, dst,
                                                          g.edata["edge_attr"], plan["ids32"], plan["ranks"],
                                                          plan["smp"][:rr], plan["row"][:rr], plan["thr"][:rr],
                                                          node_out, edge_out, xo, so, do, eao, flag), 50, 5)
    v = plan["smp"].numel()
    logits = torch.randn(v, 1, device=dev)
    base = torch.randn(b, 1, device=dev)
    phi, se, gap = (torch.empty(2, q, device=dev), torch.empty(2, q, device=dev), torch.empty(2, b, device=dev))
    reduce_ms = fastest_ms(lambda: _C.shapley_reduce(logits, base, plan["ranks"], plan["poff"], plan["voff"], phi, se, gap,
                                                     flag), 50, 5)
    assert int(flag) == 0
    call_ms = r["T64"]["ms"]
    n_pass = len(plan["passes"])
    r["kernels_T64"] = {"us_plan": 1e3 * plan_ms, "us_expand_4096_variant_pass": 1e3 * expand_ms,
                        "us_reduce": 1e3 * reduce_ms, "passes": n_pass,
                        "plan_share_of_call": plan_ms / call_ms, "reduce_share_of_call": reduce_ms / call_ms,
                        "expand_share_of_call": expand_ms * n_pass / call_ms}

    # ---- host-written baseline of the T = 16 call: torch-built edge-masked coalition batches scored by predictive ----
    t = 16
    plan = _plan(g, _edge_sizes(g, sel, t)[0], t, 5, 4096, _edge_plan)
    x3 = arr["x"].reshape(b, N, 23)
    e_per = int(arr["edge_counts"][0])
    assert bool((arr["edge_counts"] == e_per).all())
    src2, dst2, ea2 = arr["src"].reshape(b, e_per), arr["dst"].reshape(b, e_per), arr["edge_attr"].reshape(b, e_per)
    ids2 = plan["ids"].reshape(b, e_per)
    rk = plan["ranks"].reshape(-1, plan["ranks"].shape[-1]).long()
    smp, row, thr = plan["smp"], plan["row"], plan["thr"]
    v = smp.numel()

    def loop():
        with torch.no_grad():
            for lo in range(0, v, CHUNK):
                s, rw, j = smp[lo:lo + CHUNK], row[lo:lo + CHUNK], thr[lo:lo + CHUNK]
                m = s.numel()
                ids = ids2[s]
                keep = (ids < 0) | (torch.gather(rk[rw], 1, ids.clamp_min(0)) >= j[:, None])
                gb = GraphBatch(x3[s].reshape(-1, 23), src2[s][keep], dst2[s][keep], ea2[s][keep].unsqueeze(1),
                                torch.full((m,), N, dtype=torch.int64, device=dev), keep.sum(1), max_nodes=N)
                predictive(model, gb, seq[s], prop[s], eps=eps[:, s])

    hand_ms = fastest_ms(loop, 1, 1)
    r["host_built_T16"] = {"variants": v, "ms": hand_ms, "speedup_of_contact_shapley": hand_ms / r["T16"]["ms"]}
    out["contact_shapley"] = r

    line = json.dumps(out)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
