"""Cost of nearest neighbours in the classifier's feature space (immunostruct_b200/neighbors.py), on one GPU.

Workloads, HybridModelv2 in the default precision mode with scaled-up weights (latent mean x 3, classifier input layer x 4,
as in tests/test_neighbors_gpu.py), inputs resident on the device:
  ``embed`` of --bank graphs (200-node 10-NN graphs with 10 padded rows, batches of 512 and the tail batch), against the
    eval forward ``model(...)`` of the same batches.  Its features are the bank (D = 32).
  ``nearest`` leave-self-out of the bank against itself (exclude = arange), k = 16: the deep k-NN out-of-distribution
    scan of a training set.
  ``nearest`` of --queries queries (bank rows plus 5 % noise) against the bank, k = 16.
  Baselines on the same inputs, chunked by 4 096 queries (the full Q x R matrix of the query scan is 28 GB):
    exact: ``torch.cdist(..., compute_mode="donot_use_mm_for_euclid_dist")`` squared + ``topk``, the same metric;
    matmul: ``torch.cdist`` in its default mode (|q|^2 + |r|^2 - 2 q.r through a GEMM) squared + ``topk``.
  Agreement with each baseline: the queries whose index set differs, and of those the ones at an fp32 near-tie (the fp64
    distances of the k-th neighbour of both sets within 2 (D + 4) 2^-24 relative).
The arithmetic floor of a search is Q R D (FADD + FFMA) fp32 instructions; it is printed with the rate it implies.
Times are the fastest of three CUDA-event windows of --steps calls each, after --warmup calls.  The card's name and
power limit are read in the same run.  Prints one JSON line (and, with --out FILE, writes it there).

    python scripts/neighbors_timing.py [--bank 27000] [--queries 262144] [--steps 3] [--warmup 1] [--out FILE]
"""
import argparse
import json
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import immunostruct_b200 as I  # noqa: E402
from immunostruct_b200.graph import GraphBatch  # noqa: E402
from immunostruct_b200.neighbors import embed, nearest  # noqa: E402
from immunostruct_b200.synthetic import synthetic_dense, synthetic_graph_arrays  # noqa: E402

sys.path.insert(0, os.path.join(ROOT, "scripts"))
from variant_timing import KEYS, card, fastest_ms  # noqa: E402

K, BATCH, CHUNK = 16, 512, 4096


def _model(dev):
    torch.manual_seed(0)
    model = I.model_map["HybridModelv2"](vae_input_dim=5943, device=dev).to(dev)
    with torch.no_grad():
        for name, p in model.named_parameters():
            if name in ("vae_fc21.weight", "vae_fc21.bias"):
                p.mul_(3.0)
            if name == "classifier.1.weight":
                p.mul_(4.0)
    I.invalidate_caches()
    return model.eval()


def _batches(n, dev):
    out = []
    for i, s in enumerate(range(0, n, BATCH)):
        b = min(BATCH, n - s)
        arr = synthetic_graph_arrays(b, 200, 10, seed=100 + i, n_pad=10)
        dense = synthetic_dense(b, seed=100 + i)
        g = GraphBatch.from_arrays(*(arr[k] for k in KEYS), max_nodes=200).to(dev)
        out.append((g, dense["seq"].to(dev), dense["prop"].to(dev)))
    return out


def _torch_knn(query, bank, k, exact, exclude=None):
    idx, dist = [], []
    mode = "donot_use_mm_for_euclid_dist" if exact else "use_mm_for_euclid_dist_if_necessary"
    for s in range(0, query.shape[0], CHUNK):
        d = torch.cdist(query[s:s + CHUNK], bank, compute_mode=mode).square_()
        if exclude is not None:
            d.scatter_(1, exclude[s:s + CHUNK, None], float("inf"))
        v, i = torch.topk(d, k, dim=1, largest=False)
        idx.append(i)
        dist.append(v)
    return torch.cat(idx), torch.cat(dist)


def _agreement(query, bank, idx, ref_idx):
    """Queries whose index set differs from the reference's, and how many of those are fp32 near-ties."""
    a, b = idx.sort(1).values, ref_idx.sort(1).values
    diff = (a != b).any(1).nonzero().flatten()
    ties = 0
    if diff.numel():
        q = query[diff].double()
        kth = [((q[:, None, :] - bank.double()[x[diff]]) ** 2).sum(-1).max(1).values for x in (idx, ref_idx)]
        bound = 2 * (query.shape[1] + 4) * 2.0 ** -24 * torch.maximum(kth[0], kth[1])
        ties = int(((kth[0] - kth[1]).abs() <= bound).sum())
    return {"queries_differing": int(diff.numel()), "of_which_fp32_near_ties": ties}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--bank", type=int, default=27000)
    ap.add_argument("--queries", type=int, default=262144)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=1)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("neighbors_timing.py measures the GPU path and needs a CUDA device")
    dev = torch.device("cuda:0")
    res = {"card": card(), "precision": I.get_precision(), "bank": args.bank, "queries": args.queries, "k": K}

    model = _model(dev)
    batches = _batches(args.bank, dev)

    def run_embed():
        return torch.cat([embed(model, *b) for b in batches])

    def run_forward():
        with torch.no_grad():
            for b in batches:
                model(*b)

    res["embed_ms"] = fastest_ms(run_embed, args.steps, args.warmup)
    res["eval_forward_ms"] = fastest_ms(run_forward, args.steps, args.warmup)
    bank = run_embed()
    d = bank.shape[1]
    g = torch.Generator(device=dev).manual_seed(1)
    pick = torch.randint(0, args.bank, (args.queries,), generator=g, device=dev)
    query = (bank[pick] + 0.05 * bank.std(0) * torch.randn(args.queries, d, generator=g, device=dev)).contiguous()
    self_ex = torch.arange(args.bank, device=dev)

    for name, q, ex in (("self_search", bank, self_ex), ("query_search", query, None)):
        flops = 2.0 * q.shape[0] * args.bank * d
        fused = nearest(q, bank, K, exclude=ex)
        exact = _torch_knn(q, bank, K, True, ex)
        mm = _torch_knn(q, bank, K, False, ex)
        row = {"fused_ms": fastest_ms(lambda: nearest(q, bank, K, exclude=ex), args.steps, args.warmup),
               "torch_exact_ms": fastest_ms(lambda: _torch_knn(q, bank, K, True, ex), args.steps, args.warmup),
               "torch_matmul_ms": fastest_ms(lambda: _torch_knn(q, bank, K, False, ex), args.steps, args.warmup),
               "fp32_instructions": flops,
               "vs_exact": _agreement(q, bank, fused.index, exact[0]),
               "matmul_vs_exact": _agreement(q, bank, mm[0], exact[0])}
        row["fused_fp32_instr_per_s"] = flops / (row["fused_ms"] * 1e-3)
        res[name] = row
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
