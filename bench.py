#!/usr/bin/env python
"""Headline benchmark: pMHC graphs/s of the ImmunoStruct hot path on B200.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--dump-outputs DIR]

Workload (BASELINE.json configs[1]): HybridModelv2 inference (eval, no_grad) over synthetic pMHC
graphs of the named shape (200 residues, directed 10-NN contacts, 283x21 sequence one-hots), batch
512 per GPU, fp32.  A "step" is one pass of the hot path over one batch of 512 graphs: on-device
collation (CSR + CSC + segment offsets) -> 6 EGNN layers -> per-graph attention + mean pool -> VAE
and property branches -> fusion attention -> classifier -> sigmoid.
  * ``value``  : graphs/s with inputs resident in HBM (a pool of batches larger than L2 is cycled);
  * ``e2e``    : same metric through the public API from pinned HOST buffers (GraphBatch.to(device),
                 model(...), probabilities copied back) -- H2D and D2H inside the timed region;
  * ``train``  : fwd + bwd + Adam step (BCE_loss with sequence loss) at the same batch per GPU, with
                 the NCCL gradient all-reduce when N > 1 (weak scaling);
  * ``train_comparative``: BASELINE configs[2] -- one cancer fine-tune step (HybridModelv2_Comparative, 256 cancer /
                 wild-type pairs, paired contrastive loss, AdamW) at N = 1;
  * ``roofline``: the dominant kernel (EGNN edge forward) timed alone with CUDA events;
  * ``cpu_baseline``: the CPU oracle port of the same forward on this box's host cores (bounded sample).
``--impl reference`` times the reference's CPU path (oracle port; the reference is pure Python +
dgl/torch_geometric and cannot travel to this box) with all host threads on the same metric.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

BATCH = 512
N_NODES, KNN = 200, 10
VAE_IN = 5943
POOL = 8                    # resident input batches cycled through (8 x 42 MB > 126 MB of L2)
FLOP_PER_EDGE_EDGE_KERNEL = 2 * 64 * 64 * 2 + 2 * 64      # two 64x64 per-edge GEMMs + the w4 dot
# algorithmic (compulsory, each byte once) traffic of one edge-forward launch -- DESIGN.md 4.2:
BYTES_PER_NODE_EDGE_KERNEL = 512 + 12 + 4 + 256 + 12       # read PQ row, x, indptr ; write hn row, x'
BYTES_PER_EDGE_EDGE_KERNEL = 3 * 4 + 4                     # read csr_src/dst/eid + edge_attr
GATHER_BYTES_PER_EDGE = 2 * 256                            # P[src] + Q[dst] rows (served by L2)
# ncu counters of the dominant kernel (DRAM bytes per launch, pipe utilisation) are read from a committed capture
# summary, profiles/ncu_edge_fwd.json (written by scripts/ncu_to_json.py from an `ncu --set full` report; it records
# the commit and date of the capture) -- never hard-coded here.
def ncu_record(precision):
    path = os.path.join(ROOT, "profiles", "ncu_edge_fwd.json")
    if not os.path.exists(path):
        return None
    rec = json.load(open(path))
    k = rec.get("kernels", {}).get(precision)
    if k is None:
        return None
    return dict(k, source={"file": "profiles/ncu_edge_fwd.json", "commit": rec.get("commit"), "captured": rec.get("captured"),
                           "batch": rec.get("batch")})


FP32_PEAK_TFLOPS = 148 * 128 * 2 * 1.965e9 / 1e12          # 74.4


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--batch", type=int, default=BATCH)
    ap.add_argument("--precision", default="fp16x2", choices=["fp32", "bf16x3", "fp16x2", "tf32x3", "bf16"],
                    help="EGNN GEMM arithmetic of the headline run; default = the package default: fp16x2 (fp16 hi / lo operand "
                         "pairs in the no-grad forward, bf16x3 in training); fp16x2 / bf16x3 / tf32x3 = fp32-accurate tensor cores")
    ap.add_argument("--profile", action="store_true",
                    help="bracket the timed inference region with cudaProfilerStart/Stop (ncu --profile-from-start off)")
    ap.add_argument("--no-train", action="store_true")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the last timed inference step returned (probabilities and the model's recon, mu, "
                         "logvar, logits) as DIR/<name>.npy, float32, rank 0; inputs are seeded, so two builds can be "
                         "compared output for output")
    return ap.parse_args()


DUMP_LIMIT = 64 * 10 ** 6           # bytes of all dumped arrays together


def dump_outputs(path, tensors):
    """Write each tensor as <path>/<name>.npy (float32).  If they exceed DUMP_LIMIT together, the largest is cut to
    a fixed, seeded sample of its rows (the same rows in every run with the same arguments)."""
    import numpy as np
    arrays = {k: v.detach().float().cpu().numpy() for k, v in tensors.items()}
    big = max(arrays, key=lambda k: arrays[k].nbytes)
    rest = sum(a.nbytes for k, a in arrays.items() if k != big)
    a = arrays[big]
    rows = (DUMP_LIMIT - rest - 4096 * len(arrays)) // max(1, a[0].nbytes)
    if rows < 0:
        raise ValueError(f"--dump-outputs: the arrays other than {big} alone exceed {DUMP_LIMIT} bytes")
    if rows < a.shape[0]:
        idx = np.sort(np.random.default_rng(0).choice(a.shape[0], rows, replace=False))
        arrays[big] = a[idx]
    os.makedirs(path, exist_ok=True)
    for k, a in arrays.items():
        np.save(os.path.join(path, k + ".npy"), a)


def measured_peaks():
    """(HBM GB/s, dense bf16 TFLOP/s burst, source) from the driver-written MEASURED_PEAKS.json."""
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return float(d["hbm_gbs"]), float(d["bf16_tflops"]), "measured"
    return 6650.0, 1590.0, "fallback"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled during the timed region (B200_PROFILING.md)."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.proc, self.lines = index, None, []

    def __enter__(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "50"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=lambda: [self.lines.append(l) for l in self.proc.stdout], daemon=True)
            self.t.start()
        except Exception:
            self.proc = None
        return self

    def __exit__(self, *a):
        if self.proc:
            time.sleep(0.15)
            self.proc.terminate()
            self.t.join(2)

    def summary(self):
        sm, mx, reasons = [], [], set()
        for l in self.lines:
            f = [x.strip() for x in l.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        return {"sm_mhz": statistics.median(sm), "sm_max_mhz": max(mx), "reasons": sorted(reasons), "samples": len(sm)}


# --------------------------------------------------------------------------------------------------
def make_pool(batch, n_batches, seed, device):
    from immunostruct_b200.synthetic import synthetic_dense, synthetic_graph_arrays
    pool = []
    for i in range(n_batches):
        arr = synthetic_graph_arrays(batch, N_NODES, KNN, seed=seed + 31 * i, device=device)
        dense = synthetic_dense(batch, seed=seed + 31 * i, device=device)
        pool.append((arr, dense))
    return pool


def oracle_inference(params, arr, dense, eps):
    from immunostruct_b200.synthetic import split_graphs
    from oracle import reference_ops as R
    with torch.no_grad():
        g = R.dgl_batch(split_graphs(arr))
        out = R.hybrid_forward(params, g, dense["seq"], dense["prop"], eps)
        return torch.sigmoid(out[3]).squeeze()


def oracle_train_step(params, arr, dense, eps, pos_weight=4.25):
    """fwd + bwd of the CPU oracle: HybridModelv2, BCE_loss(sequence=True) (BASELINE configs[0])."""
    from immunostruct_b200.synthetic import split_graphs
    from oracle import reference_ops as R
    for p in params.values():
        p.grad = None
    g = R.dgl_batch(split_graphs(arr))
    recon, mu, logvar, out = R.hybrid_forward(params, g, dense["seq"], dense["prop"], eps)
    loss = R.bce_loss(recon, dense["seq"], mu, logvar, out, dense["target"], pos_weight)
    loss.backward()
    return loss


class ReferenceCPU:
    """The reference's CPU implementation of the path: its own model code (through oracle/shim.py) when a reference
    tree is present (/root/reference, or baseline/_ref written by oracle/install_ref.py), else the oracle port."""

    def __init__(self):
        from oracle import shim
        import immunostruct_b200 as I
        torch.manual_seed(1)
        state = I.model_map["HybridModelv2"](vae_input_dim=VAE_IN, device="cpu").state_dict()
        self.kind, self.shim = "port", shim
        if shim.reference_available():
            try:
                model_map, self.Losses, _ = shim.load_reference()
                self.model = model_map["HybridModelv2"](vae_input_dim=VAE_IN, device="cpu")
                self.model.load_state_dict(state)
                self.kind = "reference"
            except Exception as exc:                     # fall back to the port, say why
                print("reference tree present but not loadable:", repr(exc), file=sys.stderr)
        self.params = {k: v.detach().clone() for k, v in state.items()}

    def graph(self, arr):
        from immunostruct_b200.synthetic import split_graphs
        from oracle import reference_ops as R
        return self.shim.graph_from_dict(R.dgl_batch(split_graphs(arr)))

    def infer(self, arr, dense, eps):
        if self.kind == "port":
            return oracle_inference(self.params, arr, dense, eps)
        self.model.eval()
        with torch.no_grad():                            # procedures/infer.py:14-22
            out = self.model(self.graph(arr), dense["seq"], dense["prop"])[3]
            return torch.sigmoid(out).squeeze()

    def train_step(self, arr, dense, eps):
        if self.kind == "port":
            params = {k: v.requires_grad_(True) for k, v in self.params.items()}
            return oracle_train_step(params, arr, dense, eps)
        self.model.train()                               # procedures/train.py:23-27 (no optimizer step: fwd + bwd)
        self.model.zero_grad()
        recon, mu, logvar, out = self.model(self.graph(arr), dense["seq"], dense["prop"])
        loss = self.Losses(VAE_IN, [4.25, 1.0], sequence=True).BCE_loss(recon, dense["seq"], mu, logvar, out, dense["target"])
        loss.backward()
        return loss

    def describe(self):
        return ("the reference's own models/hybrid_models.py HybridModelv2 through oracle/shim.py (stand-ins for dgl / "
                "torch_geometric only)" if self.kind == "reference" else "oracle/reference_ops.py hybrid_forward (port)")


WORKLOAD = ("IEDB HybridModelv2 inference, batch 512 per GPU, 200-node 10-NN graphs, 283x21 sequence, fp32 "
            "(BASELINE configs[1])")


def cpu_reference_arm(args):
    """The reference's CPU implementation of the path, all host threads, SAME workload: every step is one 512-graph
    batch (about 1.5 s on 16 cores, so the default K = 20, W = 3 run ends in well under a minute)."""
    torch.set_num_threads(os.cpu_count() or 1)
    ref = ReferenceCPU()
    B = args.batch
    pool = make_pool(B, 2, seed=1, device="cpu")
    eps = torch.randn(B, 32)
    for i in range(args.warmup):
        ref.infer(*pool[i % 2], eps)
    t0 = time.perf_counter()
    for i in range(args.steps):
        ref.infer(*pool[i % 2], eps)
    dt = time.perf_counter() - t0
    v = B * args.steps / dt
    cores = torch.get_num_threads()
    print(json.dumps({
        "impl": "reference", "metric": "pMHC graphs/sec (HybridModelv2 inference, fp32)", "value": v,
        "unit": "graphs/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": dt / args.steps * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic",
        "config": {"workload": WORKLOAD, "batch_per_gpu": B, "nodes_per_graph": N_NODES, "edges_per_graph": N_NODES * KNN,
                   "parallelism": "cpu"},
        "cpu_baseline": {"value": v, "unit": "graphs/s", "cores": cores, "kind": ref.kind,
                         "sample": f"{args.steps} x {B}-graph batches, {ref.describe()}, torch CPU fp32"},
        "e2e": {"value": v, "unit": "graphs/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }))


def main():
    args = parse()
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        if rank == 0:
            cpu_reference_arm(args)
        return
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (no CPU fallback); use --impl reference for the CPU arm")

    import torch.distributed as dist
    import immunostruct_b200 as I
    from immunostruct_b200 import _C
    from immunostruct_b200.distributed import GradientAllReducer, broadcast_parameters
    from immunostruct_b200.graph import GraphBatch

    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    B, K, W = args.batch, args.steps, args.warmup

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(ms):
        if world == 1:
            return ms
        t = torch.tensor([ms], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t)

    I.set_precision(args.precision)
    torch.manual_seed(1)
    model = I.model_map["HybridModelv2"](vae_input_dim=VAE_IN, device=dev).to(dev)
    broadcast_parameters(model)
    pool = make_pool(B, POOL, seed=1 + 1000 * rank, device=dev)
    keys = ("x", "src", "dst", "edge_attr", "node_counts", "edge_counts")
    last = {}                                      # model outputs of the latest inference step (for --dump-outputs)

    def infer_step(arr, dense):
        gb = GraphBatch.from_arrays(*(arr[k] for k in keys), max_nodes=N_NODES)
        last["outputs"] = model(gb, dense["seq"], dense["prop"])
        return torch.sigmoid(last["outputs"][3]).squeeze()

    # ---- device-resident inference throughput (the headline `value`) ---------------------------
    model.eval()
    launches0 = None
    # clocks / throttle reasons are sampled from before the warm-up until the end of the end-to-end loops: the timed
    # region alone (K x 2.2 ms) can be shorter than nvidia-smi's sampling period, the whole stretch runs the same kernels
    clk = ClockSampler(local)
    clk.__enter__()
    time.sleep(0.3)                               # nvidia-smi start-up: the first sample must not miss the load
    with torch.no_grad():
        for i in range(20):                       # lead-in under the clock sampler (untimed, before the W warm-up steps)
            infer_step(*pool[i % POOL])
        for i in range(W):
            infer_step(*pool[i % POOL])
        barrier()
        launches0 = _C.LAUNCHES
        if args.profile:
            torch.cuda.profiler.start()
        # EXACTLY K steps per window, barrier + synchronize on both sides, max over ranks; three back-to-back windows
        # and the fastest one is reported (as in run_training: a 2.2 ms step is ~24 launches, and a busy host core on the
        # shared box can starve the queue for a whole 20-step window; all three are kept in ms_per_step_windows)
        infer_windows = []
        for w_ in range(1 if args.profile else 3):
            barrier()
            if w_ == 0:
                launches0 = _C.LAUNCHES
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for i in range(K):
                probs = infer_step(*pool[i % POOL])
            e1.record()
            barrier()
            if w_ == 0:
                launches = _C.LAUNCHES - launches0
            infer_windows.append(max_over_ranks(e0.elapsed_time(e1)))
        if args.profile:
            torch.cuda.profiler.stop()
        ms = min(infer_windows)
    value = world * B * K / (ms / 1e3)
    if args.dump_outputs and rank == 0:
        recon, mu, logvar, logits = last["outputs"]
        dump_outputs(args.dump_outputs, {"probs": probs, "recon": recon, "mu": mu, "logvar": logvar, "logits": logits})

    # ---- BASELINE configs[1], literally: a scan of 27 000 graphs = 52 full batches of 512 + one of 376 (the last,
    # partial batch of the reference's no-drop_last loader, procedures/infer.py:14-31); per rank at N > 1 ------------
    scan = None
    if B == BATCH:
        n_scan, tail = 27000, 27000 % BATCH
        tail_arr = {k: (v[:tail * N_NODES] if k in ("x",) else v[:tail * N_NODES * KNN] if k in ("src", "dst", "edge_attr")
                        else v[:tail]) for k, v in pool[1][0].items()}
        tail_dense = {k: v[:tail] for k, v in pool[1][1].items()}
        with torch.no_grad():
            infer_step(tail_arr, tail_dense)                     # warm the 376-graph shapes
            barrier()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for i in range(n_scan // BATCH):
                infer_step(*pool[i % POOL])
            p_tail = infer_step(tail_arr, tail_dense)
            e1.record()
            barrier()
            ms_scan = max_over_ranks(e0.elapsed_time(e1))
        scan = {"graphs": n_scan, "batches": n_scan // BATCH + 1, "tail_batch": tail, "ms": ms_scan,
                "value": world * n_scan / (ms_scan / 1e3), "unit": "graphs/s", "tail_outputs": int(p_tail.numel())}

    # ---- end to end from pinned host buffers through the public API -----------------------------
    host = []
    for arr, dense in pool[:4]:
        gbh = GraphBatch.from_arrays(*(arr[k].cpu() for k in keys), max_nodes=N_NODES).pin_memory()
        host.append((gbh, dense["seq"].cpu().pin_memory(), dense["prop"].cpu().pin_memory()))
    h2d = sum(t.numel() * t.element_size() for t in (host[0][0].ndata["x"], host[0][0]._src_local, host[0][0]._dst_local,
                                                     host[0][0].edata["edge_attr"], host[0][0]._node_counts,
                                                     host[0][0]._edge_counts, host[0][1], host[0][2]))
    out_host = torch.empty(B, pin_memory=True)

    def e2e_consume(item):
        gb, seq, prop = item                      # already resident: .to(dev) below is a no-op, as in the
        gb = gb.to(dev)                           # reference loop's `graph_data.to(device)` (procedures/infer.py:16)
        out = model(gb, seq.to(dev), prop.to(dev))[3]
        out_host.copy_(torch.sigmoid(out).squeeze(), non_blocking=True)

    def host_batches(n):
        for i in range(n):
            yield host[i % 4]

    with torch.no_grad():
        for item in I.DevicePrefetcher(host_batches(W), dev):
            e2e_consume(item)
        e2e_windows = []
        for w_ in range(3):                                           # fastest of three K-step windows, as above
            barrier()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for item in I.DevicePrefetcher(host_batches(K), dev):     # H2D of every batch is inside the timed region
                e2e_consume(item)
            e1.record()
            barrier()
            e2e_windows.append(max_over_ranks(e0.elapsed_time(e1)))
        ms_e2e = min(e2e_windows)
    e2e_value = world * B * K / (ms_e2e / 1e3)

    # ---- same, from the compact host format (1 byte per residue / sequence position, int32 edges): the H2D copy
    # shrinks 4.4x and csrc/unpack.cu expands bit-exactly on the device (SURVEY 8(f) row 1) ----------------------
    packed = [(I.pack_graph_batch(gbh).pin_memory(), I.pack_sequence(seq.reshape(B, -1, 21)).pin_memory(), prop)
              for gbh, seq, prop in host]
    h2d_packed = packed[0][0].nbytes + packed[0][1].nbytes + packed[0][2].numel() * 4

    def packed_batches(n):
        for i in range(n):
            yield packed[i % 4]

    with torch.no_grad():
        for item in I.DevicePrefetcher(packed_batches(W), dev):
            e2e_consume(item)
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for item in I.DevicePrefetcher(packed_batches(K), dev):
            e2e_consume(item)
        e1.record()
        barrier()
        ms_e2e_packed = max_over_ranks(e0.elapsed_time(e1))
    clk.__exit__()

    # ---- the same device-resident step in the other arithmetic modes (short runs) -----------------
    other = {}
    with torch.no_grad():
        for prec in ("fp32", "bf16x3", "fp16x2", "tf32x3", "bf16"):
            if prec == args.precision:
                continue
            I.set_precision(prec)
            for i in range(W):
                infer_step(*pool[i % POOL])
            barrier()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for i in range(K):
                infer_step(*pool[i % POOL])
            e1.record()
            barrier()
            ms_o = max_over_ranks(e0.elapsed_time(e1))
            other[prec] = {"value": world * B * K / (ms_o / 1e3), "unit": "graphs/s", "ms_per_step": ms_o / K}
    I.set_precision(args.precision)

    # ---- training step: fwd + bwd + Adam (+ NCCL gradient all-reduce) ---------------------------
    # Optimiser: immunostruct_b200.FusedAdam (one kernel over the flat parameter buffer, csrc/optim.cu); gradients
    # live in one flat buffer that distributed.BucketedGradientReducer all-reduces bucket by bucket DURING backward.
    train = None
    if not args.no_train:
        losses = I.Losses(VAE_IN, [0.81, 0.19], sequence=True)
        kt = K
        wt = max(W, 5)                 # the training path touches far more kernels / allocator blocks than inference

        def run_training(tmodel, opt, reducer, tpool, batch, steps, warm):
            tmodel.train()

            def train_step(arr, dense):
                gb = GraphBatch.from_arrays(*(arr[k] for k in keys), max_nodes=N_NODES)
                opt.zero_grad()
                recon, mu, logvar, out = tmodel(gb, dense["seq"], dense["prop"])
                loss = losses.BCE_loss(recon, dense["seq"], mu, logvar, out, dense["target"])
                loss.backward()
                reducer.step()
                opt.step()
                return loss

            for i in range(warm):
                train_step(*tpool[i % len(tpool)])
            # An eager step is ~200 launches enqueued in ~8 ms of host time against ~10.6 ms of device time: a busy host
            # core (shared box) turns it host-bound for a while.  Three back-to-back windows of `steps` steps are timed
            # on the device (max over ranks each) and the fastest is reported; all three are listed.
            windows = []
            for w_ in range(3):
                barrier()
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                for i in range(steps):
                    loss = train_step(*tpool[i % len(tpool)])
                e1.record()
                barrier()
                windows.append(max_over_ranks(e0.elapsed_time(e1)))
            ms_t = min(windows)
            tmodel.eval()
            return {"value": world * batch * steps / (ms_t / 1e3), "unit": "graphs/s", "steps": steps, "warmup": warm,
                    "ms_per_step": ms_t / steps, "ms_per_step_windows": [w_ / steps for w_ in windows],
                    "global_batch": world * batch, "loss": "BCE_loss(sequence=True)",
                    "final_loss": float(loss.detach()), "allreduce_bytes": reducer.nbytes,
                    "allreduce_buckets": len(reducer.buckets), "buckets_overlapped_with_backward": reducer.overlapped_last_step}

        import copy
        state0 = copy.deepcopy(model.state_dict())
        opt = I.FusedAdam(model.parameters(), lr=1e-3)
        train = run_training(model, opt, GradientAllReducer(model.parameters()), pool, B, kt, wt)
        train["optimizer"] = "immunostruct_b200.FusedAdam (one launch, flat buffers)"
        # the same step with torch.optim.Adam (the optimiser the reference constructs, train_IEDB_wFT.py:74), N = 1 only
        if world == 1 and not os.environ.get("BENCH_SKIP_EXTRAS"):
            tm = I.model_map["HybridModelv2"](vae_input_dim=VAE_IN, device=dev).to(dev)
            tm.load_state_dict(state0)
            t_adam = run_training(tm, torch.optim.Adam(tm.parameters(), lr=1e-3), GradientAllReducer(tm.parameters()), pool, B,
                                  kt, wt)
            train["torch_adam"] = {k: t_adam[k] for k in ("value", "unit", "ms_per_step", "final_loss")}
            del tm
        # BASELINE configs[3]: FIXED global batch of 4 096 graphs (strong scaling): 4096 / N graphs per GPU
        gb_fixed = 4096
        if gb_fixed % world == 0 and not os.environ.get("BENCH_SKIP_EXTRAS"):
            per = gb_fixed // world
            fpool = pool if per == B else make_pool(per, 2, seed=77 + 1000 * rank, device=dev)
            fm = I.model_map["HybridModelv2"](vae_input_dim=VAE_IN, device=dev).to(dev)
            fm.load_state_dict(state0)
            fixed = run_training(fm, I.FusedAdam(fm.parameters(), lr=1e-3), GradientAllReducer(fm.parameters()), fpool, per,
                                 5, 3)
            fixed.update({"scaling": "strong", "batch_per_gpu": per, "optimizer": "immunostruct_b200.FusedAdam"})
            train["fixed_global_batch_4096"] = fixed
            del fm, fpool
        model.load_state_dict(state0)
        model.eval()

    # ---- BASELINE configs[2]: cancer fine-tune step (train_Cancer_wFT.py / procedures/train.py:84-123) ---------
    # HybridModelv2_Comparative, 256 cancer / wild-type pairs (two independent graph draws sharing the target),
    # BCE + sequence loss on both members, paired contrastive loss (coefficient 0.01), AdamW(1e-4, wd 1e-6).
    train_cmp = None
    if not args.no_train and world == 1:
        P = B // 2
        torch.manual_seed(1)
        cmodel = I.model_map["HybridModelv2_Comparative"](vae_input_dim=VAE_IN, device=dev, use_wt_for_downstream=True).to(dev).train()
        copt = I.FusedAdamW(cmodel.parameters(), lr=1e-4, weight_decay=1e-6)
        closs = I.Losses(VAE_IN, [0.81, 0.19], sequence=True)
        pcl = I.PairedContrastiveLoss(embedding_dim=104, device=dev)
        cpool = make_pool(P, 4, seed=4001, device=dev)

        def cmp_step(i):
            (ac, dc), (aw, dw) = cpool[i % 4], cpool[(i + 1) % 4]
            gc = GraphBatch.from_arrays(*(ac[k] for k in keys), max_nodes=N_NODES)
            gw = GraphBatch.from_arrays(*(aw[k] for k in keys), max_nodes=N_NODES)
            embs, recons, mus, lvs, out = cmodel.forward_comparative((gc, gw), (dc["seq"], dw["seq"]), (dc["prop"], dw["prop"]))
            y = dc["target"]
            lc = closs.BCE_loss(recons[0], dc["seq"], mus[0], lvs[0], out, y)
            lw = closs.BCE_loss(recons[1], dw["seq"], mus[1], lvs[1], out, y)
            loss = (lc + lw) / 2 + 0.01 * pcl(embs[0], embs[1], y)
            copt.zero_grad()
            loss.backward()
            copt.step()
            return loss

        kc = K
        for i in range(max(W, 5)):
            cmp_step(i)
        cwin = []
        for w_ in range(3):                              # fastest of three windows, see run_training
            barrier()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for i in range(kc):
                loss = cmp_step(i)
            e1.record()
            barrier()
            cwin.append(e0.elapsed_time(e1))
        ms_c = min(cwin)
        train_cmp = {"value": P * kc / (ms_c / 1e3), "unit": "pairs/s", "graphs_per_s": 2 * P * kc / (ms_c / 1e3), "steps": kc,
                     "ms_per_step": ms_c / kc, "ms_per_step_windows": [w_ / kc for w_ in cwin], "pairs_per_step": P, "model": "HybridModelv2_Comparative", "optimizer": "immunostruct_b200.FusedAdamW",
                     "loss": "BCE_loss(sequence=True) on both members + 0.01 * PairedContrastiveLoss", "final_loss": float(loss.detach())}
        del cmodel, copt, cpool

    # ---- roofline of the dominant kernel (EGNN edge forward), timed alone ------------------------
    roofline = None
    if rank == 0:
        arr, dense = pool[0]
        gb = GraphBatch.from_arrays(*(arr[k] for k in keys), max_nodes=N_NODES)
        layer = model.GCN_layers[1]
        W1, b1, W2, b2, W3, b3, w4 = [t.detach().contiguous() for t in layer.kernel_params()[:7]]
        n, e = gb.n_nodes, gb.n_edges
        h = torch.randn(n, 64, device=dev)
        PQ, hn, xo = torch.empty(n, 128, device=dev), torch.empty(n, 64, device=dev), torch.empty(n, 3, device=dev)
        x = arr["x"][:, 20:]
        _C.egnn_node_pre_fwd(h, W1, b1, PQ)
        flush = torch.empty(64 * 1024 * 1024, device=dev)          # 256 MB > L2
        hbm_peak, tensor_peak, src = measured_peaks()

        def time_kernel(fn):
            times = []
            for it in range(3 + 10):
                flush.zero_()
                s0, s1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                s0.record()
                fn()
                s1.record()
                torch.cuda.synchronize()
                if it >= 3:
                    times.append(s0.elapsed_time(s1))
            return statistics.mean(times) / 1e3

        variants = {
            "fp32": lambda: _C.egnn_edge_fwd(gb, PQ, x, arr["edge_attr"], 64, W1, W2, b2, W3, b3, w4, True, hn, xo),
            "bf16x3": lambda: _C.egnn_edge_fwd_tc(gb, PQ, x, arr["edge_attr"], 64, W1, W2, b2, W3, b3, w4, True, _C.PREC_BF16X3, hn, xo, fast_act=True),
            "fp16x2": lambda: _C.egnn_edge_fwd_tc(gb, PQ, x, arr["edge_attr"], 64, W1, W2, b2, W3, b3, w4, True, _C.PREC_FP16X2, hn, xo, fast_act=True),
            "tf32x3": lambda: _C.egnn_edge_fwd_tc(gb, PQ, x, arr["edge_attr"], 64, W1, W2, b2, W3, b3, w4, True, _C.PREC_TF32X3, hn, xo, fast_act=True),
            "bf16": lambda: _C.egnn_edge_fwd_tc(gb, PQ, x, arr["edge_attr"], 64, W1, W2, b2, W3, b3, w4, True, _C.PREC_BF16, hn, xo),
            # first-generation tensor-core kernel (SIMT destination-side sums), for comparison
            "bf16x3_gen1": lambda: _C.egnn_edge_fwd_tc(gb, PQ, x, arr["edge_attr"], 64, W1, W2, b2, W3, b3, w4, True, _C.PREC_BF16X3 | 16, hn, xo, fast_act=True),
            "bf16_gen1": lambda: _C.egnn_edge_fwd_tc(gb, PQ, x, arr["edge_attr"], 64, W1, W2, b2, W3, b3, w4, True, _C.PREC_BF16 | 16, hn, xo),
        }
        t_all = {k: time_kernel(fn) for k, fn in variants.items()}
        ncu = ncu_record(args.precision)
        t_k = t_all[args.precision]
        flops = e * FLOP_PER_EDGE_EDGE_KERNEL
        nbytes = e * BYTES_PER_EDGE_EDGE_KERNEL + n * BYTES_PER_NODE_EDGE_KERNEL
        gbs = nbytes / t_k / 1e9
        kname = {"fp32": "is::edge_fwd_kernel<true> (fp32 SIMT)",
                 "tf32x3": "is::edge_fwd_tc_kernel<tf32x3, true> (tcgen05 + TMEM, lock-step)"}.get(
            args.precision, f"is::edge_fwd_ws_kernel<{args.precision}, true> (tcgen05 + TMEM, warp-specialised)")
        # The fused kernel's two roofline terms: compulsory bytes / HBM peak and GEMM flops / tensor peak.
        # The byte term is the larger one, so "hbm" is the bound the schema asks for; in practice the
        # kernel is limited by the SIMT work per edge -- 192 SiLUs (2 MUFU each in the fp32-accurate mode:
        # 91 us of MUFU pipe per launch) and ~100 issued warp-instructions -- see `simt` below and
        # profiles/r02_ws_*_edge_fwd_full.md (issue slots 53 %, MUFU 50 %, tensor pipe 37 %, DRAM 5 %).  The unit that is
        # nearly full is the shared-memory / L1 data pipe (128 B / clk / SM), which the LSU (operand stores, gathers, bias
        # reads) and the tensor core's operand reads share: `ncu.l1_pipe_lsu_pct` + `ncu.l1_pipe_tensor_operand_pct`.
        roofline = {"kernel": kname, "bound": "hbm", "achieved": gbs, "peak": hbm_peak, "unit": "GB/s",
                    "frac": gbs / hbm_peak, "traffic": (ncu or {}).get("dram_bytes") if B == BATCH else None,
                    "peak_source": src, "launch_ms": t_k * 1e3, "edges_per_launch": e,
                    "algorithmic_bytes_per_launch": nbytes, "algorithmic_flops_per_launch": flops,
                    "tensor": {"achieved": flops / t_k / 1e12, "peak": tensor_peak, "unit": "TFLOP/s",
                               "frac": flops / t_k / 1e12 / tensor_peak},
                    "l2_gather_gbs": e * GATHER_BYTES_PER_EDGE / t_k / 1e9,
                    "ncu": ncu,
                    "simt": {"mufu_floor_ms": e * 192 * (1 if args.precision == "bf16" else 2) / (148 * 16 * 1.965e9) * 1e3,
                             "note": "192 SiLU per edge, 1 (bf16: tanh.approx) or 2 (ex2 + rcp) MUFU ops each, 16 MUFU lanes / clk / SM"},
                    "roofline_time_ms": {"hbm": nbytes / hbm_peak / 1e6, "tensor": flops / tensor_peak / 1e9},
                    "launch_ms_by_precision": {k: v * 1e3 for k, v in t_all.items()},
                    "note": "edge-forward kernel of one EGNN layer (batch 512) timed alone with CUDA events after an "
                            "L2 flush; bytes = each input/output byte once (PQ rows, coordinates, CSR ids, edge_attr, hn, "
                            "x'); FLOPs = two 64x64 per-edge GEMMs + w4 dot (split-precision extra MMAs not counted); "
                            "traffic = ncu dram bytes of the same launch"}

    # ---- CPU baseline on this box's host cores, rank 0 at N=1 only: the reference's CPU path (its own model code when
    # baseline/_ref is present, else the oracle port), inference and -- BASELINE configs[0] -- fwd + bwd at batch 64 ---
    cpu_baseline = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        torch.set_num_threads(os.cpu_count() or 1)
        ref = ReferenceCPU()
        sample = 64
        cpool = make_pool(sample, 1, seed=1, device="cpu")
        eps = torch.randn(sample, 32)
        ref.infer(*cpool[0], eps)
        t0 = time.perf_counter()
        reps = 0
        while reps < 3 or time.perf_counter() - t0 < 8.0:
            ref.infer(*cpool[0], eps)
            reps += 1
        dt = time.perf_counter() - t0
        ref.train_step(*cpool[0], eps)
        t1 = time.perf_counter()
        reps_t = 0
        while reps_t < 2 or time.perf_counter() - t1 < 10.0:
            ref.train_step(*cpool[0], eps)
            reps_t += 1
        dt_t = time.perf_counter() - t1
        cpu_baseline = {"value": sample * reps / dt, "unit": "graphs/s", "cores": torch.get_num_threads(),
                        "kind": ref.kind, "sample": f"{reps} x {sample}-graph batches (same graph shape), {ref.describe()}, "
                                                  "torch CPU fp32",
                        "train": {"value": sample * reps_t / dt_t, "unit": "graphs/s", "ms_per_step": dt_t / reps_t * 1e3,
                                  "sample": f"{reps_t} x fwd + bwd of a {sample}-graph batch, BCE_loss(sequence=True) "
                                            "(BASELINE configs[0]), no optimizer step"}}

    # (last: a failed capture may leave the process RNG / allocator in capture mode)
    # ---- the same step captured once in a CUDA graph and replayed (SURVEY 8(f) row 3): fixed shapes, no host
    # synchronisation inside the step, FusedAdam(capturable=True): the step count lives on the device; the host only
    # copies the next batch into the static input buffers and replays
    if world == 1 and not args.no_train:
        model.train()
        try:
            opt_g = I.FusedAdam(model.parameters(), lr=1e-3, capturable=True)

            def graph_body(t):
                gb = GraphBatch.from_arrays(*(t[k] for k in keys), max_nodes=N_NODES)
                opt_g.zero_grad(set_to_none=True)
                recon, mu, logvar, out = model(gb, t["seq"], t["prop"])
                loss = losses.BCE_loss(recon, t["seq"], mu, logvar, out, t["target"])
                loss.backward()
                opt_g.step()
                return loss

            captured = I.CapturedStep(graph_body, {**{k: pool[0][0][k] for k in keys},
                                                   **{k: pool[0][1][k] for k in ("seq", "prop", "target")}})
            loss_s = None

            def graph_step(arr, dense):
                nonlocal loss_s
                loss_s = captured({**{k: arr[k] for k in keys}, **{k: dense[k] for k in ("seq", "prop", "target")}})

            for i in range(wt):
                graph_step(*pool[i % POOL])
            barrier()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for i in range(kt):
                graph_step(*pool[i % POOL])
            e1.record()
            barrier()
            ms_g = e0.elapsed_time(e1)
            train["cuda_graph"] = {"value": B * kt / (ms_g / 1e3), "unit": "graphs/s", "ms_per_step": ms_g / kt,
                                   "final_loss": float(loss_s), "note": "immunostruct_b200.CapturedStep: whole step (collation, fwd, loss, bwd, FusedAdam capturable) captured once, inputs copied into static buffers per step"}
            del captured
        except Exception as exc:                      # capture is an optimisation: report, never fail the bench
            train["cuda_graph"] = {"error": f"{type(exc).__name__}: {exc}"[:300]}
            print("cuda graph capture failed:", repr(exc), file=sys.stderr)

    if rank == 0:
        print(json.dumps({
            "metric": "pMHC graphs/sec (HybridModelv2 inference, fp32)", "value": value, "unit": "graphs/s",
            "precision": args.precision, "other_precisions": other,
            "n_gpus": world, "steps": K, "warmup": W, "ms_per_step": ms / K,
            "ms_per_step_windows": [w_ / K for w_ in infer_windows], "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "bf16" if args.precision == "bf16" else "f32", "data": "synthetic",
            "config": {"workload": WORKLOAD,
                       "batch_per_gpu": B, "nodes_per_graph": N_NODES, "edges_per_graph": N_NODES * KNN,
                       "parallelism": f"dp{world}", "l2": f"{POOL} resident input batches (~42 MB each) cycled: inputs > L2"},
            "clocks": clk.summary(),
            "e2e": {"value": e2e_value, "unit": "graphs/s", "ms_per_step": ms_e2e / K,
                    "ms_per_step_windows": [w_ / K for w_ in e2e_windows], "h2d_bytes_per_step": h2d,
                    "d2h_bytes_per_step": B * 4,
                    "compact_input": {"value": world * B * K / (ms_e2e_packed / 1e3), "unit": "graphs/s",
                                      "ms_per_step": ms_e2e_packed / K, "h2d_bytes_per_step": h2d_packed,
                                      "note": "same call path fed from immunostruct_b200.PackedGraphBatch / PackedSequence"}},
            "gpu_launches": launches, "scan_27000": scan,
            "train_graphs_per_s": None if train is None else train["value"],
            "train_fixed4096_graphs_per_s": None if train is None or "fixed_global_batch_4096" not in train
            else train["fixed_global_batch_4096"]["value"],
            "train": train, "train_comparative": train_cmp, "roofline": roofline, "cpu_baseline": cpu_baseline,
        }))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
