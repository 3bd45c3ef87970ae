"""bpr_step.py — the BPR training step (--loss bpr) on the configs[3] graph.

configs[3] graph (10 M users x 5 M items, 1e9 interactions, 2e9 edges, D=64, K=3), B = 2048 triples drawn on the device
(spex_sample_bpr), receptive field on:
  one_gpu      the single-GPU step: ops.propagate_mean(rows_needed) + ops.bpr_loss, loss + decay * reg backward,
               spex_adam_f32 - against the BCE step of the same loop at B = 256 (ops.bce_loss);
  partitioned  PartitionedTrainer.bpr_step with the fused tail (the L2 gradient added in the Adam epilogue, z_add)
               against fused_tail=False (added in the last layer's Z, then spex_adam_f32 over the slice), at world N;
               that arm also runs without what only the fused tail has (receptive field, locally assembled gradient
               table), so the difference is the fused path's, not the added term's alone.
Arms alternated, 3 runs each, median; step times are the slowest rank's (events, all-reduce max).

Run on B200s:  torchrun --nproc-per-node N profiles/microbench/bpr_step.py [--scale 1.0] [--out FILE]
(the one-GPU arms run at N = 1 only; the exchange is the one bench.py picks: push below 4 GPUs, mcast from 4 on)
"""
import argparse
import json
import os
import statistics
import subprocess
import sys

import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from bench import K_LAYERS, sample_train_batch  # noqa: E402
from spex_b200 import dataloader, ops, synthetic  # noqa: E402
from spex_b200.dist import PartitionedPropagator, PartitionedTrainer  # noqa: E402
from spex_b200.graph import partition_rows_by_nnz  # noqa: E402

D = 64
DECAY = 1e-4


def card(i):
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i",
                        str(i)], capture_output=True, text=True, timeout=30).stdout.strip()
    return q or torch.cuda.get_device_name(i)


def timed(fn, steps, dev):
    """Mean ms of `steps` calls after 2 untimed ones, the slowest rank's."""
    for _ in range(2):
        fn()
    torch.cuda.synchronize()
    if dist.get_world_size() > 1:
        dist.barrier()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(steps):
        fn()
    b.record()
    torch.cuda.synchronize()
    ms = torch.tensor([a.elapsed_time(b) / steps], dtype=torch.float64, device=dev)
    dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    return float(ms.item())


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--scale", type=float, default=1.0)
    ap.add_argument("--batch", type=int, default=2048)
    ap.add_argument("--steps", type=int, default=8, help="timed steps per run")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
    local_rank = int(os.environ.get("LOCAL_RANK", rank))
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    dist.init_process_group("nccl", device_id=dev)
    exchange = "mcast" if world >= 4 else "push"
    lines = []

    def emit(key, value):
        if rank == 0:
            s = json.dumps({key: value})
            print(s, flush=True)
            lines.append(s)

    emit("card", card(local_rank))
    nu, m, ni = int(10_000_000 * args.scale), int(5_000_000 * args.scale), int(1_000_000_000 * args.scale)
    nur = nu + 1
    N = nur + m
    keys = synthetic.generate_interactions(nu, m, ni, seed=2020, device=dev)
    g, _, _ = synthetic.build_norm_adj_device(keys, nu, m)
    del keys
    g.mark_hot_columns(D)
    table = synthetic.xavier_table(nur, m, D, 2020, dev)
    B = args.batch
    # triples from the adjacency's user rows (items listed as nur + item, hot bit masked by the sampler)
    users, pos, neg = dataloader.uniform_sample_bpr_device(g.rowptr, g.col, nur, m, nur, B, seed=7)
    gen = torch.Generator(device=dev)
    gen.manual_seed(11)
    bu, bi, bl = sample_train_batch(torch, g, nur, m, 256, gen)
    emit("workload", f"{nu} users x {m} items, nnz(A)={g.nnz}, D={D}, K={K_LAYERS}, B={B} triples, decay={DECAY}, "
                     f"{world} GPU(s), exchange={exchange}, receptive field on")

    if world == 1:
        ops.enable_persistent_workspaces(True)
        p = table.clone().requires_grad_(True)
        mo, vo = torch.zeros_like(table), torch.zeros_like(table)
        t = [0]

        def one_gpu(kind):
            def step():
                if kind == "bpr":
                    rows = torch.cat([users, pos + nur, neg + nur])
                    out = ops.propagate_mean(p, g, K_LAYERS, rows_needed=rows)
                    loss, reg = ops.bpr_loss(out, p, nur, users, pos, neg)
                    loss = loss + DECAY * reg
                else:
                    out = ops.propagate_mean(p, g, K_LAYERS, rows_needed=torch.cat([bu, bi + nur]))
                    loss = ops.bce_loss(out, nur, bu, bi, bl)
                loss.backward()
                t[0] += 1
                ops.adam_step(p.data, p.grad, mo, vo, 1e-3, 0.9, 0.999, 1e-8, t[0])
                p.grad = None
            return step

        runs = {"bpr": [], "bce": []}
        for _ in range(3):
            for arm in ("bpr", "bce"):
                runs[arm].append(timed(one_gpu(arm), args.steps, dev))
        emit("one_gpu_step", {"bpr_B2048_ms": [round(x, 2) for x in runs["bpr"]],
                              "bce_B256_ms": [round(x, 2) for x in runs["bce"]],
                              "median_bpr_ms": round(statistics.median(runs["bpr"]), 2),
                              "median_bce_ms": round(statistics.median(runs["bce"]), 2),
                              "note": f"{args.steps} timed steps per run after 2 untimed, events; arms alternated; "
                                      "ops.propagate_mean(rows_needed) + loss + backward + spex_adam_f32"})
        del p, mo, vo
        ops.enable_persistent_workspaces(False)
        torch.cuda.empty_cache()
    else:
        emit("one_gpu_step", "not measured at this world size (N = 1 only)")

    rp_host = g.rowptr.cpu().numpy()
    bounds = partition_rows_by_nnz(rp_host, world)
    r0, r1 = bounds[rank], bounds[rank + 1]
    lo, hi = int(rp_host[r0]), int(rp_host[r1])
    lg = ops.DeviceGraph((g.rowptr[r0: r1 + 1] - lo).contiguous(), g.col[lo:hi].clone(), g.val[lo:hi].clone(), N,
                         None, g.seg_len, row_offset=r0, col_hot=g.col_hot, values_symmetric=g.values_symmetric)
    W_start = table[r0:r1].clone()
    del g, table
    torch.cuda.empty_cache()
    prop = PartitionedPropagator(lg, bounds, D, K_LAYERS, mode=exchange, device=dev)
    if exchange == "push" and world == 2:
        prop.e0_exchange = "push"   # as bench.py at 2 GPUs

    def partitioned(fused_tail):
        def run():
            tr = PartitionedTrainer(prop, W_start.clone(), nur, lr=1e-3, fused_tail=fused_tail, decay=DECAY)
            prop._staged = None      # the table of the previous arm is not this one's
            ms = timed(lambda: tr.bpr_step(users, pos, neg), args.steps, dev)
            del tr
            return ms
        return run

    runs = {True: [], False: []}
    for _ in range(3):
        for arm in (True, False):
            runs[arm].append(partitioned(arm)())
    emit("partitioned_bpr_step", {"fused_tail_ms": [round(x, 2) for x in runs[True]],
                                  "unfused_tail_ms": [round(x, 2) for x in runs[False]],
                                  "median_fused_tail_ms": round(statistics.median(runs[True]), 2),
                                  "median_unfused_tail_ms": round(statistics.median(runs[False]), 2),
                                  "note": f"{args.steps} timed steps per run after 2 untimed, events, slowest rank; "
                                          "arms alternated; B=2048, receptive field"})
    prop.close()
    if rank == 0 and args.out:
        with open(args.out, "w") as f:
            f.write(f"# torchrun --nproc-per-node {world} profiles/microbench/bpr_step.py --scale {args.scale}\n")
            f.write("\n".join(lines) + "\n")
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
