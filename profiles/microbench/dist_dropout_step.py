"""dist_dropout_step.py — what edge dropout (--dropout 2) costs in the row-partitioned training step.

configs[3] graph (10 M users x 5 M items, 2e9 edges, D=64, K=3) cut into nnz-balanced row blocks, one per GPU;
PartitionedTrainer's receptive-field step (B=256, fused Adam tail) with keep_prob 0.3 against no dropout, arms
alternated, 3 runs each, median.  Also the dropout kernel alone on a rank's block (val and valT, no tpos: the
synthetic graph's values are symmetric bit for bit).  Step times are the slowest rank's (events, all-reduce max).

Run on B200s:  torchrun --nproc-per-node N profiles/microbench/dist_dropout_step.py [--exchange push|mcast]
               [--scale 1.0] [--out FILE]
The default exchange is the one bench.py picks: push below 4 GPUs, mcast from 4 on.
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
from spex_b200 import ops, synthetic  # noqa: E402
from spex_b200.dist import PartitionedPropagator, PartitionedTrainer  # noqa: E402
from spex_b200.graph import partition_rows_by_nnz  # noqa: E402

D = 64


def card(i):
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i",
                        str(i)], capture_output=True, text=True, timeout=30).stdout.strip()
    return q or torch.cuda.get_device_name(i)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--scale", type=float, default=1.0)
    ap.add_argument("--keep-prob", type=float, default=0.3)
    ap.add_argument("--exchange", choices=("push", "mcast"), default=None)
    ap.add_argument("--steps", type=int, default=8, help="timed steps per run")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
    local_rank = int(os.environ.get("LOCAL_RANK", rank))
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    dist.init_process_group("nccl", device_id=dev)
    exchange = args.exchange or ("mcast" if world >= 4 else "push")
    kp = args.keep_prob
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
    gen = torch.Generator(device=dev)
    gen.manual_seed(11)
    users, items, labels = sample_train_batch(torch, g, nur, m, 256, gen)
    rp_host = g.rowptr.cpu().numpy()
    bounds = partition_rows_by_nnz(rp_host, world)
    r0, r1 = bounds[rank], bounds[rank + 1]
    lo, hi = int(rp_host[r0]), int(rp_host[r1])
    lg = ops.DeviceGraph((g.rowptr[r0: r1 + 1] - lo).contiguous(), g.col[lo:hi].clone(), g.val[lo:hi].clone(), N,
                         None, g.seg_len, row_offset=r0, col_hot=g.col_hot, values_symmetric=g.values_symmetric)
    W_start = table[r0:r1].clone()
    emit("workload", f"{nu} users x {m} items, nnz(A)={g.nnz}, D={D}, K={K_LAYERS}, keep_prob={kp}, {world} GPU(s), "
                     f"exchange={exchange}, rank 0 block: {r1 - r0} rows, {hi - lo} edges")
    del g, table
    torch.cuda.empty_cache()

    # the kernel alone on this rank's block
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    lg.device_dropout_values(1, kp)
    torch.cuda.synchronize()
    e0.record()
    for s in range(5):
        lg.device_dropout_values(2 + s, kp)
    e1.record()
    torch.cuda.synchronize()
    t = torch.tensor([e0.elapsed_time(e1) / 5], dtype=torch.float64, device=dev)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    emit("kernel_on_block", {"ms_max_over_ranks": round(float(t.item()), 3)})

    prop = PartitionedPropagator(lg, bounds, D, K_LAYERS, mode=exchange, device=dev)
    if exchange == "push" and world == 2:
        prop.e0_exchange = "push"   # as bench.py at 2 GPUs

    def run(keep_prob):
        tr = PartitionedTrainer(prop, W_start.clone(), nur, lr=1e-3, keep_prob=keep_prob)
        prop._staged = None          # the table of the previous arm is not this one's
        for _ in range(2):
            tr.step(users, items, labels)
        torch.cuda.synchronize()
        dist.barrier()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(args.steps):
            tr.step(users, items, labels)
        b.record()
        torch.cuda.synchronize()
        ms = torch.tensor([a.elapsed_time(b) / args.steps], dtype=torch.float64, device=dev)
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        del tr
        return float(ms.item())

    torch.manual_seed(2020)   # the dropout seeds of the steps
    runs = {None: [], kp: []}
    for _ in range(3):
        for arm in (None, kp):
            runs[arm].append(run(arm))
    base, drop = statistics.median(runs[None]), statistics.median(runs[kp])
    emit("train_step", {"no_dropout_ms": [round(x, 2) for x in runs[None]],
                        "dropout_ms": [round(x, 2) for x in runs[kp]],
                        "median_no_dropout_ms": round(base, 2), "median_dropout_ms": round(drop, 2),
                        "overhead_ms": round(drop - base, 2),
                        "note": f"{args.steps} timed steps per run after 2 untimed, events, slowest rank; arms "
                                "alternated; B=256, receptive field, fused Adam tail"})
    prop.close()
    if rank == 0 and args.out:
        with open(args.out, "w") as f:
            f.write(f"# torchrun --nproc-per-node {world} profiles/microbench/dist_dropout_step.py --scale {args.scale} "
                    f"--exchange {exchange}\n")
            f.write("\n".join(lines) + "\n")
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
