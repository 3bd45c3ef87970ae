"""fullrank_eval.py — cost of full-ranking evaluation with the metrics on the device against the host path.

Workload: U [users, 64] and I [items, 64] seeded xavier tables (synthetic.xavier_table, as bench.py's eval sweep
initialises them; 10 M x 5 M by default), a seeded training mask of 10 items per user, held-out truth of 1 item
per user (the reference data's shape) or 10 items per user, k = 50 with cutoffs [10, 20, 50], f16 scorer, users in
blocks of ops.EVAL_USER_BLOCK.  Arms, alternated, `--runs` each, per truth variant:
  (a) topk       FullRanker.topk sweep over all users (ids and scores stay on the device)
  (b) evaluate   FullRanker.evaluate sweep over all users (ranking + spex_fullrank_metrics per block + reduce)
  (c) host       FullRanker.topk + .cpu() + metrics.fullrank_recall_ndcg at each cutoff, on the first
                 `--host-users` users: measured there; the 10 M-user figure is that time scaled, labelled
                 extrapolated
Times are host clocks around work that ends in a device synchronise.  The metric kernel alone: CUDA events over
`--reps` launches on the stored top-50 ids of all users from arm (a); algorithmic bytes B k 4 + B 8 + truth 4.
(c) is checked against (b) on the same users.  The card's name and power limit are read before and after.
    python profiles/microbench/fullrank_eval.py [--users 10000000] [--items 5000000] [--runs 3]
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from spex_b200 import metrics, ops, synthetic  # noqa: E402
from spex_b200._capi import call, ptr, stream_ptr  # noqa: E402

K, CUTOFFS, D, MASK_PER_USER = 50, [10, 20, 50], 64, 10


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 else "unknown"


def emit(**kw):
    print(json.dumps(kw), flush=True)


def seeded_rows(n, per, m, seed, dev):
    """CSR (rowptr int64, col int32) with `per` seeded items per row, each row ascending."""
    g = torch.Generator(device=dev)
    g.manual_seed(seed)
    col = torch.randint(0, m, (n, per), generator=g, device=dev, dtype=torch.int32)
    col = torch.sort(col, dim=1).values.reshape(-1).contiguous()
    return torch.arange(0, n * per + 1, per, dtype=torch.int64, device=dev), col


def wall(fn):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    out = fn()
    torch.cuda.synchronize()
    return time.perf_counter() - t0, out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--users", type=int, default=10_000_000)
    ap.add_argument("--items", type=int, default=5_000_000)
    ap.add_argument("--host-users", type=int, default=200_000)
    ap.add_argument("--runs", type=int, default=3)
    ap.add_argument("--reps", type=int, default=20)
    a = ap.parse_args()
    dev = torch.device("cuda:0")
    B, m = a.users, a.items
    emit(card=card(), users=B, items=m, D=D, k=K, cutoffs=CUTOFFS, user_block=ops.EVAL_USER_BLOCK)
    table = synthetic.xavier_table(B, m, D, 2020, dev)
    U, I = table[:B], table[B:]
    users = torch.arange(B, device=dev)
    mrp, mcol = seeded_rows(B, MASK_PER_USER, m, 7, dev)
    ranker = ops.FullRanker(I, "f16")
    blk = ops.EVAL_USER_BLOCK
    nh = min(a.host_users, B)
    for per in (1, 10):
        trp, tcol = seeded_rows(B, per, m, 11 + per, dev)
        # warm-up of every shape the timed window uses
        ranker.topk(U, users[:blk], K, mrp, mcol, blk)
        ranker.evaluate(U, users[:blk], CUTOFFS, trp[: blk + 1], tcol, mrp, mcol, blk)
        idx = None
        for run in range(a.runs):
            del idx
            t_a, (idx, val) = wall(lambda: ranker.topk(U, users, K, mrp, mcol, blk))
            del val
            emit(truth_per_user=per, arm="a_topk", run=run, s=round(t_a, 3))
            t_b, res = wall(lambda: ranker.evaluate(U, users, CUTOFFS, trp, tcol, mrp, mcol, blk))
            emit(truth_per_user=per, arm="b_evaluate", run=run, s=round(t_b, 3),
                 **{n: res[n].tolist() for n in ops.METRIC_NAMES})

            def host():
                i, _ = ranker.topk(U, users[:nh], K, mrp, mcol, blk)
                i = i.cpu().numpy()
                rp, col = trp[: nh + 1].cpu().numpy(), tcol[: nh * per].cpu().numpy()
                return [metrics.fullrank_recall_ndcg(i, rp, col, c) for c in CUTOFFS]

            t_c, ref = wall(host)
            emit(truth_per_user=per, arm="c_host", run=run, users_measured=nh, s_measured=round(t_c, 3),
                 s_extrapolated_to_all_users=round(t_c * B / nh, 1))
        dsub = ranker.evaluate(U, users[:nh], CUTOFFS, trp[: nh + 1], tcol, mrp, mcol, blk)
        dev_vs_host = max(max(abs(dsub["recall"][j] - r.mean()), abs(dsub["ndcg"][j] - n.mean()))
                          for j, (r, n) in enumerate(ref))
        emit(truth_per_user=per, check="evaluate_vs_host_on_host_users", max_abs_diff=dev_vs_host)
        # the metric kernel alone on the stored top-50 ids of all users
        disc, idcg = (torch.from_numpy(x).to(dev) for x in ops.rank_discounts(K))
        n_chunks = (B + ops.METRICS_CHUNK - 1) // ops.METRICS_CHUNK
        cs = torch.empty(n_chunks, len(CUTOFFS), 4, dtype=torch.float64, device=dev)
        cut = (C.c_int32 * len(CUTOFFS))(*CUTOFFS)

        def kernel():
            call("spex_fullrank_metrics", ptr(idx), B, K, ptr(trp), ptr(tcol), cut, len(CUTOFFS), ptr(disc),
                 ptr(idcg), None, ptr(cs), stream_ptr())

        for _ in range(2):
            kernel()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(a.reps):
            kernel()
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / a.reps
        nbytes = B * K * 4 + B * 8 + B * per * 4
        emit(truth_per_user=per, arm="metric_kernel", ms=round(ms, 3), bytes=nbytes,
             gb_per_s=round(nbytes / ms / 1e6, 1), reps=a.reps)
        del idx, trp, tcol
    emit(card_after=card())


if __name__ == "__main__":
    main()
