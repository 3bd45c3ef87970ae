"""rank_pairs.py — full-ranking metrics from held-out ranks (FullRanker.rank_metrics: spex_rank_pairs_f16 +
spex_rank_metrics) against the same metrics from top-k lists (FullRanker.evaluate), on the same users.

Workload: U [users, D] and I [items, D] seeded xavier tables (synthetic.xavier_table, as bench.py initialises
them; 10 M x 5 M by default), D = 64 and 128, a seeded training mask of 10 items per user (the bench-shaped graph
of fullrank_eval.py), one held-out non-training item per user in two flavours:
  random  a seeded random item: ranks spread over the catalogue, most item tiles hold scores on both sides of the
          held-out score (the worst case for counting);
  best    the user's best non-training item (FullRanker.topk with k = 1): rank 0, as after training.
Cutoffs [10, 20, 50]; evaluate ranks at k = 50.  The two arms alternate, `--runs` each; times are host clocks
around work that ends in a device synchronise.  TFLOP/s = 2 users items D / t.  The card's name and power limit
are read before and after.  Both arms' recall/ndcg/hit are printed; they must agree.
    python profiles/microbench/rank_pairs.py [--users 10000000] [--items 5000000] [--runs 3] [--dims 64 128]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from spex_b200 import ops, synthetic  # noqa: E402

CUTOFFS, MASK_PER_USER = [10, 20, 50], 10


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
    ap.add_argument("--runs", type=int, default=3)
    ap.add_argument("--dims", type=int, nargs="+", default=[64, 128])
    ap.add_argument("--flavours", nargs="+", default=["best", "random"])
    a = ap.parse_args()
    dev = torch.device("cuda:0")
    B, m = a.users, a.items
    emit(card=card(), users=B, items=m, cutoffs=CUTOFFS, mask_per_user=MASK_PER_USER)
    users = torch.arange(B, device=dev)
    mrp, mcol = seeded_rows(B, MASK_PER_USER, m, 7, dev)
    for D in a.dims:
        table = synthetic.xavier_table(B, m, D, 2020, dev)
        U, I = table[:B], table[B:]
        ranker = ops.FullRanker(I, "f16")
        flops = 2.0 * B * m * D
        for flavour in a.flavours:
            if flavour == "best":
                best, _ = ranker.topk(U, users, 1, mrp, mcol, ops.EVAL_USER_BLOCK)
                tcol = best[:, 0].contiguous()
                del best
            else:
                g = torch.Generator(device=dev)
                g.manual_seed(13)
                tcol = torch.randint(0, m, (B,), generator=g, device=dev, dtype=torch.int32)
            trp = torch.arange(B + 1, dtype=torch.int64, device=dev)
            w = min(B, 4096)                                   # warm-up of both arms
            ranker.evaluate(U, users[:w], CUTOFFS, trp[: w + 1], tcol, mrp, mcol)
            ranker.rank_metrics(U, users[:w], CUTOFFS, trp[: w + 1], tcol, mrp, mcol)
            for run in range(a.runs):
                for arm in ("evaluate", "rank_metrics"):
                    fn = getattr(ranker, arm)
                    t, res = wall(lambda: fn(U, users, CUTOFFS, trp, tcol, mrp, mcol))
                    extra = {"mrr": res["mrr"], "auc": res["auc"]} if arm == "rank_metrics" else {}
                    emit(D=D, flavour=flavour, arm=arm, run=run, s=round(t, 3), tflops=round(flops / t / 1e12, 1),
                         recall=res["recall"].tolist(), ndcg=res["ndcg"].tolist(), hit=res["hit"].tolist(), **extra)
            del tcol, trp
        del table, U, I, ranker
        torch.cuda.empty_cache()
    emit(card_after=card())


if __name__ == "__main__":
    main()
