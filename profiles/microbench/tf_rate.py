"""tf_rate.py — rate of the two tcgen05 scorers on the bench shape (37 888 users x 5 M items, D=64,
k=20), random xavier-like tables, no mask (kernel alone, CUDA events, 3 launches after 2 warm-ups).
    python profiles/microbench/tf_rate.py [--users 37888] [--items 5000000] [--D 64] [--k 20]
Also prints the slow-path statistics of the f16 kernel (tiles that entered the survivor path and
8-column group calls, summed over epilogue warps).
"""
import argparse
import ctypes as C
import hashlib
import json
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from spex_b200 import _capi, ops  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--users", type=int, default=148 * 2 * 128)
    ap.add_argument("--items", type=int, default=5_000_000)
    ap.add_argument("--D", type=int, default=64)
    ap.add_argument("--k", type=int, default=20)
    ap.add_argument("--norm-spread", type=float, default=0.0, help="item row norms in [1, 1+spread]")
    args = ap.parse_args()
    dev = torch.device("cuda:0")
    g = torch.Generator(device=dev)
    g.manual_seed(1)
    a = (6.0 / (args.items + args.D)) ** 0.5
    I = torch.empty(args.items, args.D, device=dev).uniform_(-a, a, generator=g)
    if args.norm_spread > 0:
        I *= 1.0 + args.norm_spread * torch.rand(args.items, 1, device=dev, generator=g)
    U = torch.empty(args.users, args.D, device=dev).uniform_(-a, a, generator=g)
    users = torch.arange(args.users, device=dev)
    idx = torch.empty(args.users, args.k, dtype=torch.int32, device=dev)
    val = torch.empty(args.users, args.k, dtype=torch.float32, device=dev)
    flops = 2.0 * args.users * args.items * args.D
    out = {"users": args.users, "items": args.items, "D": args.D, "k": args.k}

    def timed(fn):
        for _ in range(2):
            fn()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(3):
            fn()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / 3

    Ih, m_pad, imeta = ops.pack_f16(I, None, ops.TC_ITEM_MULTIPLE)
    Uh, b_pad, umeta = ops.pack_f16(U, users, ops.TC_USER_MULTIPLE)
    stats = torch.zeros(8, dtype=torch.int64, device=dev)
    _capi.lib.spex_debug_tf_stats.argtypes = [C.c_void_p]
    _capi.lib.spex_debug_tf_stats.restype = None
    _capi.lib.spex_debug_tf_stats(C.c_void_p(stats.data_ptr()))
    ops.score_topk_f16(Uh, umeta, args.users, b_pad, Ih, imeta, args.items, m_pad, args.D, args.k, None, None, None, idx, val)
    torch.cuda.synchronize()
    st = stats.tolist()
    _capi.lib.spex_debug_tf_stats(C.c_void_p(0))
    ms = timed(lambda: ops.score_topk_f16(Uh, umeta, args.users, b_pad, Ih, imeta, args.items, m_pad, args.D, args.k,
                                          None, None, None, idx, val))
    n_warp_tiles = (b_pad // 128) * 4 * (m_pad // 128)
    nw = (b_pad // 128) * 4
    out["f16"] = {"ms": round(ms, 3), "tflops": round(flops / ms / 1e9, 1), "slow_tiles_frac": st[0] / n_warp_tiles,
                  "block_calls_per_warp": st[1] / nw, "slow_path_cycles_per_warp": st[2] / nw,
                  "inserts_per_warp": st[3] / nw, "exact_settlements_per_warp": st[4] / nw,
                  "exact_settlement_cycles_per_warp": st[5] / nw}
    # digest of the f16 result bits: two builds of the exact scorer must agree on it
    out["f16"]["out_sha256"] = hashlib.sha256(idx.cpu().numpy().tobytes() + val.cpu().numpy().tobytes()).hexdigest()
    i16 = idx.clone()
    if args.D == 64:
        Ib, m_pad2 = ops.pack_bf16(I, None, ops.TC_ITEM_MULTIPLE)
        Ub, b_pad2 = ops.pack_bf16(U, users, ops.TC_USER_MULTIPLE)
        ms = timed(lambda: ops.score_topk_bf16(Ub, args.users, b_pad2, Ib, args.items, m_pad2, args.k, None, None, None,
                                               idx, val))
        out["bf16"] = {"ms": round(ms, 3), "tflops": round(flops / ms / 1e9, 1)}
        out["top_k_agreement_f16_vs_bf16"] = float((i16 == idx).float().mean())
    print(json.dumps(out))


if __name__ == "__main__":
    main()
