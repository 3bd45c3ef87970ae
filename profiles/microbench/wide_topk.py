"""wide_topk.py — rate of the full-ranking scorers at k above 64 on the tf_rate.py shape (37 888 users x 5 M items,
xavier-like tables, no mask; D = 64, then the D = 128 NGCF case): spex_score_topk_f16 at k = 20 / 64,
spex_score_topk_f16_wide at k = 65 .. 512 and spex_score_topk_f32 at k = 100 / 128, the last two alternated on the
same inputs.  Kernel time by CUDA events (2 warm-ups, then `--reps` launches); TFLOP/s = 2 B m D / t.  Also the
workspace bytes per call, the compaction counts of the wide kernel (fast / exact, per epilogue warp) and the card.
    python profiles/microbench/wide_topk.py [--users 37888] [--items 5000000] [--reps 3]
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from spex_b200 import _capi, ops  # noqa: E402


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 else "unknown"


def timed(fn, reps):
    for _ in range(2):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps


def run(D, n_u, m, reps, ks_wide, f32_ks):
    dev = torch.device("cuda:0")
    g = torch.Generator(device=dev)
    g.manual_seed(1)
    a = (6.0 / (m + D)) ** 0.5
    I = torch.empty(m, D, device=dev).uniform_(-a, a, generator=g)
    U = torch.empty(n_u, D, device=dev).uniform_(-a, a, generator=g)
    users = torch.arange(n_u, device=dev)
    flops = 2.0 * n_u * m * D
    Ih, m_pad, imeta = ops.pack_f16(I, None, ops.TC_ITEM_MULTIPLE)
    Uh, b_pad, umeta = ops.pack_f16(U, users, ops.TC_USER_MULTIPLE)
    args = (Uh, umeta, n_u, b_pad, Ih, imeta, m, m_pad, D)
    rows = []

    def rate(name, k, ms, **kw):
        r = {"D": D, "scorer": name, "k": k, "ms": round(ms, 3), "tflops": round(flops / ms / 1e9, 1), **kw}
        rows.append(r)
        print(json.dumps(r), flush=True)

    for k in (20, 64):
        oi = torch.empty(n_u, k, dtype=torch.int32, device=dev)
        ov = torch.empty(n_u, k, dtype=torch.float32, device=dev)
        rate("f16", k, timed(lambda: ops.score_topk_f16(*args, k, None, None, None, oi, ov), reps))
    stats = torch.zeros(8, dtype=torch.int64, device=dev)
    _capi.lib.spex_debug_tf_stats.argtypes = [C.c_void_p]
    _capi.lib.spex_debug_tf_stats.restype = None
    nw = (b_pad // 128) * 4
    for k in ks_wide:
        oi = torch.empty(n_u, k, dtype=torch.int32, device=dev)
        ov = torch.empty(n_u, k, dtype=torch.float32, device=dev)
        stats.zero_()
        _capi.lib.spex_debug_tf_stats(C.c_void_p(stats.data_ptr()))
        ops.score_topk_f16_wide(*args, k, None, None, None, oi, ov)
        torch.cuda.synchronize()
        _capi.lib.spex_debug_tf_stats(C.c_void_p(0))
        st = stats.tolist()
        ws = int(_capi.call("spex_score_topk_f16_wide_workspace_bytes", b_pad, k))
        wide = lambda: ops.score_topk_f16_wide(*args, k, None, None, None, oi, ov)  # noqa: E731
        if k in f32_ks:
            # alternated with the fp32 scorer on the same inputs (fp32 tables, as its callers pass them)
            fi = torch.empty(n_u, k, dtype=torch.int32, device=dev)
            for rnd in range(2):
                ms_w = timed(wide, reps)
                rate("f16_wide", k, ms_w, round=rnd, workspace_bytes=ws)
                t32 = timed(lambda: fi.copy_(ops.score_topk_f32(U, I, users, k)[0]), 1)
                rate("f32", k, t32, round=rnd)
            agree = float((fi == oi).float().mean())
            print(json.dumps({"D": D, "k": k, "ids_equal_f16_wide_vs_f32": agree}), flush=True)
        else:
            rate("f16_wide", k, timed(wide, reps), workspace_bytes=ws)
        print(json.dumps({"D": D, "k": k, "compactions_per_warp": st[3] / nw, "exact_per_warp": st[4] / nw,
                          "fast_per_warp": (st[3] - st[4]) / nw, "compaction_cycles_per_warp": st[5] / nw,
                          "slow_tiles_frac": st[0] / (nw * (m_pad // 128))}), flush=True)
    return rows


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--users", type=int, default=148 * 2 * 128)
    ap.add_argument("--items", type=int, default=5_000_000)
    ap.add_argument("--reps", type=int, default=3)
    a = ap.parse_args()
    print(json.dumps({"card": card(), "users": a.users, "items": a.items}), flush=True)
    run(64, a.users, a.items, a.reps, (65, 100, 128, 256, 512), (100, 128))
    run(128, a.users, a.items, a.reps, (100, 512), (100,))
    print(json.dumps({"card_after": card()}), flush=True)


if __name__ == "__main__":
    main()
