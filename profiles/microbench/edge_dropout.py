"""edge_dropout.py — what edge dropout costs on the configs[3] graph (10 M users x 5 M items, 2e9 edges, D=64, K=3).

Reports, for the counter-based device mask (--dropout 2, spex_edge_dropout_f32):
  1. the kernel alone, val and valT written, no tpos (the synthetic graph's values are symmetric bit for bit):
     16 B per edge (col, val in; val, valT out) + 8 B per row, against the HBM copy peak (DESIGN.md §4);
  2. the receptive-field training step as bench.py's bench_train_step runs it (persistent workspaces, B=256, Adam):
     without dropout and with device dropout at keep_prob 0.3, arms alternated, 3 runs each, median;
  3. over all edges: the kept fraction, and the fraction of interactions kept in both directions, against kp^2;
  4. at --scale <= 0.01 only: the reference-stream path for contrast (CPU torch.rand(nnz), mask, host-to-device
     copy, the two gathers; tpos built on the host first and timed separately).
Run on a B200:  python profiles/microbench/edge_dropout.py [--scale 1.0] [--out FILE]
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from bench import K_LAYERS, sample_train_batch  # noqa: E402
from spex_b200 import ops, synthetic  # noqa: E402
from spex_b200.graph import CSRGraph, transpose_positions  # noqa: E402

HBM_COPY_PEAK_GBPS = 6547.5   # DESIGN.md §4 (MEASURED_PEAKS.json)
D = 64


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i",
                        "0"], capture_output=True, text=True, timeout=30).stdout.strip()
    return q or torch.cuda.get_device_name(0)


def events_ms(fn, reps):
    fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--scale", type=float, default=1.0)
    ap.add_argument("--keep-prob", type=float, default=0.3)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r05_edge_dropout.txt"))
    args = ap.parse_args()
    dev = torch.device("cuda:0")
    kp = args.keep_prob
    lines = []

    def emit(key, value):
        s = json.dumps({key: value})
        print(s, flush=True)
        lines.append(s)

    emit("card", card())
    nu, m, ni = int(10_000_000 * args.scale), int(5_000_000 * args.scale), int(1_000_000_000 * args.scale)
    keys = synthetic.generate_interactions(nu, m, ni, seed=2020, device=dev)
    g, _, _ = synthetic.build_norm_adj_device(keys, nu, m)
    del keys
    g.mark_hot_columns(D)
    nur = nu + 1
    emit("workload", f"{nu} users x {m} items, nnz(A)={g.nnz}, D={D}, K={K_LAYERS}, keep_prob={kp}")

    # 1. the kernel alone
    seed = [1]

    def kernel():
        seed[0] += 1
        return g.device_dropout_values(seed[0], kp)

    val, valT = kernel()
    del val, valT
    ms = events_ms(kernel, 5)
    nbytes = 16 * g.nnz + 8 * (g.n_rows + 1)
    gbps = nbytes / ms / 1e6
    emit("kernel", {"ms": round(ms, 3), "bytes": nbytes, "GBps": round(gbps, 1),
                    "frac_of_hbm_copy_peak": round(gbps / HBM_COPY_PEAK_GBPS, 3),
                    "note": "events over 5 launches, fresh seed each; the traffic is larger than the 126 MB L2, no flush"})

    # 3. statistics over every edge (each interaction is stored twice, so the both-ways fraction over all edges
    #    is the fraction over interactions)
    val, valT = g.device_dropout_values(2020, kp)
    kv, kt = val != 0, valT != 0
    n = g.nnz
    kept = int(kv.sum())
    both = int((kv & kt).sum())
    emit("mask", {"edges": n, "kept_fraction": kept / n, "kept_sigma": ((kp * (1 - kp) / n) ** 0.5),
                  "both_ways_fraction": both / n, "kp_squared": kp * kp,
                  "both_sigma": ((kp * kp * (1 - kp * kp) / n) ** 0.5)})
    del val, valT, kv, kt

    # 2. receptive-field training step, no dropout vs device dropout, alternated
    ops.enable_persistent_workspaces(True)
    W = synthetic.xavier_table(nur, m, D, 2020, dev).requires_grad_(True)
    mom, var = torch.zeros_like(W), torch.zeros_like(W)
    gen = torch.Generator(device=dev)
    gen.manual_seed(11)
    users, items, labels = sample_train_batch(torch, g, nur, m, 256, gen)
    rows = torch.cat([users, items + nur])
    step_no = [0]

    def train_step(dropout):
        W.grad = None
        val = valT = None
        if dropout:
            seed[0] += 1
            val, valT = g.device_dropout_values(seed[0], kp)
        out = ops.propagate_mean(W, g, K_LAYERS, val, valT, rows_needed=rows)
        loss = ops.bce_loss(out, nur, users, items, labels)
        loss.backward()
        step_no[0] += 1
        ops.adam_step(W.data, W.grad, mom, var, 1e-3, 0.9, 0.999, 1e-8, step_no[0])

    runs = {False: [], True: []}
    for arm in (False, True):   # warm both shapes
        for _ in range(2):
            train_step(arm)
    for _ in range(3):
        for arm in (False, True):
            runs[arm].append(events_ms(lambda: train_step(arm), 4))
    base, drop = statistics.median(runs[False]), statistics.median(runs[True])
    emit("train_step", {"no_dropout_ms": [round(x, 2) for x in runs[False]],
                        "device_dropout_ms": [round(x, 2) for x in runs[True]],
                        "median_no_dropout_ms": round(base, 2), "median_device_dropout_ms": round(drop, 2),
                        "overhead_ms": round(drop - base, 2),
                        "note": "4 steps per run, events; arms alternated; B=256, receptive field, Adam"})
    ops.enable_persistent_workspaces(False)
    del W, mom, var

    # 4. the reference-stream path for contrast (host RNG + mask + copy + gathers), small graphs only
    if args.scale <= 0.01:
        t0 = time.perf_counter()
        host = CSRGraph(g.n_rows, g.n_cols, g.rowptr.cpu().numpy(), g.clean_col().cpu().numpy(), g.val.cpu().numpy())
        g.tpos = torch.from_numpy(transpose_positions(host)).to(dev)
        torch.cuda.synchronize()
        t_tpos = time.perf_counter() - t0

        def host_path():
            keep = (torch.rand(g.nnz) + kp).int().bool()
            v = g.dropout_values(keep, kp)
            return v, g.transposed_values(v)

        host_path()
        torch.cuda.synchronize()
        ts = []
        for _ in range(3):
            t0 = time.perf_counter()
            host_path()
            torch.cuda.synchronize()
            ts.append((time.perf_counter() - t0) * 1e3)
        g.tpos = None
        dev_ms = events_ms(kernel, 5)
        emit("host_mask_path", {"ms_per_step": [round(x, 2) for x in ts], "tpos_build_s": round(t_tpos, 2),
                                "device_kernel_ms": round(dev_ms, 3),
                                "note": "host clock around work ending in a synchronise; tpos built once per graph"})

    with open(args.out, "w") as f:
        f.write(f"# python profiles/microbench/edge_dropout.py --scale {args.scale}\n")
        f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
