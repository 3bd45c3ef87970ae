"""Probe the column-blocked long-row plan on the 1B-interaction graph: per-block statistics and the
throughput of the segment kernel on sub-ranges of the segment list."""
import os, sys, ctypes as C
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__)))))
import torch
from spex_b200 import ops, synthetic, _capi
from spex_b200._capi import LongPlan, call, ptr, stream_ptr

dev = torch.device("cuda:0")
scale = float(sys.argv[1]) if len(sys.argv) > 1 else 1.0
nu, m, ni = int(10_000_000 * scale), int(5_000_000 * scale), int(1_000_000_000 * scale)
keys = synthetic.generate_interactions(nu, m, ni, seed=2020, device=dev)
g, _, _ = synthetic.build_norm_adj_device(keys, nu, m)
del keys
D = 64
N = g.n_rows
X = synthetic.xavier_table(nu + 1, m, D, 1, dev)
print("n_long", g.n_long, "n_seg", g.n_seg, "blocked", g.n_hub_seg > 0)
cnt = g.seg_count.long()
print("segment edges: mean %.1f  median %d  p90 %d  max %d  total %d" % (
    cnt.float().mean(), cnt.median(), cnt.float().quantile(0.9), cnt.max(), cnt.sum()))
first_col = g.col[g.seg_start].long()
blk = first_col // (ops.DeviceGraph.L2_WINDOW_BYTES // (D * 4))
print("segments are block-major:", bool((blk[1:] >= blk[:-1]).all()), "blocks used", int(blk.max()) + 1)
nb = int(blk.max()) + 1
seg_per_blk = torch.bincount(blk, minlength=nb)
edges_per_blk = torch.bincount(blk, weights=cnt.double(), minlength=nb)
print("segments per block: min %d max %d ; edges per block: min %.3g max %.3g" % (
    seg_per_blk.min(), seg_per_blk.max(), edges_per_blk.min(), edges_per_blk.max()))
partial = torch.empty(g.n_seg * D, dtype=torch.float32, device=dev)
lib = _capi.lib

def run(s0, s1, reps=3):
    """time spex's segment kernel on segments [s0, s1) through a plan whose lists are offset"""
    n = s1 - s0
    # a plan with only these segments: reuse the fix kernel trivially (n_long = 1 dummy) is awkward, so time
    # the full SpMM API on a CSR made of the segments as rows instead (same gathers, same order)
    rowptr = torch.zeros(n + 1, dtype=torch.int64, device=dev)
    rowptr[1:] = torch.cumsum(cnt[s0:s1], 0)
    idx = torch.repeat_interleave(g.seg_start[s0:s1], cnt[s0:s1]) + (
        torch.arange(int(rowptr[-1]), device=dev) - torch.repeat_interleave(rowptr[:-1], cnt[s0:s1]))
    col = g.col[idx].contiguous()
    val = g.val[idx].contiguous()
    G = ops.DeviceGraph(rowptr, col, val, N)
    Y = torch.empty(n, D, device=dev)
    ops.spmm(G, X, Y=Y)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        ops.spmm(G, X, Y=Y)
    e1.record(); torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / reps
    edges = int(rowptr[-1])
    return ms, edges, (edges * 264 + n * 264) / ms / 1e6

bounds = torch.searchsorted(blk, torch.arange(nb + 1, device=dev)).tolist()
for b in (0, 10, 40):
    ms, e, gbs = run(bounds[b], bounds[b + 1])
    print(f"block {b}: {bounds[b+1]-bounds[b]} segments, {e} edges, {ms:.3f} ms, {gbs:.0f} GB/s algorithmic")
ms, e, gbs = run(bounds[0], bounds[8])
print(f"blocks 0-7 together: {e} edges, {ms:.3f} ms, {gbs:.0f} GB/s algorithmic")
# same segments but in ROW-major (random window) order for contrast
