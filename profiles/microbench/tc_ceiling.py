"""Bring-up: time the tcgen05 scorer on the bench shape (37 888 users x 5 M items, k=20)."""
import os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__)))))
import torch
from spex_b200 import ops

dev = torch.device("cuda:0")
torch.manual_seed(0)
n_u, m, D = 148 * 2 * 128, int(os.environ.get("M_ITEMS", 5_000_000)), 64
U = torch.randn(n_u, D, device=dev) * 0.1
I = torch.randn(m, D, device=dev) * 0.1
users = torch.arange(n_u, device=dev)
Ib, m_pad = ops.pack_bf16(I, None, ops.TC_ITEM_MULTIPLE)
Ub, b_pad = ops.pack_bf16(U, users, ops.TC_USER_MULTIPLE)
for _ in range(2):
    ops.score_topk_bf16(Ub, n_u, b_pad, Ib, m, m_pad, 20, users, None, None)
torch.cuda.synchronize()
e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
e0.record()
for _ in range(3):
    ops.score_topk_bf16(Ub, n_u, b_pad, Ib, m, m_pad, 20, users, None, None)
e1.record()
torch.cuda.synchronize()
ms = e0.elapsed_time(e1) / 3
print(f"{ms:.2f} ms  {2.0 * n_u * m * D / ms / 1e9:.0f} TFLOP/s")

if os.environ.get("CLOCKS"):
    # SM clock and board power while the scorer runs back to back for ~1.5 s
    import subprocess, time
    p = subprocess.Popen(["nvidia-smi", "--query-gpu=clocks.sm,power.draw,clocks_event_reasons.active",
                          "--format=csv,noheader", "-lms", "100"], stdout=subprocess.PIPE, text=True)
    time.sleep(0.3)
    e0.record()
    for _ in range(60):
        ops.score_topk_bf16(Ub, n_u, b_pad, Ib, m, m_pad, 20, users, None, None)
    e1.record()
    torch.cuda.synchronize()
    time.sleep(0.1)
    p.terminate()
    out = p.communicate()[0].strip().splitlines()
    ms = e0.elapsed_time(e1) / 60
    print(f"sustained 60 launches: {ms:.2f} ms each, {2.0 * n_u * m * D / ms / 1e9:.0f} TFLOP/s")
    print("clocks.sm, power, reasons:", " | ".join(out[2:14]))
