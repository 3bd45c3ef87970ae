#!/usr/bin/env python
"""bench.py — LightGCN_SPEX propagation throughput (GEdges/s) + full-rank top-20 users/s on B200.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--scale S] [--dump-outputs DIR]

One "step" = one computer() forward of the reference model
(/root/reference/LightGCN_SPEX/code/utility1/model.py:66-97): K_layers = 3 propagation layers over
the normalised adjacency + layer mean, D = 64, fp32.  Workload (BASELINE.json configs[3]): synthetic
10 M users x 5 M items, ~10^9 interaction edges => nnz(A) ~ 2*10^9 (both directions are stored and
processed, dataloader.py:200-201).  Metric: GEdges/s = nnz(A) * K_layers / t_step, whole job.

N > 1 (torchrun, one rank per GPU): the graph is row-partitioned by nnz, each layer ends with an
exchange of the embedding slices over NVLink (strong scaling: the graph is fixed).

JSON keys beyond the base contract:
  roofline      dominant kernel (CSR SpMM): algorithmic bytes per launch (nnz+N)*264 (DESIGN.md §4)
                / CUDA-event time per launch, against MEASURED_PEAKS.json hbm_gbs
  cpu_baseline  the CPU oracle (torch.sparse.mm path, the reference's own backend) on a bounded sample
  e2e           same metric through the public API with HOST tables: H2D of the fused embedding
                table and D2H of the propagated table inside the timed region
  eval          secondary metric: full-ranking top-20 users/s (tcgen05 scoring GEMM + mask + top-k)
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

G_USERS, G_ITEMS, G_INTER = 10_000_000, 5_000_000, 1_000_000_000
D, K_LAYERS, TOPK = 64, 3, 20
METRIC, UNIT = "lightgcn_propagation_gedges_per_s", "GEdges/s"


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--scale", type=float, default=1.0, help="fraction of the 10M x 5M x 1B workload")
    ap.add_argument("--exchange", default=os.environ.get("SPEX_EXCHANGE", "auto"),
                    choices=["auto", "nccl", "push", "mcast"],
                    help="auto = mcast (NVLS multicast stores) when the box supports it, else push")
    ap.add_argument("--e0-exchange", default=os.environ.get("SPEX_E0_EXCHANGE"), choices=["nccl", "push", "copy", "mcast"],
                    help="how E^(0) is all-gathered in push / mcast mode")
    ap.add_argument("--eval-users", type=int, default=0,
                    help="users ranked by the evaluation sweep, whole job (0 = all users of the workload)")
    ap.add_argument("--eval-scorer", default="f16", choices=["f16", "bf16"],
                    help="f16: fp16-accumulator filter + exact re-score (r02); bf16: round 1's fp32-accumulator kernel")
    ap.add_argument("--no-train", action="store_true")
    ap.add_argument("--no-small-configs", action="store_true", help="skip the configs[1] / configs[2] legs")
    ap.add_argument("--train-batch", type=int, default=256, help="samples per train step (main_rec.py:20: 256)")
    ap.add_argument("--loss-bench-batch", type=int, default=1 << 20,
                    help="batch on which the loss / scatter kernels are timed alone for their rooflines")
    ap.add_argument("--no-eval", action="store_true")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--cpu-sample-scale", type=float, default=0.01)
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the last timed step returned to DIR/*.npy (see dump_outputs), so that two builds "
                         "can be compared output for output")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be >= 1 and --warmup >= 0")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs dumps the GPU step (--impl ours)")
    return args


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        j = json.load(open(p))
        return j["hbm_gbs"], j["bf16_tflops"], j.get("bf16_tflops_sustained", j["bf16_tflops"]), "measured"
    return 6650.0, 1590.0, 1400.0, "fallback"


def profile_metric(names, key):
    """Sum of metric `key` (a byte count) over the kernels named in `names`, from the newest committed ncu
    summary that lists them all with that metric; None if there is none."""
    import glob

    unit = {"byte": 1.0, "Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9, "Tbyte": 1e12}
    for path in sorted(glob.glob(os.path.join(ROOT, "profiles", "r*_ncu_*.json")), reverse=True):
        try:
            rows = json.load(open(path))
        except Exception:
            continue
        tot, seen = 0.0, set()
        for r in rows:
            kn = r.get("Kernel Name", "")
            hit = next((n for n in names if n in kn), None)
            if hit is None or hit in seen or key not in r:
                continue
            try:
                v, u = r[key].split()
                tot += float(v) * unit[u]
            except Exception:
                break
            seen.add(hit)
        if len(seen) == len(names):
            return tot
    return None


def profile_traffic(names):
    """DRAM bytes (read + write) of the kernels whose name contains one of `names`, summed, from the newest
    ncu summary under profiles/ that lists them all (profiles/ncu_summary.py output); (None, None) if there is
    none.  The bench line reports it as profile-derived, with the file name, never as measured by this run."""
    import glob
    import re

    unit = {"byte": 1.0, "Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9, "Tbyte": 1e12}
    for path in sorted(glob.glob(os.path.join(ROOT, "profiles", "r*_ncu_*.json")), reverse=True):
        try:
            rows = json.load(open(path))
        except Exception:
            continue
        tot, seen = 0.0, set()
        for r in rows:
            kn = r.get("Kernel Name", "")
            hit = next((n for n in names if n in kn), None)
            if hit is None or hit in seen:
                continue
            try:
                for key in ("dram__bytes_read.sum", "dram__bytes_write.sum"):
                    v, u = r[key].split()
                    tot += float(v) * unit[u]
            except Exception:
                break
            seen.add(hit)
        if len(seen) == len(names):
            return tot, os.path.relpath(path, ROOT)
    return None, None


def workload(scale):
    return (max(int(G_USERS * scale), 1000), max(int(G_ITEMS * scale), 500),
            max(int(G_INTER * scale), 10000))


# ---- clocks sampling ---------------------------------------------------------------------------------
class Clocks:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        self.p = None
        try:
            self.p = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                       "-lms", "200", "-i", str(gpu_index)], stdout=self.f,
                                      stderr=subprocess.DEVNULL)
        except OSError:
            self.p = None
        self.t0 = self.t1 = None

    def mark(self, start):
        if start:
            self.t0 = time.time()
        else:
            self.t1 = time.time()

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": []}
        if self.p is None:
            return out
        time.sleep(0.25)
        self.p.terminate()
        try:
            self.p.wait(timeout=5)
        except subprocess.TimeoutExpired:
            self.p.kill()
        self.f.flush()
        self.f.seek(0)
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for line in self.f.read().splitlines():
            c = [x.strip() for x in line.split(",")]
            if len(c) < 9:
                continue
            try:
                sm.append(float(c[1]))
                mx.append(float(c[2]))
            except ValueError:
                continue
            for n, v in zip(names, c[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        os.unlink(self.f.name)
        if sm:
            # the sampler runs over the whole timed phase; under-load samples dominate the upper half
            s = sorted(sm)
            out["sm_mhz"] = s[len(s) // 2]
            out["sm_max_mhz"] = max(mx)
            out["samples"] = len(sm)
        out["reasons"] = sorted(reasons)
        return out


def pin_to_gpu_numa(gpu_index):
    """Run this rank (and first-touch its pinned host buffers) on the CPUs local to its GPU, so that
    the e2e host<->device copies of the ranks do not all cross one NUMA node.  Returns the cpulist."""
    try:
        bus = subprocess.run(["nvidia-smi", "--query-gpu=pci.bus_id", "--format=csv,noheader", "-i", str(gpu_index)],
                             capture_output=True, text=True, timeout=20).stdout.strip().lower()
        if not bus:
            return None
        if bus.count(":") == 2 and len(bus.split(":")[0]) == 8:   # 00000000:1B:00.0 -> 0000:1b:00.0
            bus = bus[4:]
        path = f"/sys/bus/pci/devices/{bus}/local_cpulist"
        if not os.path.exists(path):
            return None
        txt = open(path).read().strip()
        cpus = set()
        for part in txt.split(","):
            if "-" in part:
                a, b = part.split("-")
                cpus.update(range(int(a), int(b) + 1))
            elif part:
                cpus.add(int(part))
        cpus &= set(os.sched_getaffinity(0))
        if cpus:
            os.sched_setaffinity(0, cpus)
            return txt
    except Exception:
        return None
    return None


def table_hash(t, row0, torch):
    """Order-independent 64-bit checksum of an fp32 [rows, D] slice whose first row is global row `row0`:
    sum over elements of bits * (1 + global element index) mod 2^64 (int64 wrap-around).  Equal at every N
    iff the propagated tables are bit-identical."""
    D = t.shape[1]
    h = torch.zeros((), dtype=torch.int64, device=t.device)
    step = 1 << 22
    for a in range(0, t.shape[0], step):
        x = t[a: a + step].contiguous().view(torch.int32).to(torch.int64)
        idx = (torch.arange(x.shape[0], device=t.device, dtype=torch.int64) + (row0 + a))[:, None] * D + \
            torch.arange(1, D + 1, device=t.device, dtype=torch.int64)[None, :]
        h += (x * idx).sum()
    return h


DUMP_ROWS = 1 << 17   # 32 MB of fp32 rows at D = 64: the whole dump stays under 64 MB


def dump_outputs(path, res, bounds, rank, world, torch, dist):
    """Write what the timed step returned (the propagated [N, D] fp32 table; this rank holds global rows
    bounds[rank]:bounds[rank + 1] of it) to `path`, on rank 0:
      propagated_sample.npy       fp32 [S, D]  S = min(N, DUMP_ROWS) rows drawn with seed 0, in row order
      propagated_sample_rows.npy  fp64 [S]     their global row ids
      propagated_col_sum.npy      fp64 [D]     column sums over all N rows, so that no row goes unchecked
    The inputs are seeded, so the same arguments give the same files on the same build."""
    import numpy as np

    n_rows = bounds[-1]
    rows = np.sort(np.random.default_rng(0).choice(n_rows, min(n_rows, DUMP_ROWS), replace=False))
    owner = np.searchsorted(bounds, rows, side="right") - 1
    dev = res.device
    sample = torch.zeros(rows.size, res.shape[1], dtype=res.dtype, device=dev)
    mine = owner == rank
    sample[torch.from_numpy(mine).to(dev)] = res[torch.from_numpy(rows[mine] - bounds[rank]).to(dev)]
    col_sum = res.sum(0, dtype=torch.float64)
    if world > 1:
        parts = torch.empty(world * rows.size, res.shape[1], dtype=res.dtype, device=dev)
        dist.all_gather_into_tensor(parts, sample)
        sample = parts.view(world, rows.size, -1)[torch.from_numpy(owner).to(dev), torch.arange(rows.size, device=dev)]
        dist.all_reduce(col_sum)
    if rank == 0:
        os.makedirs(path, exist_ok=True)
        np.save(os.path.join(path, "propagated_sample.npy"), sample.cpu().numpy())
        np.save(os.path.join(path, "propagated_sample_rows.npy"), rows.astype(np.float64))
        np.save(os.path.join(path, "propagated_col_sum.npy"), col_sum.cpu().numpy())


# ---- CPU legs (oracle = the reference's torch CPU path restated; the checker, not the product) -------
def cpu_sample_graph(scale):
    import numpy as np
    from oracle import lightgcn_oracle as O

    nu, m, ni = workload(scale)
    u, i = O.random_bipartite(nu, m, ni, 2020)
    A = O.to_sparse_tensor(O.norm_adj_scipy(u, i, nu + 1, m))
    return A, nu, m


def cpu_time_computer(A, nu, m, steps, warmup):
    import torch
    from oracle import lightgcn_oracle as O

    torch.manual_seed(2020)
    uw = torch.empty(nu + 1, D)
    iw = torch.empty(m, D)
    torch.nn.init.xavier_uniform_(uw)
    torch.nn.init.xavier_uniform_(iw)
    with torch.no_grad():
        for _ in range(warmup):
            O.computer(uw, iw, A, K_LAYERS)
        t0 = time.perf_counter()
        for _ in range(steps):
            O.computer(uw, iw, A, K_LAYERS)
        dt = (time.perf_counter() - t0) / steps
    return A._nnz() * K_LAYERS / dt / 1e9, dt


def run_reference(args):
    """--impl reference: the reference's own CPU implementation of the path (oracle port of
    model.py:66-97, same torch.sparse.mm backend) on all host threads, bounded sample."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import torch

    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    A, nu, m = cpu_sample_graph(args.cpu_sample_scale)
    ge, dt = cpu_time_computer(A, nu, m, args.steps, max(args.warmup, 1))
    sample = (f"computer() K={K_LAYERS} D={D} on {nu} users x {m} items, nnz(A)={A._nnz()} "
              f"({args.cpu_sample_scale:g} of the 10Mx5Mx1B workload), uniform synthetic")
    line = {
        "impl": "reference", "metric": METRIC, "value": ge, "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt * 1e3, "higher_is_better": True,
        "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": f"synthetic {G_USERS} users x {G_ITEMS} items, {G_INTER} interactions, D={D}, "
                               f"K={K_LAYERS} (BASELINE.json configs[3]) - timed on a bounded sample of it",
                   "sample": sample, "parallelism": f"{cores} host threads (torch.sparse.mm)"},
        "cpu_baseline": {"value": ge, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": ge, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ---- BASELINE.json configs[1] and configs[2]: small graphs, timed through the drop-in model classes --------
def bench_small_configs(torch, dev):
    """configs[1]: LightGCN_SPEX main_11.py rec + path multi-task step on a weibo-shaped synthetic graph
    (6 812 users, Trust_SPEX/code/main_trust.py:41-42; items and density from epinion2's ratios, SURVEY §8d;
    50 random trust paths of 2-5 hops per user, data_process_path.py:14-15).
    configs[2]: NGCF_SPEX propagation (SpMM + W1/W2 layer) on a twitter-shaped synthetic graph (8 930 users,
    main_trust.py:43-44): fused inference forward, training step (forward + BCE + backward + Adam on the
    library's kernels), and full ranking of every user on the tcgen05 scorer at D = 128."""
    import argparse

    import numpy as np

    from spex_b200 import ops as ops_
    from spex_b200.dataloader import SyntheticDataset
    from spex_b200.optim import FusedAdam

    def timed(fn, reps, warm=2):
        for _ in range(warm):
            fn()
        torch.cuda.synchronize()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(reps):
            fn()
        b.record()
        torch.cuda.synchronize()
        return a.elapsed_time(b) / reps

    out = {}
    rng = np.random.default_rng(2020)
    # ---- configs[1] ----
    from spex_b200.model_expert_s import LightGCN as LightGCNExpert
    from spex_b200.path_data import Data

    nu = 6812
    m = int(nu * 3.9)
    ds = SyntheticDataset(nu, m, nu * 66, seed=2020)
    args = argparse.Namespace(recdim=64, layer=3, keepprob=0.6, A_split=0, dropout=0, a_fold=1, dataset="weibo-shaped",
                              lr=1e-3, seed=2020, hiddenSize=64, nb_heads=3, batchSize=256, nonhybrid=False, act="relu",
                              batch_size=256)
    torch.manual_seed(2020)
    model = LightGCNExpert(args, ds).to(dev)
    paths = [[int(x) for x in rng.integers(0, nu, rng.integers(2, 6))] for _ in range(nu * 50)]
    targets = rng.integers(0, nu, len(paths)).tolist()
    trust = Data((paths, targets), nu, shuffle=False)
    by_user = {}
    for i, pth in enumerate(paths):
        by_user.setdefault(pth[0], []).append(i)
    opt = FusedAdam(model.parameters(), lr=1e-3)
    B = 256
    users = torch.from_numpy(rng.integers(0, nu, B)).to(dev)
    items = torch.from_numpy(rng.integers(0, m, B)).to(dev)
    labels = torch.from_numpy((rng.random(B) < 1 / 6).astype(np.float32)).to(dev)
    n_batches = -(-(ds.trainDataSize * 6) // B)
    tbs = max(len(paths) // n_batches, 1)
    idx = []
    for u in set(users.tolist()):
        idx.extend(by_user.get(u, []))
    idx = np.array(sorted(idx)[:tbs], dtype=int)

    def step11():
        model.train()
        opt.zero_grad(set_to_none=True)
        l1, l2 = model(users=users, items=items, labels=labels, slice_indices=idx, trust_data=trust, flag=0)
        (l1 + l2).backward()
        opt.step()

    def prop11():
        with torch.no_grad():
            model.computer()

    ms_step = timed(step11, 5)
    ms_prop = timed(prop11, 10)
    nnz = int(model.device_graph().nnz)
    out["configs[1] main_11 weibo-shaped"] = {
        "workload": f"{nu} users x {m} items, {ds.trainDataSize} interactions (nnz(A)={nnz}), {len(paths)} trust paths, "
                    f"batch {B} + {idx.size} paths", "train_step_ms": round(ms_step, 3),
        "computer_forward_ms": round(ms_prop, 4), "computer_gedges_per_s": nnz * 3 / (ms_prop * 1e-3) / 1e9,
        "note": "the path branch (GraphAttentionLayer python loops, utility2/layers.py:19-40) is host-loop bound and out "
                "of scope as a kernel target (SURVEY §2); it dominates the step"}
    del model, opt, trust
    # ---- configs[2] ----
    from spex_b200.ngcf import Model_Wrapper, build_ngcf_norm_adj

    nu2 = 8930
    m2 = int(nu2 * 3.9)
    ds2 = SyntheticDataset(nu2, m2, nu2 * 66, seed=2021, with_test=False)
    adj = build_ngcf_norm_adj(ds2.trainUser, ds2.trainItem, nu2, m2)
    torch.manual_seed(2020)
    ng = Model_Wrapper({"n_users": nu2, "n_items": m2, "norm_adj": adj}, dev).to(dev)
    opt2 = FusedAdam(ng.parameters(), lr=1e-3)
    bu = rng.integers(0, nu2, 1024)
    bi = rng.integers(0, m2, 1024)
    bl = (rng.random(1024) < 1 / 6).astype(np.float32)

    def ngcf_infer():
        ng.eval()
        with torch.no_grad():
            ng(None, None, None, 1)

    def ngcf_train():
        ng.train()
        opt2.zero_grad(set_to_none=True)
        loss = ng(bu, bi, bl, 0)
        loss.backward()
        opt2.step()

    def ngcf_rank():
        ng.eval()
        ng.rank_topk(torch.arange(nu2, device=dev), k=20)

    def ngcf_rank_tc():
        ng.eval()
        ng.rank_topk(torch.arange(nu2, device=dev), k=20, probe=False)

    ms_inf = timed(ngcf_infer, 10)
    ms_tr = timed(ngcf_train, 5)
    ms_rank = timed(ngcf_rank, 3)
    ms_rank_tc = timed(ngcf_rank_tc, 2, warm=1)
    ng.eval()
    with torch.no_grad():
        ua_, ia_ = ng.propagate()
        selective = ops_.f16_filter_is_selective(ua_.contiguous(), ia_.contiguous(), torch.arange(nu2, device=dev))
    out["configs[2] NGCF twitter-shaped"] = {
        "workload": f"{nu2} users x {m2} items, {ds2.trainDataSize} interactions, nnz(D^-1(A+I))={adj.nnz}, 1 layer, "
                    "outputs [N, 128]", "propagation_forward_ms": round(ms_inf, 4),
        "propagation_gedges_per_s": adj.nnz / (ms_inf * 1e-3) / 1e9, "train_step_ms_batch1024": round(ms_tr, 3),
        "fullrank_top20_all_users_ms": round(ms_rank, 3), "fullrank_users_per_s": nu2 / (ms_rank * 1e-3),
        "fullrank_scorer": "f16 tcgen05 (D=128)" if selective else "exact fp32 (the near-tie probe routed it: the random-init "
                           "model's normalised outputs are almost parallel, every score ties within the fp16 filter band)",
        "fullrank_top20_forced_tcgen05_ms": round(ms_rank_tc, 3),
        "scorer_tflops_d128": 2.0 * nu2 * m2 * 128 / (ms_rank * 1e-3) / 1e12}
    return out


# ---- training step -------------------------------------------------------------------------------------
def sample_train_batch(torch, g, nur, m, n, gen):
    """n samples drawn like the reference (LightGCN_SPEX/code/utility1/dataloader.py:250-265): users uniform, one
    positive per user uniform among the user's interactions (so popular items are drawn often) + 5 rejection-
    sampled negatives (device sampler).  Needs the full adjacency `g` on the device."""
    from spex_b200.dataloader import sample_negatives_device

    dev = g.rowptr.device
    nu = nur - 1
    u = torch.randint(0, nu, (n // 6 + 1,), device=dev, generator=gen)
    e = g.rowptr[u] + (torch.rand(u.numel(), device=dev, generator=gen) * (g.rowptr[u + 1] - g.rowptr[u])).long()
    pos = (g.col[e] & 0x7FFFFFFF).long() - nur
    neg = sample_negatives_device(g.rowptr, g.col, nur, m, u, 5, seed=int(n) + 1)
    users = torch.cat([u, u.repeat_interleave(5)])[:n].contiguous()
    items = torch.cat([pos, neg.reshape(-1)])[:n].contiguous()
    labels = torch.cat([torch.ones_like(u), torch.zeros(u.numel() * 5, dtype=u.dtype, device=dev)])[:n]
    return users, items, labels.float().contiguous()


def bench_train_step(args, torch, ops, _capi, g, table, nur, m, N, hbm_peak, peak_kind, dev):
    """One optimiser step of the reference loop (LightGCN_SPEX/code/main_rec.py:30-37) on the bench graph:
    computer() forward, gather + dot + BCEWithLogits, backward (deterministic scatter, K A^T SpMMs), dense
    Adam over the fused table - through the public operators, persistent workspaces on.  Per-phase CUDA
    events, and the loss / scatter / Adam / dropout-value kernels timed alone on a large batch for their
    HBM rooflines (algorithmic bytes per sample or element as in DESIGN.md §4)."""
    ops.enable_persistent_workspaces(True)
    W = table.clone().requires_grad_(True)
    mom, var = torch.zeros_like(W), torch.zeros_like(W)
    gen = torch.Generator(device=dev)
    gen.manual_seed(11)
    B = args.train_batch
    nu = nur - 1

    def batch(n):
        return sample_train_batch(torch, g, nur, m, n, gen)

    def ev():
        e = torch.cuda.Event(enable_timing=True)
        e.record()
        return e

    step_no = [0]

    def train_step(users, items, labels, marks=None, receptive=True):
        W.grad = None
        t0 = ev() if marks is not None else None
        # receptive=True is what spex_b200.model.LightGCN.forward does in training mode: every layer restricted
        # to the rows the batch depends on (bit-identical loss and gradients, tests/test_gpu_receptive.py);
        # receptive=False is the reference's literal step: computer() over all N rows (main_rec.py:34)
        rows = torch.cat([users, items + nur]) if receptive else None
        out = ops.propagate_mean(W, g, K_LAYERS, rows_needed=rows)
        t1 = ev() if marks is not None else None
        loss = ops.bce_loss(out, nur, users, items, labels)
        t2 = ev() if marks is not None else None
        loss.backward()
        t3 = ev() if marks is not None else None
        step_no[0] += 1
        ops.adam_step(W.data, W.grad, mom, var, 1e-3, 0.9, 0.999, 1e-8, step_no[0])
        t4 = ev() if marks is not None else None
        if marks is not None:
            marks.append((t0, t1, t2, t3, t4))
        return loss

    users, items, labels = batch(B)

    def measure(receptive):
        for _ in range(2):
            train_step(users, items, labels, receptive=receptive)
        torch.cuda.synchronize()
        n_steps = 4
        e0 = ev()
        for _ in range(n_steps):
            loss = train_step(users, items, labels, receptive=receptive)
        e1 = ev()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / n_steps
        marks = []
        train_step(users, items, labels, marks, receptive=receptive)
        torch.cuda.synchronize()
        t0, t1, t2, t3, t4 = marks[0]
        ph = {"forward_propagate_ms": t0.elapsed_time(t1), "bce_forward_ms": t1.elapsed_time(t2),
              "backward_scatter_plus_propagate_ms": t2.elapsed_time(t3), "adam_ms": t3.elapsed_time(t4)}
        return ms, ph, float(loss.item())

    # both arms start from the same weights and moments, so their first timed losses are comparable
    W0 = W.detach().clone()
    ms_full, phases_full, loss_full = measure(False)
    W_full = W.detach().clone()          # weights after the 7 literal steps
    with torch.no_grad():
        W.copy_(W0)
        mom.zero_()
        var.zero_()
    step_no[0] = 0
    ms_step, phases, loss_val = measure(True)
    same_weights = bool(torch.equal(W.detach(), W_full))   # the same 7 steps on the receptive-field path: same bits
    del W0, W_full
    S_rows = torch.unique(torch.cat([users, items + nur]))
    R = ops.receptive_rows(g, S_rows, K_LAYERS)
    rf_rows = [None if r is None else int(r.numel()) for r in R[1:]]
    rf_edges = [None if r is None else g.degree_sum(r) for r in R[1:]]

    # kernels alone, large batch, with their algorithmic bytes
    def timed(fn, reps=5):
        fn()
        torch.cuda.synchronize()
        a = ev()
        for _ in range(reps):
            fn()
        b = ev()
        torch.cuda.synchronize()
        return a.elapsed_time(b) / reps

    Bl = args.loss_bench_batch
    ul, il, ll = batch(Bl)
    out = ops.propagate_mean(W.detach(), g, K_LAYERS)
    U, I = out[:nur], out[nur:]
    row = 4 * D
    gam = torch.empty(Bl, device=dev)
    dgam = torch.empty(Bl, device=dev)
    lo = torch.empty(1, device=dev)
    kern = {}
    ms = timed(lambda: _capi.call("spex_bce_fwd_f32", _capi.ptr(U), _capi.ptr(I), D, _capi.ptr(ul), _capi.ptr(il),
                                  _capi.ptr(ll), Bl, _capi.ptr(gam), _capi.ptr(lo), _capi.ptr(dgam), _capi.stream_ptr()))
    kern["bce_fwd_kernel"] = (ms, Bl * (2 * row + 16 + 4 + 8))
    gbuf = torch.zeros_like(out)
    work, wb = ops._scatter_workspace(Bl, dev)
    ms = timed(lambda: _capi.call("spex_bce_bwd_ws_f32", _capi.ptr(U), _capi.ptr(I), D, _capi.ptr(ul), _capi.ptr(il),
                                  _capi.ptr(dgam), None, Bl, _capi.ptr(gbuf[:nur]), _capi.ptr(gbuf[nur:]),
                                  _capi.ptr(work), wb, _capi.stream_ptr()))
    # two lists: each entry reads one row and its run writes one row; + sort traffic 2 x 4 passes x 16 B
    kern["scatter_sorted (keys + radix sort + scatter_sorted_kernel, x2 lists)"] = (ms, 2 * Bl * (2 * row + 16 + 128))
    pu, pp, pn = ul, il, torch.randint(0, m, (Bl,), device=dev, generator=gen)
    out2, dsc, wk = torch.empty(2, device=dev), torch.empty(Bl, device=dev), torch.empty(2 * Bl, device=dev)
    Wd = W.detach()
    ms = timed(lambda: _capi.call("spex_bpr_fwd_f32", _capi.ptr(U), _capi.ptr(I), _capi.ptr(Wd[:nur]), _capi.ptr(Wd[nur:]),
                                  D, _capi.ptr(pu), _capi.ptr(pp), _capi.ptr(pn), Bl, _capi.ptr(out2), _capi.ptr(dsc),
                                  _capi.ptr(wk), _capi.stream_ptr()))
    kern["bpr_fwd_kernel"] = (ms, Bl * (6 * row + 24 + 12))
    del gbuf
    gg = torch.empty_like(Wd)
    gg.normal_(generator=gen)
    ms = timed(lambda: ops.adam_step(Wd, gg, mom, var, 1e-3, 0.9, 0.999, 1e-8, 3))
    kern["adam_kernel"] = (ms, W.numel() * 28)
    del gg
    keep = torch.ones(g.nnz, device=dev)
    vout = torch.empty_like(g.val)
    ms = timed(lambda: _capi.call("spex_gather_f32", _capi.ptr(g.val), None, _capi.ptr(keep), 0.6, _capi.ptr(vout), g.nnz,
                                  _capi.stream_ptr()), reps=3)
    kern["gather_scale_kernel (edge-dropout values, model.py:46-55)"] = (ms, g.nnz * 12)
    del keep, vout
    roofs = {k: {"ms": round(v[0], 4), "algorithmic_bytes": v[1], "achieved": v[1] / v[0] / 1e6, "unit": "GB/s",
                 "peak": hbm_peak, "frac": v[1] / v[0] / 1e6 / hbm_peak, "peak_kind": peak_kind, "bound": "hbm"}
             for k, v in kern.items()}
    ops.enable_persistent_workspaces(False)
    return {"metric": "lightgcn_train_step_ms", "value": ms_step, "unit": "ms", "higher_is_better": False,
            "steps_per_s": 1e3 / ms_step, "batch": B, "loss": loss_val, "phases_ms": {k: round(v, 3) for k, v in phases.items()},
            "receptive_field": {"rows_per_layer": rf_rows, "edges_per_layer": rf_edges, "nnz": g.nnz,
                                "note": "layers 1..K of the forward restricted to the rows the batch depends on (null = "
                                        "all rows); the backward mirrors it and skips the gathers of rows known to be "
                                        "zero (x_nonzero masks); loss and gradients bit-identical to the full step"},
            "full_computer_step": {"value": ms_full, "unit": "ms", "loss": loss_full,
                                   "phases_ms": {k: round(v, 3) for k, v in phases_full.items()},
                                   "note": "the reference's literal step: computer() over all N rows in forward and "
                                           "backward (main_rec.py:34-35)", "same_loss_as_receptive_path": loss_full == loss_val,
                                   "same_weights_after_7_steps_as_receptive_path": same_weights},
            "config": {"workload": f"main_rec.py:30-37 step on the bench graph: forward(K={K_LAYERS}) + BCE (1 positive + 5 "
                                   f"negatives per user, device sampler) + backward + dense Adam over {N} x {D}",
                       "edges_per_step": 2 * K_LAYERS * g.nnz},
            # edges actually traversed per second: quoted on the FULL step (the receptive path skips edges)
            "gedges_per_s_fwd_plus_bwd": 2 * K_LAYERS * g.nnz / (ms_full * 1e-3) / 1e9,
            "kernel_rooflines": roofs, "loss_bench_batch": Bl}


# ---- our arm -----------------------------------------------------------------------------------------
def run_ours(args):
    import torch
    import torch.distributed as dist

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py (impl=ours) needs a B200: there is no CPU fallback")
    numa_cpus = pin_to_gpu_numa(local_rank) if world > 1 else None
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        # NCCL_DEBUG is left as the caller set it: the driver reads NCCL's own lines to count ranks
        dist.init_process_group("nccl", device_id=dev)

    from spex_b200 import ops, synthetic
    from spex_b200 import _capi
    from spex_b200.dist import PartitionedPropagator
    from spex_b200.graph import partition_rows_by_nnz, rebalance_bounds

    _capi.device_check()
    hbm_peak, tc_burst, tc_sust, peak_kind = peaks()
    nu, m, ni = workload(args.scale)
    nur = nu + 1
    N = nur + m

    t_gen = time.time()
    keys = synthetic.generate_interactions(nu, m, ni, seed=2020, device=dev)
    g, mask_rp, mask_col = synthetic.build_norm_adj_device(keys, nu, m)
    del keys
    n_hot = 0 if os.environ.get("SPEX_NO_HOT") else g.mark_hot_columns(
        D, budget_bytes=(int(os.environ["SPEX_HOT_MB"]) << 20) if os.environ.get("SPEX_HOT_MB") else None)
    # optional (SPEX_TWO_PASS=1, N = 1): hot edges of every user row in a first pass, cold edges in a
    # second one.  Measured slower than the single pass (197 vs 184 ms), so it is off by default.
    hot_edges = 0
    if world == 1 and n_hot > 0 and os.environ.get("SPEX_TWO_PASS"):
        hot_edges = g.split_hot_cold(nur)
    # optional (SPEX_INTERLEAVE=1): schedule user rows (L2-served gathers of popular items) and item rows
    # (DRAM-served gathers of random users) interleaved.  Measured slower (184.9 vs 176.7 ms): off.
    if world == 1 and os.environ.get("SPEX_INTERLEAVE"):
        g.set_row_classes(nur)
    nnz = g.nnz
    table = synthetic.xavier_table(nur, m, D, 2020, dev)
    torch.cuda.synchronize()
    t_gen = time.time() - t_gen

    launches0 = _capi.launch_count()
    clocks = Clocks(local_rank) if rank == 0 else None

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- propagation: device-resident ----
    if world == 1:
        out = torch.empty_like(table)
        tmp0, tmp1 = torch.empty_like(table), torch.empty_like(table)

        def step():
            _capi.call("spex_propagate_mean_f32", _capi.ptr(g.rowptr), _capi.ptr(g.col), _capi.ptr(g.val),
                       _capi.ptr(table), N, D, K_LAYERS, _capi.ptr(out), _capi.ptr(tmp0), _capi.ptr(tmp1),
                       g.plan(D), _capi.stream_ptr())
            return out
        local_nnz = nnz
        local_rows = N
        prop = None
        balance_log = None
    else:
        rp_host = g.rowptr.cpu().numpy()
        bounds = partition_rows_by_nnz(rp_host, world)
        # set-up (untimed): equalise the MEASURED local SpMM time of the ranks.  Blocks of user rows
        # (popular item rows hit L2) and of item rows (random user rows do not) cost differently
        # per edge, so a pure nnz balance leaves the item-row ranks as stragglers.
        if args.exchange == "auto":   # NVLS multicast needs NVSwitch + driver support: probe once
            try:
                probe = PartitionedPropagator(None, [0] * world + [16], D, K_LAYERS, mode="mcast", device=dev)
                probe.close()
                ok = torch.ones(1, device=dev)
            except Exception:
                ok = torch.zeros(1, device=dev)
            dist.all_reduce(ok, op=dist.ReduceOp.MIN)
            # one multicast store replaces P-1 peer stores: pays from 4 GPUs on (2 GPUs measured:
            # push 62.9 vs mcast 60.6 GEdges/s; 8 GPUs: 197.1 vs 200.9)
            args.exchange = "mcast" if (float(ok.item()) > 0 and world >= 4) else "push"
        balance_log = []
        n_bal = int(os.environ.get("SPEX_BALANCE_ROUNDS", 6))   # measured rounds + 1; the block holding the user/item boundary converges last
        for it in range(n_bal):
            r0, r1 = bounds[rank], bounds[rank + 1]
            lo, hi = int(rp_host[r0]), int(rp_host[r1])
            lg = ops.DeviceGraph((g.rowptr[r0: r1 + 1] - lo).contiguous(), g.col[lo:hi], g.val[lo:hi], N,
                                 None, g.seg_len, row_offset=r0, col_hot=g.col_hot)
            if it == n_bal - 1:
                break
            y = torch.empty(r1 - r0, D, dtype=torch.float32, device=dev)
            tprop = None
            if args.exchange in ("push", "mcast"):
                # time the real thing: the layer kernel WITH its P2P stores into every peer's table
                # (a rank with many short rows is bound by NVLink egress, not by the gathers)
                tprop = PartitionedPropagator(lg, bounds, D, K_LAYERS, mode=args.exchange, device=dev)
                tprop._all_gather_rows(tprop._X[0], table[r0:r1])
                tprop._stream_barrier()
                add = table[r0:r1]

                def one():
                    tprop._layer(tprop._X[0], None, add, y, 1.0, push_buf=1)
            else:
                def one():
                    ops.spmm(lg, table, Y=y)
            for _ in range(2):
                one()
                if tprop is not None:
                    tprop._stream_barrier()
            torch.cuda.synchronize()
            if world > 1:
                dist.barrier()
            ms_sum = 0.0
            for _ in range(3):
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                one()
                e1.record()
                if tprop is not None:
                    tprop._stream_barrier()   # all ranks run the layer at the same time
                torch.cuda.synchronize()
                ms_sum += e0.elapsed_time(e1)
            if tprop is not None:
                tprop.close()
                del tprop
            tl = torch.tensor([ms_sum / 3], dtype=torch.float64, device=dev)
            allt = [torch.zeros_like(tl) for _ in range(world)]
            dist.all_gather(allt, tl)
            times = [float(x.item()) for x in allt]
            balance_log.append([round(x, 3) for x in times])
            bounds = rebalance_bounds(rp_host, bounds, times)
            del y, lg
        lg = ops.DeviceGraph(lg.rowptr, lg.col.clone(), lg.val.clone(), N, None, g.seg_len, row_offset=r0,
                             col_hot=g.col_hot)
        E0_local = table[r0:r1].clone()
        train_batch = None
        if not args.no_train:   # the same sampling as at N = 1 (same seed on every rank), while the full graph is here
            gen_t = torch.Generator(device=dev)
            gen_t.manual_seed(11)
            train_batch = sample_train_batch(torch, g, nur, m, args.train_batch, gen_t)
        del g, table
        torch.cuda.empty_cache()
        prop = PartitionedPropagator(lg, bounds, D, K_LAYERS, mode=args.exchange, device=dev)
        if args.e0_exchange is not None and args.exchange != "nccl":
            prop.e0_exchange = args.e0_exchange   # default: nccl in push mode, mcast in mcast mode
        elif args.exchange == "push" and world == 2:
            prop.e0_exchange = "push"             # 2 GPUs: one peer, P2P stores beat the NCCL path (95 vs 115 ms/step)
        local_nnz, local_rows = hi - lo, r1 - r0
        out_local = torch.empty_like(E0_local)
        prefetch = prop.can_prefetch() and not os.environ.get("SPEX_NO_PREFETCH")

        def step():
            # the table of the NEXT step (here: the same resident table) is published to all ranks by a
            # background kernel while this step's last layer runs (dist.py: ring of three tables)
            return prop.propagate(E0_local, out=out_local, next_E0_local=E0_local if prefetch else None)

    for _ in range(args.warmup):
        step()
    barrier()
    if clocks:
        clocks.mark(True)
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record()
    for _ in range(args.steps):
        res = step()
    ev1.record()
    barrier()
    ms = ev0.elapsed_time(ev1)
    t = torch.tensor([ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_step = float(t.item()) / args.steps
    value = nnz * K_LAYERS / (ms_step * 1e-3) / 1e9
    launches_timed = _capi.launch_count() - launches0
    if args.dump_outputs:   # before the parity check below reuses the work buffers
        dump_outputs(args.dump_outputs, res, [0, N] if world == 1 else bounds, rank, world, torch, dist)
    # parity at full size, untimed: D^-1/2 A D^-1/2 has the eigenvector sqrt(deg) (eigenvalue 1), so
    # propagating a table whose columns are multiples of sqrt(deg) must return it unchanged
    gsrc = g if world == 1 else lg
    deg = (gsrc.rowptr[1:] - gsrc.rowptr[:-1]).to(torch.float32)
    Echk = deg.sqrt()[:, None] * (1.0 + torch.arange(D, device=dev, dtype=torch.float32) / D)[None, :]
    if world == 1:
        ochk = torch.empty_like(Echk)
        _capi.call("spex_propagate_mean_f32", _capi.ptr(g.rowptr), _capi.ptr(g.col), _capi.ptr(g.val),
                   _capi.ptr(Echk), N, D, K_LAYERS, _capi.ptr(ochk), _capi.ptr(tmp0), _capi.ptr(tmp1),
                   g.plan(D), _capi.stream_ptr())
    else:
        ochk = prop.propagate(Echk)
    nzr = deg > 0
    relerr = ((ochk[nzr] - Echk[nzr]).abs() / Echk[nzr]).max().to(torch.float64).reshape(1)
    if world > 1:
        dist.all_reduce(relerr, op=dist.ReduceOp.MAX)
    parity = {"check": "sqrt(deg) is a fixed point of every layer and of the layer mean (all edges, all ranks)",
              "max_rel_err": float(relerr.item()), "tolerance": 1e-5, "ok": bool(float(relerr.item()) < 1e-5)}
    del Echk, ochk, deg, nzr
    res = step()   # (the parity check above used the work buffers)
    hsh = table_hash(res, 0 if world == 1 else r0, torch)
    if world > 1:
        dist.all_reduce(hsh)
    out_hash = f"{int(hsh.item()) & 0xFFFFFFFFFFFFFFFF:016x}"
    phase_log = None
    if prop is not None:   # one extra (untimed) step with per-phase CUDA events, max over ranks
        prop.timing = []
        step()
        ph = prop.phase_ms()
        prop.timing = None
        tl = torch.tensor([x for _, x in ph], dtype=torch.float64, device=dev)
        dist.all_reduce(tl, op=dist.ReduceOp.MAX)
        phase_log = [[n, round(float(x), 3)] for (n, _), x in zip(ph, tl.tolist())]
    launches_per_step = launches_timed // max(args.warmup + args.steps, 1)

    # roofline of the dominant kernel (CSR SpMM), per launch = one layer over this rank's rows.
    # Algorithmic bytes per layer (DESIGN.md §4): every edge reads col(4)+val(4)+one 256 B row,
    # every row reads rowptr(8) and writes/reads D*4 of output: (nnz + rows) * 264.
    alg_bytes = (local_nnz + local_rows) * (8 + 4 * D)
    t_launch = ms_step * 1e-3 / K_LAYERS
    achieved = alg_bytes / t_launch / 1e9
    # DRAM traffic per layer: NOT measured by this run - read from the newest committed `ncu --set full` summary
    # of this exact workload (full scale, one GPU) under profiles/, and labelled with its file name
    traffic, traffic_src = (None, None)
    l2_bytes = None
    if world == 1 and args.scale == 1.0:
        l2_bytes = profile_metric(["spmm_rows_kernel<64", "spmm_seg_list_kernel<64", "spmm_long_fix_list_kernel<64"],
                                  "l1tex__m_xbar2l1tex_read_bytes.sum")
        traffic, traffic_src = profile_traffic(["spmm_rows_kernel<64", "spmm_seg_list_kernel<64", "spmm_long_fix_list_kernel<64"])
    roofline = {"bound": "hbm", "kernel": "spmm_rows_kernel<64,8,1,1> + spmm_seg_list_kernel<64,8,1,1> + "
                                          "spmm_long_fix_list_kernel<64,8> (one layer = one launch of each)",
                "achieved": achieved, "peak": hbm_peak, "unit": "GB/s", "frac": achieved / hbm_peak,
                "peak_kind": peak_kind, "traffic": traffic, "traffic_source": traffic_src,
                "algorithmic_bytes_per_launch": alg_bytes,
                # frac > 1 is possible: the algorithmic bytes assume no cache reuse, L2 serves part of
                # the gathers.  The DRAM-side view of the same launch: measured traffic / time / peak.
                "dram_achieved": (traffic / t_launch / 1e9) if traffic else None,
                "dram_frac": (traffic / t_launch / 1e9 / hbm_peak) if traffic else None,
                # what actually bounds the layer (DESIGN.md 4.1): bytes the L2 slices deliver to the SMs
                # (ncu l1tex__m_xbar2l1tex_read_bytes, same committed capture), against the ~6300 B/clk LTS cap
                # that B300_MICROARCH.md measures (no B200 figure in MEASURED_PEAKS.json: reported, not a frac)
                "l2_to_sm_bytes": l2_bytes,
                "l2_to_sm_achieved": (l2_bytes / t_launch / 1e9) if l2_bytes else None,
                "l2_to_sm_cap_note": "~6300 B/clk full chip = 10.7 TB/s at 1.7 GHz, 12.4 TB/s at 1.965 GHz (guide, B300)",
                "note": "per-launch time = step time / K (exchange included at N>1); traffic from ncu, "
                        "per layer"}

    # ---- e2e: host tables in, host tables out, through the public operator ----
    # Every step copies ITS OWN fused embedding table from pinned host memory (H2D) and ITS OWN
    # propagated table back (D2H); copies run on two side streams so that step i+1's upload and
    # step i-1's download overlap step i's kernels (double-buffered device tables), as a serving
    # loop would do.  All copies are inside the timed region.
    e2e = None
    if not args.no_e2e:
        rows = N if world == 1 else local_rows
        src = table if world == 1 else E0_local
        h_in = torch.empty(rows, D, dtype=torch.float32).pin_memory()
        h_in.copy_(src.cpu())
        h_out = [torch.empty(rows, D, dtype=torch.float32).pin_memory() for _ in range(2)]
        d_in = [src.clone(), torch.empty_like(src)]
        d_out = [torch.empty_like(src) for _ in range(2)]
        s_h2d, s_d2h = torch.cuda.Stream(), torch.cuda.Stream()
        main = torch.cuda.current_stream()

        def e2e_run(n_steps):
            up = [torch.cuda.Event() for _ in range(n_steps)]
            done = [torch.cuda.Event() for _ in range(n_steps)]
            free_in = [None, None]     # compute finished reading d_in[b]
            free_out = [None, None]    # download of d_out[b] finished
            uploaded = [False] * (n_steps + 1)
            for i in range(n_steps):
                b = i & 1
                if not uploaded[i]:
                    with torch.cuda.stream(s_h2d):
                        if free_in[b] is not None:
                            s_h2d.wait_event(free_in[b])
                        d_in[b].copy_(h_in, non_blocking=True)
                        up[i].record(s_h2d)
                main.wait_event(up[i])
                if free_out[b] is not None:
                    main.wait_event(free_out[b])
                if world == 1:
                    _capi.call("spex_propagate_mean_f32", _capi.ptr(g.rowptr), _capi.ptr(g.col),
                               _capi.ptr(g.val), _capi.ptr(d_in[b]), N, D, K_LAYERS, _capi.ptr(d_out[b]),
                               _capi.ptr(tmp0), _capi.ptr(tmp1), g.plan(D), _capi.stream_ptr())
                else:
                    # straight into the caller's buffer; the NEXT step's table (already on its way up on
                    # the copy stream) is published to the other ranks during this step's last layer
                    nxt = i + 1 < n_steps and prefetch
                    if nxt:
                        nb = (i + 1) & 1
                        with torch.cuda.stream(s_h2d):
                            if free_in[nb] is not None:
                                s_h2d.wait_event(free_in[nb])
                            d_in[nb].copy_(h_in, non_blocking=True)
                            up[i + 1].record(s_h2d)
                        uploaded[i + 1] = True
                    prop.propagate(d_in[b], out=d_out[b], next_E0_local=d_in[(i + 1) & 1] if nxt else None,
                                   next_ready=up[i + 1] if nxt else None)
                done[i].record(main)
                free_in[b] = done[i]
                with torch.cuda.stream(s_d2h):
                    s_d2h.wait_event(done[i])
                    h_out[b].copy_(d_out[b], non_blocking=True)
                    ev = torch.cuda.Event()
                    ev.record(s_d2h)
                    free_out[b] = ev
            main.wait_stream(s_d2h)
            main.wait_stream(s_h2d)

        e2e_run(2)
        barrier()
        n_e2e = max(20, args.steps)   # enough steps to amortise the pipeline fill (first upload) and drain (last download)
        ev0.record()
        e2e_run(n_e2e)
        ev1.record()
        barrier()
        t = torch.tensor([ev0.elapsed_time(ev1)], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms_e2e = float(t.item()) / n_e2e
        # the copies alone (same buffers, same streams, no kernels): what the host link allows per step
        def copies_only(n_steps):
            for i in range(n_steps):
                b = i & 1
                with torch.cuda.stream(s_h2d):
                    d_in[b].copy_(h_in, non_blocking=True)
                with torch.cuda.stream(s_d2h):
                    h_out[b].copy_(d_out[b], non_blocking=True)
            main.wait_stream(s_d2h)
            main.wait_stream(s_h2d)

        copies_only(2)
        barrier()
        ev0.record()
        copies_only(n_e2e)
        ev1.record()
        barrier()
        tc = torch.tensor([ev0.elapsed_time(ev1)], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(tc, op=dist.ReduceOp.MAX)
        ms_copy = float(tc.item()) / n_e2e
        e2e = {"value": nnz * K_LAYERS / (ms_e2e * 1e-3) / 1e9, "unit": UNIT,
               "copies_alone_ms_per_step": ms_copy,
               "host_link_gbs_per_direction_whole_job": N * D * 4 / (ms_copy * 1e-3) / 1e9,
               "h2d_bytes_per_step": N * D * 4, "d2h_bytes_per_step": N * D * 4,  # summed over ranks
               "ms_per_step": ms_e2e, "steps": n_e2e,
               "note": "pinned host <-> device copies of every step's table on side streams, overlapped "
                       "with the previous/next step's kernels; result checked equal to the resident run"}
        if world == 1:
            assert torch.equal(h_out[(n_e2e - 1) & 1].to(dev), res), "e2e result differs from the resident run"
    if clocks:
        clocks.mark(False)

    # ---- e2e buffers are no longer needed: make room for the evaluation and training legs ----
    if not args.no_e2e:
        del h_in, h_out, d_in, d_out
    torch.cuda.empty_cache()

    # ---- secondary: full-ranking top-20 over ALL users (BASELINE.json configs[4]) ----
    # users sharded by rank (no communication), the propagated item table replicated; one step = the
    # whole sweep: per block of users, pack the user rows (fp16, scaled) + one launch of the tcgen05
    # scorer (filter + mask + top-k); results stay on the device ([users, 20] ids and scores).
    evalj = None
    if not args.no_eval:
        if world == 1:
            U_all, I_all = res[:nur], res[nur:]
        else:
            # every rank needs all propagated item rows: gather once (evaluation set-up, untimed)
            full = torch.empty(N, D, dtype=torch.float32, device=dev)
            prop._all_gather_rows(full, res)
            U_all, I_all = full[:nur], full[nur:]
        n_total = min(args.eval_users, nu) if args.eval_users > 0 else nu
        u_lo, u_hi = (n_total * rank) // world, (n_total * (rank + 1)) // world
        n_eval = u_hi - u_lo
        users = torch.arange(u_lo, u_hi, device=dev)
        blk = 148 * 2 * 128 * 4
        idx = torch.empty(n_eval, TOPK, dtype=torch.int32, device=dev)
        val = torch.empty(n_eval, TOPK, dtype=torch.float32, device=dev)
        if args.eval_scorer == "f16":
            Ih, m_pad, imeta = ops.pack_f16(I_all, None, ops.TC_ITEM_MULTIPLE)
        else:
            Ib, m_pad = ops.pack_bf16(I_all, None, ops.TC_ITEM_MULTIPLE)

        def eval_sweep(limit=None):
            hi = n_eval if limit is None else min(limit, n_eval)
            for a in range(0, hi, blk):
                ub = users[a: min(a + blk, hi)]
                if args.eval_scorer == "f16":
                    Uh, b_pad, umeta = ops.pack_f16(U_all, ub, ops.TC_USER_MULTIPLE)
                    ops.score_topk_f16(Uh, umeta, ub.numel(), b_pad, Ih, imeta, m, m_pad, D, TOPK, ub, mask_rp,
                                       mask_col, idx[a: a + ub.numel()], val[a: a + ub.numel()])
                else:
                    Ub, b_pad = ops.pack_bf16(U_all, ub, ops.TC_USER_MULTIPLE)
                    ops.score_topk_bf16(Ub, ub.numel(), b_pad, Ib, m, m_pad, TOPK, ub, mask_rp, mask_col,
                                        idx[a: a + ub.numel()], val[a: a + ub.numel()])

        eval_sweep(blk)   # warm-up on one block
        barrier()
        ev0.record()
        eval_sweep()
        ev1.record()
        barrier()
        t = torch.tensor([ev0.elapsed_time(ev1)], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms_ev = float(t.item())
        flops = 2.0 * n_eval * m * D
        tf = flops / (ms_ev * 1e-3) / 1e12
        # untimed sanity on the last block: sorted best-first, in range, and equal to the exact fp32 scorer
        # on 256 of its users (same top-20 scores to 2e-3 relative: fp16 / bf16 operand rounding)
        chk = torch.arange(max(n_eval - 256, 0), n_eval, device=dev)
        i32, v32 = ops.score_topk_f32(U_all, I_all, users[chk], TOPK, mask_rp, mask_col)
        sc = float(v32.abs().max())
        eval_ok = bool((val[chk][:, :-1] >= val[chk][:, 1:]).all()) and bool((idx[chk] >= 0).all()) and \
            bool((idx[chk] < m).all()) and float((val[chk] - v32).abs().max()) <= (2e-3 if args.eval_scorer == "f16" else 1e-2) * sc
        agree = float((idx[chk] == i32).float().mean())
        # CPU leg of metric 2 (rank 0, N = 1): torch.matmul + masked_fill + topk on the same tables
        cpu_eval = None
        if rank == 0 and world == 1 and not args.no_cpu_baseline:
            cores = os.cpu_count() or 1
            torch.set_num_threads(cores)
            n_cpu = 128
            Uc, Ic = U_all[:n_cpu].cpu(), I_all.cpu()
            rp_c, col_c = mask_rp[: n_cpu + 1].cpu(), mask_col[: int(mask_rp[n_cpu].item())].cpu().long()
            rows_c = torch.repeat_interleave(torch.arange(n_cpu), rp_c[1:] - rp_c[:-1])

            def cpu_rank():
                sco = torch.matmul(Uc, Ic.t())
                sco[rows_c, col_c] = float("-inf")
                return torch.topk(sco, TOPK, dim=1)

            cpu_rank()
            t0 = time.perf_counter()
            for _ in range(2):
                cv, ci = cpu_rank()
            dtc = (time.perf_counter() - t0) / 2
            same = float((ci.to(dev).int() == ops.score_topk_f32(U_all, I_all, torch.arange(n_cpu, device=dev), TOPK,
                                                                 mask_rp, mask_col)[0]).float().mean())
            cpu_eval = {"value": n_cpu / dtc, "unit": "users/s", "cores": cores, "kind": "port",
                        "sample": f"torch.matmul + masked_fill + topk(20), {n_cpu} users x {m} items, D={D}, fp32, "
                                  f"2 timed runs, {dtc * 1e3:.0f} ms each; top-20 ids equal to the fp32 GPU scorer: {same:.4f}"}
            del Uc, Ic
        evalj = {"metric": "fullrank_top20_users_per_s", "value": n_total / (ms_ev * 1e-3),
                 "unit": "users/s", "users_ranked": n_total, "users_per_gpu": n_eval, "m_items": m, "ms_per_sweep": ms_ev,
                 "scorer": args.eval_scorer, "check": {"ok": eval_ok, "top20_ids_equal_to_fp32_scorer": agree},
                 "config": {"workload": f"full-ranking top-20 sweep, {n_total} users x {m} items, D={D}, user-sharded x{world} "
                                        "(BASELINE.json configs[4])"},
                 # B200_PROFILING.md: the burst peak is for a kernel timed alone, the sustained one for a kernel
                 # timed inside a long step - a sweep of seconds runs under the power cap like the sustained GEMM
                 "roofline": {"bound": "tensor", "kernel": "score_topk_f16_kernel<64,1>" if args.eval_scorer == "f16"
                              else "score_topk_tc_kernel<1>", "achieved": tf,
                              "peak": tc_sust if ms_ev > 1000.0 else tc_burst, "unit": "TFLOP/s",
                              "frac": tf / (tc_sust if ms_ev > 1000.0 else tc_burst),
                              "peak_kind": peak_kind + (" (sustained bf16 GEMM: the sweep runs for seconds)"
                                                        if ms_ev > 1000.0 else " (burst bf16 GEMM)"),
                              "frac_of_burst_peak": tf / tc_burst, "frac_of_sustained_peak": tf / tc_sust,
                              "traffic": None},
                 "cpu_baseline": cpu_eval}
        del idx, val, users
        if world > 1:
            del full

    # ---- training step (main_rec.py:30-37): forward + BCE + backward + dense Adam, N = 1 ----
    trainj = None
    if world == 1 and not args.no_train:
        trainj = bench_train_step(args, torch, ops, _capi, g, table, nur, m, N, hbm_peak, peak_kind, dev)
    elif world > 1 and not args.no_train:
        # row-partitioned training step (spex_b200/dist.py: PartitionedTrainer): table / gradient / Adam
        # moments owned by row, the batch replicated (same seed on every rank), backward = the same
        # partitioned propagation applied to the gradient
        from spex_b200.dist import PartitionedTrainer

        Bt = args.train_batch
        tu, ti, tl = train_batch
        W_start = E0_local.clone()

        def measure_tr(receptive):
            tr = PartitionedTrainer(prop, W_start.clone(), nur, lr=1e-3)
            tr.receptive_field = receptive
            prop._staged = None        # the table of the previous arm is not this one's
            for _ in range(2):
                tr.step(tu, ti, tl)
            barrier()
            n_tr = 4
            ev0.record()
            for _ in range(n_tr):
                tloss = tr.step(tu, ti, tl)
            ev1.record()
            barrier()
            t = torch.tensor([ev0.elapsed_time(ev1)], dtype=torch.float64, device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            return float(t.item()) / n_tr, float(tloss.item()), tr.W.detach().clone()

        ms_tr_full, loss_full, W_a = measure_tr(False)
        ms_tr, loss_rf, W_b = measure_tr(True)
        same_w = torch.tensor([1.0 if torch.equal(W_a, W_b) else 0.0], device=dev)
        dist.all_reduce(same_w, op=dist.ReduceOp.MIN)     # every rank's slice of the weights after the 6 steps
        del W_a, W_b
        sets = prop.receptive_sets(torch.unique(torch.cat([tu, ti + nur])))
        trainj = {"metric": "lightgcn_train_step_ms", "value": ms_tr, "unit": "ms", "higher_is_better": False,
                  "steps_per_s": 1e3 / ms_tr, "batch": Bt, "loss": loss_rf,
                  "receptive_field": {"rows_per_layer": [None if r is None else int(r.numel()) for r in sets[1:]],
                                      "note": "forward layers restricted to the rows the batch depends on (null = all "
                                              "rows), restricted rows exchanged by the same fused epilogue; the "
                                              "backward mirrors it (first layer restricted, written into zeroed "
                                              "tables); loss and weights bit-identical to the full step"},
                  "full_computer_step": {"value": ms_tr_full, "unit": "ms", "loss": loss_full,
                                         "same_loss_as_receptive_path": loss_full == loss_rf,
                                         "same_weights_after_6_steps_as_receptive_path": bool(same_w.item() > 0)},
                  # edges actually traversed per second: quoted on the FULL step
                  "gedges_per_s_fwd_plus_bwd": 2 * K_LAYERS * nnz / (ms_tr_full * 1e-3) / 1e9,
                  "config": {"workload": f"main_rec.py:30-37 step, row-partitioned x{world}: forward + BCE (1 positive + 5 "
                                         f"negatives per user, as at N=1) + backward (partitioned propagation of the "
                                         f"gradient) + row-owned Adam fused into the last backward layer, exchange={args.exchange}"}}

    smallj = None
    if rank == 0 and world == 1 and not args.no_small_configs:
        try:
            smallj = bench_small_configs(torch, dev)
        except Exception as e:   # secondary legs must never cost the headline line
            smallj = {"error": f"{type(e).__name__}: {e}"}
    launches_total = _capi.launch_count() - launches0
    ck = clocks.stop() if clocks else None

    # ---- CPU baseline on a bounded sample (rank 0, N = 1 only) ----
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        cores = os.cpu_count() or 1
        torch.set_num_threads(cores)
        A, snu, sm_ = cpu_sample_graph(args.cpu_sample_scale)
        ge, dt = cpu_time_computer(A, snu, sm_, 3, 1)
        cpu = {"value": ge, "unit": UNIT, "cores": cores, "kind": "port",
               "sample": f"oracle computer() (torch.sparse.mm, the reference's CPU backend) K={K_LAYERS} D={D} "
                         f"on {snu} users x {sm_} items, nnz(A)={A._nnz()}, 3 timed runs, {dt * 1e3:.0f} ms each",
               "larger_sample_on_record": "1/10 scale (1 M x 500 k, nnz 2e8), same box type: 0.0111 GEdges/s, 54 s per "
                                          "K=3 step (profiles/r02_reference_arm_scale_0.1.json; --cpu-sample-scale 0.1): "
                                          "the CPU path gets slower per edge as the table outgrows its caches, so "
                                          "the 1/100 sample flatters it"}

    if rank == 0:
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_step, "higher_is_better": True, "scaling": "strong",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": f"synthetic {nu} users x {m} items, {nnz // 2} unique interactions "
                                   f"(nnz(A)={nnz}), D={D}, K={K_LAYERS} (BASELINE.json configs[3], scale {args.scale:g})",
                       "edges_definition": "nnz(A) = 2*|R| per layer", "l2": "inputs larger than L2 (no flush needed)"
                       if nnz * 8 > 200e6 else "inputs smaller than L2: timing is L2-warm",
                       "parallelism": f"row-partition x{world}" + (f" exchange={args.exchange}" + (f" e0={prop.e0_exchange}" if args.exchange != "nccl" else "")
                                                                       if world > 1 else ""),
                       "graph_build_s": round(t_gen, 2), "hot_rows_kept_in_l2": n_hot,
                       "two_pass_hot_edges": hot_edges, "interleaved_row_classes": int(world == 1 and g.interleave_split > 0) if world == 1 else 0,
                       "balance_ms_per_rank": balance_log if world > 1 else None,
                       "e0_prefetch_during_last_layer": bool(world > 1 and prefetch),
                       "numa_cpus_rank0": numa_cpus,
                       "phase_ms_max_over_ranks": phase_log},
            "roofline": roofline, "cpu_baseline": cpu, "e2e": e2e, "eval": evalj, "train_step": trainj, "small_configs": smallj,
            "parity": parity,
            "output_table_hash64": out_hash,
            "gpu_launches": launches_total, "gpu_launches_per_step": launches_per_step, "clocks": ck,
        }
        print(json.dumps(line), flush=True)
    if prop is not None:
        prop.close()
    if world > 1:
        dist.destroy_process_group()


def main():
    args = parse()
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
