"""PartitionedTrainer.bpr_step at world size 2 on CPU (gloo): the BPR orchestration of spex_b200.dist (propagated and
ego rows of the batch assembled by one exact all-reduce, the two gradient scatters, the ego rows' L2 gradient added in
the last backward layer) with the oracle's SpMM and _TorchTrainOps, against upstream LightGCN's loss + autograd +
torch.optim.Adam run in one process.  The CUDA kernels take those slots on GPUs (test_dist_bpr_gpu.py)."""
import os
import socket

import numpy as np
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from helpers import oracle_graph, random_graph
from oracle import lightgcn_oracle as O

DECAY = 0.05     # large enough that the L2 term moves the weights visibly


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _batches(nu, m, B=64, steps=3):
    rng = np.random.default_rng(0)
    out = []
    for _ in range(steps):
        users = torch.from_numpy(rng.integers(0, nu, B))
        pos = torch.from_numpy(rng.integers(0, m, B))
        neg = torch.from_numpy(rng.integers(0, m, B))
        users[:10] = users[0]                  # duplicated users
        pos[5:12] = pos[5]                     # duplicated positives, also drawn as negatives below
        neg[20:26] = pos[5]
        neg[30:33] = neg[30]
        out.append((users, pos, neg))
    return out


def _train_worker(rank, world, port, K, q):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        from spex_b200.dist import PartitionedPropagator, PartitionedTrainer, _TorchTrainOps
        from spex_b200.graph import build_norm_adj, partition_rows_by_nnz

        nu, m, D = 120, 80, 16
        u, i = random_graph(nu, m, 1500, 5)
        g = build_norm_adj(u, i, nu + 1, m)
        bounds = partition_rows_by_nnz(g.rowptr, world)
        r0, r1 = bounds[rank], bounds[rank + 1]
        blk = g.row_block(r0, r1)
        rows = torch.from_numpy(blk.rows_of_entries())
        Ablk = torch.sparse_coo_tensor(torch.stack([rows, torch.from_numpy(blk.col.astype(np.int64))]),
                                       torch.from_numpy(blk.val), (blk.n_rows, g.n_cols)).coalesce()
        torch.manual_seed(3)
        W = torch.randn(g.n_rows, D, dtype=torch.float64).float() * 0.1
        prop = PartitionedPropagator(Ablk, bounds, D, K, mode="nccl", device=torch.device("cpu"),
                                     local_spmm=lambda A, X: torch.sparse.mm(A, X))
        tr = PartitionedTrainer(prop, W[r0:r1].clone(), nu + 1, lr=1e-2, train_ops=_TorchTrainOps(), decay=DECAY)
        batches = _batches(nu, m)
        losses = [float(tr.bpr_step(*b)) for b in batches]
        # the ego rows a batch touches on this rank are flagged, the others not
        users, pos, neg = batches[-1]
        touched = torch.unique(torch.cat([users, pos + nu + 1, neg + nu + 1]))
        touched = touched[(touched >= r0) & (touched < r1)] - r0
        flags_ok = bool(tr.g0_rows[touched].all()) and int(tr.g0_rows.sum()) == touched.numel()
        # single process: upstream LightGCN's loss + decay * reg, autograd, torch.optim.Adam
        uw = W[: nu + 1].clone().requires_grad_(True)
        iw = W[nu + 1:].clone().requires_grad_(True)
        opt = torch.optim.Adam([uw, iw], lr=1e-2)
        A = oracle_graph(u, i, nu + 1, m)
        ref_losses = []
        for users, pos, neg in batches:
            opt.zero_grad()
            loss, reg = O.bpr_loss(uw, iw, A, K, users, pos, neg)
            total = loss + DECAY * reg
            total.backward()
            opt.step()
            ref_losses.append(float(total))
        want = torch.cat([uw, iw]).detach()[r0:r1]
        err = float((tr.W - want).abs().max() / want.abs().max())
        lerr = max(abs(a - b) / abs(b) for a, b in zip(losses, ref_losses))
        # decay 0: the L2 term must not move anything (its gradient is added, not a stale one)
        W_plain = PartitionedTrainer(prop, W[r0:r1].clone(), nu + 1, lr=1e-2, train_ops=_TorchTrainOps(), decay=0.0)
        for b in batches:
            W_plain.bpr_step(*b)
        moved = float((W_plain.W - tr.W).abs().max())
        q.put((rank, err, lerr, flags_ok, moved))
    finally:
        dist.destroy_process_group()


def test_partitioned_bpr_world2_matches_single_process_oracle():
    """Three BPR steps with duplicated users and items and decay != 0, K = 3 and K = 0: weights and losses match
    upstream LightGCN's bpr_loss + autograd + torch.optim.Adam in one process (the bounds of the BCE test at K = 3);
    the ego rows a batch touches are the flagged ones, and decay 0 trains other weights."""
    world = 2
    ctx = mp.get_context("spawn")
    for K in (3, 0):
        q = ctx.Queue()
        port = _free_port()
        procs = [ctx.Process(target=_train_worker, args=(r, world, port, K, q)) for r in range(world)]
        for p in procs:
            p.start()
        res = [q.get(timeout=180) for _ in range(world)]
        for p in procs:
            p.join(timeout=60)
            assert p.exitcode == 0
        for rank, err, lerr, flags_ok, moved in res:
            # K = 0: the gradient is the batch's alone, and the oracle's L2 gradient goes through the norm
            # (x * 2|x| / |x|), rounded differently from x: Adam's normalisation magnifies that on rows whose two
            # gradient terms nearly cancel (2.3e-5 measured with this batch)
            assert err < (2e-5 if K else 5e-5), (K, rank, err)
            assert lerr < 1e-5, (K, rank, lerr)
            assert flags_ok, (K, rank)
            assert moved > 1e-4, (K, rank, moved)
