"""Edge dropout in the row-partitioned trainer, on CPU: the row blocks' transposed values (host), and the world-2
gloo orchestration of PartitionedTrainer(keep_prob=...) against the single-process oracle on A_drop built from the
numpy replica of the device mask (test_edge_dropout.mask_keep)."""
import os
import socket

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from helpers import oracle_graph, random_graph
from oracle import lightgcn_oracle as O
from spex_b200.graph import build_norm_adj, partition_rows_by_nnz


def _weighted_pairs(nu, m, n, seed):
    """Interactions with duplicate pairs (weight 3 after the builder sums them): values not symmetric bit for bit."""
    u, i = random_graph(nu, m, n, seed)
    return np.concatenate([u, u[::7], u[::7]]), np.concatenate([i, i[::7], i[::7]])


# ---- host: row blocks that produce their transposed values -------------------------------------------------------
def test_weighted_row_block_carries_its_transposed_values():
    nu, m = 300, 120
    u, i = _weighted_pairs(nu, m, 3000, 21)
    g = build_norm_adj(u, i, nu + 1, m)
    assert not np.array_equal(g.val, g.val[g.tpos])
    bounds = partition_rows_by_nnz(g.rowptr, 3)
    carried = 0
    for r0, r1 in zip(bounds[:-1], bounds[1:]):
        lo, hi = int(g.rowptr[r0]), int(g.rowptr[r1])
        blk = g.row_block(r0, r1, transposed_values=True)
        want = g.val[g.tpos[lo:hi]]
        assert blk.tpos is None and blk.row_offset == r0
        if blk.tval is None:
            assert blk.values_symmetric and np.array_equal(blk.val.view(np.uint32), want.view(np.uint32))
        else:
            assert not blk.values_symmetric
            assert np.array_equal(blk.tval.view(np.uint32), want.view(np.uint32))
            carried += 1
    assert carried > 0


def test_symmetric_row_block_needs_no_transposed_values():
    nu, m = 300, 120
    u, i = random_graph(nu, m, 3000, 22)
    g = build_norm_adj(u, i, nu + 1, m)
    blk = g.row_block(10, 200, transposed_values=True)
    assert blk.values_symmetric and blk.tval is None
    plain = g.row_block(10, 200)                    # without the option: the block of before, nothing extra
    assert not plain.values_symmetric and plain.tval is None
    g.tpos = None
    with pytest.raises(ValueError, match="transpose map"):
        g.row_block(10, 200, transposed_values=True)


# ---- gloo, world 2: the trainer with dropout against the single-process oracle -----------------------------------
def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _sparse(blk, n_cols, val=None):
    rows = torch.from_numpy(blk.rows_of_entries())
    idx = torch.stack([rows, torch.from_numpy(blk.col.astype(np.int64))])
    return torch.sparse_coo_tensor(idx, torch.from_numpy(blk.val) if val is None else val,
                                   (blk.n_rows, n_cols)).coalesce()


def _train_worker(rank, world, port, weighted, q):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        from test_edge_dropout import mask_keep, mask_u
        from spex_b200.dist import PartitionedPropagator, PartitionedTrainer, _TorchTrainOps
        from spex_b200.model import dropout_seed

        nu, m, D, K, kp = 120, 80, 16, 3, 0.3
        u, i = _weighted_pairs(nu, m, 1500, 5) if weighted else random_graph(nu, m, 1500, 5)
        g = build_norm_adj(u, i, nu + 1, m)
        bounds = partition_rows_by_nnz(g.rowptr, world)
        r0, r1 = bounds[rank], bounds[rank + 1]
        blk = g.row_block(r0, r1, transposed_values=True)
        Ablk = _sparse(blk, g.n_cols)

        class MaskOps(_TorchTrainOps):
            """The device mask through the numpy replica: (val, valT) of this rank's block."""

            def dropout_values(self, A, seed, keep_prob):
                rows = A.indices()[0].numpy() + r0
                cols = A.indices()[1].numpy()
                v = A.values()
                vt = v if blk.tval is None else torch.from_numpy(blk.tval)
                fwd = torch.from_numpy(mask_keep(seed, rows, cols, keep_prob)).float()
                bwd = torch.from_numpy(mask_keep(seed, cols, rows, keep_prob)).float()
                return v * fwd / keep_prob, vt * bwd / keep_prob

        def local_spmm(A, X, val=None):
            return torch.sparse.mm(A if val is None else torch.sparse_coo_tensor(A.indices(), val, A.shape), X)

        torch.manual_seed(3)
        W = torch.randn(g.n_rows, D, dtype=torch.float64).float() * 0.1
        prop = PartitionedPropagator(Ablk, bounds, D, K, mode="nccl", device=torch.device("cpu"), local_spmm=local_spmm)
        tr = PartitionedTrainer(prop, W[r0:r1].clone(), nu + 1, lr=1e-2, train_ops=MaskOps(), keep_prob=kp)
        batches = []
        rng = np.random.default_rng(0)
        for _ in range(3):
            users = torch.from_numpy(rng.integers(0, nu, 64))
            users[:10] = users[0]
            items = torch.from_numpy(rng.integers(0, m, 64))
            labels = torch.from_numpy(rng.integers(0, 2, 64))
            batches.append((users, items, labels))
        torch.manual_seed(77)
        losses = [float(tr.step(us, it, lb.float())) for us, it, lb in batches]
        torch.manual_seed(77)
        seeds = [dropout_seed() for _ in batches]   # the draws the trainer made, one per step
        # single-process oracle: the reference's forward + autograd + torch.optim.Adam on A_drop of each step
        uw = W[: nu + 1].clone().requires_grad_(True)
        iw = W[nu + 1:].clone().requires_grad_(True)
        opt = torch.optim.Adam([uw, iw], lr=1e-2)
        A = oracle_graph(u, i, nu + 1, m).coalesce()
        idx = A.indices().numpy()
        ref_losses = []
        for seed, (us, it, lb) in zip(seeds, batches):
            Adrop = O.dropout_graph(A, kp, rand=torch.from_numpy(mask_u(seed, idx[0], idx[1])))
            opt.zero_grad()
            loss = O.bce_forward(uw, iw, Adrop, K, us, it, lb)
            loss.backward()
            opt.step()
            ref_losses.append(float(loss))
        want = torch.cat([uw, iw]).detach()[r0:r1]
        err = float((tr.W - want).abs().max() / want.abs().max())
        lerr = max(abs(a - b) / abs(b) for a, b in zip(losses, ref_losses))
        # without dropout the same batches give other weights: the values were not ignored
        torch.manual_seed(77)
        tr0 = PartitionedTrainer(prop, W[r0:r1].clone(), nu + 1, lr=1e-2, train_ops=MaskOps())
        for us, it, lb in batches:
            tr0.step(us, it, lb.float())
        moved = float((tr0.W - tr.W).abs().max())
        q.put((rank, err, lerr, moved, blk.tval is not None))
    finally:
        dist.destroy_process_group()


@pytest.mark.parametrize("weighted", [False, True])
def test_partitioned_training_with_dropout_world2_matches_single_process_oracle(weighted):
    """Every rank draws the step's seed like the one-GPU model, makes val / valT of its own rows and runs the
    forward with val and the backward with valT: after three steps the weights match the reference's forward +
    autograd + torch.optim.Adam on the same dropped graphs."""
    world = 2
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_train_worker, args=(r, world, port, weighted, q)) for r in range(world)]
    for p in procs:
        p.start()
    res = [q.get(timeout=180) for _ in range(world)]
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    for rank, err, lerr, moved, _ in res:
        assert err < 2e-5, (rank, err)
        assert lerr < 1e-5, (rank, lerr)
        assert moved > 1e-4, (rank, moved)
    assert any(carried for *_, carried in res) == weighted
