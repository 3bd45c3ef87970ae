"""Edge dropout (--dropout 2) in the row-partitioned propagation and trainer on GPUs, against the single-GPU model.

A rank makes the dropped values of its own rows (spex_edge_dropout_f32 over its block, global rows through
row_offset) - for a weighted graph from the transposed values its block was cut with.  Checked on a graph whose
values are symmetric bit for bit and on a weighted one (duplicate pairs).  The partitioned tests run one process
per GPU: world 2 needs two devices and is skipped below that; world 1 runs the same code on one device."""
import os
import socket

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from helpers import make_args, random_graph

pytestmark = pytest.mark.gpu

KP = 0.3


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _pairs(weighted, nu=5000, m=3000, n=120000, seed=21):
    u, i = random_graph(nu, m, n, seed, hub_items=3, hub_degree=2500)
    if weighted:   # duplicate pairs: weight 3 after the builder sums them, values no longer symmetric bit for bit
        u, i = np.concatenate([u, u[::7], u[::7]]), np.concatenate([i, i[::7], i[::7]])
    return u, i


def _dataset(weighted, *args):
    from spex_b200.dataloader import SyntheticDataset

    ds = SyntheticDataset(*args)
    if weighted:
        ds.trainUser = np.concatenate([ds.trainUser, ds.trainUser[::7], ds.trainUser[::7]])
        ds.trainItem = np.concatenate([ds.trainItem, ds.trainItem[::7], ds.trainItem[::7]])
    return ds


# ---- one GPU: a block's values are its slice of the whole graph's ----------------------------------------------
@pytest.mark.parametrize("weighted", [False, True])
def test_row_blocks_make_their_slice_of_the_dropout_values(cuda_device, weighted):
    from spex_b200 import ops
    from spex_b200.graph import build_norm_adj, partition_rows_by_nnz

    nu, m = 5000, 3000
    host = build_norm_adj(*_pairs(weighted), nu + 1, m)
    full = ops.DeviceGraph.from_host(host, cuda_device)
    bounds = partition_rows_by_nnz(host.rowptr, 4)
    for seed, kp in ((42, KP), (7, 1.0)):
        val, valT = full.device_dropout_values(seed, kp)
        carried = 0
        for r0, r1 in zip(bounds[:-1], bounds[1:]):
            blk = host.row_block(r0, r1, transposed_values=True)
            carried += blk.tval is not None
            lg = ops.DeviceGraph.from_host(blk, cuda_device)
            bv, bvt = lg.device_dropout_values(seed, kp)
            lo, hi = int(host.rowptr[r0]), int(host.rowptr[r1])
            assert bv.shape == (hi - lo,) and bvt.shape == (hi - lo,)
            assert torch.equal(bv, val[lo:hi]) and torch.equal(bvt, valT[lo:hi]), (r0, r1, kp)
        assert (carried > 0) == weighted
    bare = ops.DeviceGraph.from_host(host.row_block(0, 100), cuda_device)
    if not bare.values_symmetric:
        with pytest.raises(RuntimeError, match="transpose map"):
            bare.device_dropout_values(1, KP)


# ---- one process per GPU ---------------------------------------------------------------------------------------
def _forward(rank, world, dev, res):
    """Partitioned propagate with the block's val (and valT) equal to the single-GPU propagate_mean on the same
    values: nccl and push, K = 1..3, seg_len 32 (long rows), and restricted to the receptive sets of a batch."""
    from spex_b200 import ops
    from spex_b200.dist import PartitionedPropagator
    from spex_b200.graph import build_norm_adj, partition_rows_by_nnz

    nu, m, D = 5000, 3000, 64
    for weighted in (False, True):
        host = build_norm_adj(*_pairs(weighted), nu + 1, m)
        N = host.n_rows
        full = ops.DeviceGraph.from_host(host, dev, seg_len=32)
        bounds = partition_rows_by_nnz(host.rowptr, world)
        r0, r1 = bounds[rank], bounds[rank + 1]
        lo, hi = int(host.rowptr[r0]), int(host.rowptr[r1])
        lg = ops.DeviceGraph.from_host(host.row_block(r0, r1, transposed_values=True), dev, seg_len=32)
        assert lg.n_long > 0
        val, valT = full.device_dropout_values(1234, KP)
        bv, bvt = lg.device_dropout_values(1234, KP)
        res[f"block/w{weighted}"] = torch.equal(bv, val[lo:hi]) and torch.equal(bvt, valT[lo:hi])
        E = (torch.randn(N, D, generator=torch.Generator().manual_seed(5)) * 0.1).to(dev)
        S = torch.unique(torch.from_numpy(np.random.default_rng(3).integers(0, N, 40)).to(dev))
        own = S[(S >= r0) & (S < r1)]
        for K in (1, 2, 3):
            want = ops.propagate_mean(E, full, K, val)
            wantT = ops.propagate_mean(E, full, K, valT)
            for mode in ("nccl", "push"):
                prop = PartitionedPropagator(lg, bounds, D, K, mode=mode, device=dev)
                a = prop.propagate(E[r0:r1].clone(), val=bv)
                b = prop.propagate(E[r0:r1].clone(), val=bvt)
                c = prop.propagate(E[r0:r1].clone())                    # no val: the graph's values again
                ok = torch.equal(a, want[r0:r1]) and torch.equal(b, wantT[r0:r1])
                ok = ok and torch.equal(c, ops.propagate_mean(E, full, K)[r0:r1])
                if mode == "push":
                    sets = prop.receptive_sets(S)
                    engaged = sets[K] is not None
                    d = prop.propagate(E[r0:r1].clone(), row_sets=sets, val=bv)
                    ok = ok and engaged and torch.equal(d[own - r0], want[own])
                prop.close()
                res[f"forward/w{weighted}/K{K}/{mode}"] = bool(ok)


def _train(rank, world, dev, res):
    """Three steps of PartitionedTrainer(keep_prob) against LightGCN(dropout=2) + FusedAdam from the same seeds."""
    from spex_b200 import ops
    from spex_b200.dist import PartitionedPropagator, PartitionedTrainer
    from spex_b200.graph import partition_rows_by_nnz
    from spex_b200.model import LightGCN
    from spex_b200.optim import FusedAdam

    rng = np.random.default_rng(0)
    for weighted in (False, True):
        ds = _dataset(weighted, 400, 250, 6000, 4)
        torch.manual_seed(2020)
        model = LightGCN(make_args(dropout=2, keepprob=KP), ds).to(dev)
        W0 = model._table.detach().clone()
        opt = FusedAdam(model.parameters(), lr=1e-2)
        batches = []
        for _ in range(3):
            users = torch.from_numpy(rng.integers(0, ds.n_users, 256)).to(dev)
            users[:40] = users[0]
            items = torch.from_numpy(rng.integers(0, ds.m_items, 256)).to(dev)
            labels = torch.from_numpy(rng.integers(0, 2, 256)).float().to(dev)
            batches.append((users, items, labels))
        model.train()
        torch.manual_seed(500)
        ref_losses = []
        for b in batches:
            opt.zero_grad(set_to_none=True)
            loss = model(*b, flag=0)
            loss.backward()
            opt.step()
            ref_losses.append(float(loss))
        W_ref = model._table.detach()
        host = ds.getCSR()
        bounds = partition_rows_by_nnz(host.rowptr, world)
        r0, r1 = bounds[rank], bounds[rank + 1]
        lg = ops.DeviceGraph.from_host(host.row_block(r0, r1, transposed_values=True), dev)

        def run(mode, keep_prob):
            prop = PartitionedPropagator(lg, bounds, 64, 3, mode=mode, device=dev)
            if mode == "push":
                prop.e0_exchange = "push"
            tr = PartitionedTrainer(prop, W0[r0:r1].clone(), ds.n_users + 1, lr=1e-2, keep_prob=keep_prob)
            torch.manual_seed(500)
            ls = [float(tr.step(*b)) for b in batches]
            torch.cuda.synchronize()
            prop.close()
            return ls, tr.W.clone()

        for mode in ("nccl", "push"):
            ls, W = run(mode, KP)
            werr = float((W - W_ref[r0:r1]).abs().max() / W_ref.abs().max())
            lerr = max(abs(a - b) / abs(b) for a, b in zip(ls, ref_losses))
            _, W_plain = run(mode, None)
            res[f"train/w{weighted}/{mode}"] = (ls[0] == ref_losses[0], lerr, werr, not torch.equal(W, W_plain))
            if not weighted:   # keep_prob 1 keeps every edge at its value: the trainer without dropout, bit for bit
                res[f"kp1/{mode}"] = torch.equal(run(mode, 1.0)[1], W_plain)
    # receptive field on and off: bit-identical weights (a graph large enough for the restriction to engage)
    for weighted in (False, True):
        ds = _dataset(weighted, 20000, 8000, 150000, 8)
        torch.manual_seed(11)
        W0 = LightGCN(make_args(), ds)._table.detach().clone().to(dev)
        host = ds.getCSR()
        bounds = partition_rows_by_nnz(host.rowptr, world)
        r0, r1 = bounds[rank], bounds[rank + 1]
        lg = ops.DeviceGraph.from_host(host.row_block(r0, r1, transposed_values=True), dev, seg_len=32)
        b2 = [(torch.from_numpy(rng.integers(0, ds.n_users, 48)).to(dev),
               torch.from_numpy(rng.integers(0, ds.m_items, 48)).to(dev),
               torch.from_numpy(rng.integers(0, 2, 48)).float().to(dev)) for _ in range(3)]
        got = {}
        for rf in (False, True):
            prop = PartitionedPropagator(lg, bounds, 64, 3, mode="push", device=dev)
            prop.e0_exchange = "push"
            tr = PartitionedTrainer(prop, W0[r0:r1].clone(), ds.n_users + 1, lr=1e-2, keep_prob=KP)
            tr.receptive_field = rf
            if rf:
                sets = prop.receptive_sets(torch.unique(torch.cat([b2[0][0], b2[0][1] + ds.n_users + 1])))
                engaged = sets[3] is not None and sets[2] is not None
            torch.manual_seed(900)
            ls = [float(tr.step(*b)) for b in b2]
            torch.cuda.synchronize()
            got[rf] = (ls, tr.W.clone())
            prop.close()
        res[f"receptive/w{weighted}"] = engaged and got[True][0] == got[False][0] and torch.equal(got[True][1],
                                                                                                 got[False][1])


def _worker(rank, world, port, q):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    torch.cuda.set_device(rank)
    dev = torch.device("cuda", rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
    try:
        res = {}
        try:
            _forward(rank, world, dev, res)
            _train(rank, world, dev, res)
        except Exception:   # reported, not hung: the parent waits on the queue
            import traceback

            res["error"] = traceback.format_exc()
        q.put((rank, res))
    finally:
        dist.destroy_process_group()


@pytest.mark.parametrize("world", [1, 2])
def test_partitioned_dropout_matches_single_gpu(world):
    if torch.cuda.device_count() < world:
        pytest.skip(f"needs {world} GPUs")
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_worker, args=(r, world, port, q)) for r in range(world)]
    for p in procs:
        p.start()
    out = [q.get(timeout=600) for _ in range(world)]
    for p in procs:
        p.join(60)
        assert p.exitcode == 0
    for rank, res in out:
        assert "error" not in res, (rank, res.get("error"))
        for key, v in res.items():
            if key.startswith("train/"):
                first_equal, lerr, werr, differs = v
                assert first_equal, (rank, key)          # same values, same arithmetic: bit-equal first loss
                assert lerr < 1e-5 and werr < 1e-5, (rank, key, lerr, werr)
                assert differs, (rank, key)              # the dropped values were not ignored
            else:
                assert v, (rank, key)
