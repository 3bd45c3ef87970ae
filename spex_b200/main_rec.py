"""Rec-only training / evaluation entry point: `python -m spex_b200.main_rec --dataset epinion2 ...`

Same flow, same printed lines as /root/reference/LightGCN_SPEX/code/main_rec.py:
    per epoch: Train() prints '%d,%.5f' % (epoch, total_loss)                     (main_rec.py:38)
               Test()  prints 'Rec:  Epoch %d : recall=[...],  ndcg=[...]'        (main_rec.py:51-54)
    at the end '--- Train Best ---' and the best line                             (main_rec.py:72-74)
Differences in HOW: batches are sliced from the epoch's arrays with one torch.randperm (the same
draw DataLoader(shuffle=True)'s RandomSampler makes, so a shared seed visits the same batches), the
loss is accumulated on the device and read once per epoch instead of `.item()` per step
(main_rec.py:36), Test() propagates once instead of once per user (batch_test.py:33), and the
optimiser is the fused dense Adam.
"""
from __future__ import annotations

import time

import numpy as np
import torch

from . import batch_test, dataloader, utils
from .lg_parser import parse_args_r
from .model import LightGCN
from .optim import FusedAdam

BATCH = 256  # hard-coded in the reference (main_rec.py:20)


def epoch_batches(n: int, batch: int, generator=None):
    """Index batches in the order DataLoader(shuffle=True) would produce them, consuming the default
    generator identically: the DataLoader iterator draws its base seed (one int64), then the
    RandomSampler draws its own seed (one int64) and shuffles with torch.randperm(n, seeded)."""
    torch.empty((), dtype=torch.int64).random_(generator=generator)  # DataLoader's _base_seed
    seed = int(torch.empty((), dtype=torch.int64).random_(generator=generator).item())
    g = torch.Generator()
    g.manual_seed(seed)
    perm = torch.randperm(n, generator=g)
    return [perm[i: i + batch] for i in range(0, n, batch)]


def Train(train_dataset, recommend_model, epoch, optimizer, device, batch=BATCH):
    train_dataset.ng_sample()
    recommend_model.train()
    users, items, labels = (torch.from_numpy(a) for a in train_dataset.arrays())
    # the epoch's samples live on the device; each step slices its batch there
    users_d, items_d = users.to(device), items.to(device)
    labels_d = labels.to(device=device, dtype=torch.float32)
    total = torch.zeros((), dtype=torch.float64, device=device)
    for idx in epoch_batches(users.numel(), batch):
        idx = idx.to(device)
        optimizer.zero_grad(set_to_none=True)
        loss = recommend_model(users=users_d[idx], items=items_d[idx], labels=labels_d[idx], flag=0)
        loss.backward()
        total += loss.detach().double()
        optimizer.step()
    total_loss = float(total.item())
    print("%d,%.5f" % (epoch, total_loss))
    return total_loss


def Test(dataset, Recmodel, epoch, best_recall, best_ndcg, best_iter):
    Recmodel = Recmodel.eval()
    with torch.no_grad():
        ret = batch_test.test(Recmodel, dataset.testRatings, dataset.testNegatives)
    perf_str = "Rec:  Epoch %d : recall=[%.4f, %.4f, %.4f],  ndcg=[%.4f, %.4f, %.4f]" % (
        epoch, ret["recall"][0], ret["recall"][1], ret["recall"][2], ret["ndcg"][0], ret["ndcg"][1],
        ret["ndcg"][2])
    print(perf_str)
    if ret["recall"][0] > best_recall[0]:
        best_recall, best_iter[0] = ret["recall"], epoch
    if ret["ndcg"][0] > best_ndcg[0]:
        best_ndcg, best_iter[1] = ret["ndcg"], epoch
    return best_recall, best_ndcg, best_iter


class _GatheredTables:
    """What batch_test.test() needs from a model, backed by the all-gathered propagated table."""

    def __init__(self, table, n_user_rows):
        self._t, self._n = table, n_user_rows

    def final_embeddings(self):
        return self._t[: self._n], self._t[self._n:]

    computer = final_embeddings


def main_distributed(args):
    """`torchrun --nproc-per-node P -m spex_b200.main_rec ...`: the same epochs with the table, its
    gradient and the Adam moments row-partitioned over P GPUs (spex_b200.dist.PartitionedTrainer).
    Every rank runs the same seeded host-side sampling (replicated, no communication), the batches are
    visited in the single-GPU order, rank 0 prints the reference's lines.  Edge dropout is not
    supported in this mode (the partitioned backward relies on the symmetric adjacency)."""
    import os

    import torch.distributed as dist

    from . import ops
    from .dist import PartitionedPropagator, PartitionedTrainer
    from .graph import partition_rows_by_nnz

    if args.dropout:
        raise SystemExit(f"--dropout {args.dropout} is not supported with torchrun (row-partitioned backward needs the symmetric graph)")
    rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
    local_rank = int(os.environ.get("LOCAL_RANK", rank))
    torch.cuda.set_device(local_rank)
    device = torch.device("cuda", local_rank)
    dist.init_process_group("nccl", device_id=device)
    utils.set_seed(args.seed)
    import contextlib
    import io

    with (contextlib.nullcontext() if rank == 0 else contextlib.redirect_stdout(io.StringIO())):
        dataset = dataloader.Loader(args)
    train_dataset = dataloader.LightTrainData(dataset.rec_train_data, dataset.m_item, dataset.train_mat)
    model = LightGCN(args, dataset)            # same RNG consumption as one GPU => same initial weights
    nur, D, K = model.n_user_rows, model.latent_dim, model.n_layers
    host = dataset.getCSR()
    bounds = partition_rows_by_nnz(host.rowptr, world)
    r0, r1 = bounds[rank], bounds[rank + 1]
    lg = ops.DeviceGraph.from_host(host.row_block(r0, r1), device, D_hint=D)
    prop = PartitionedPropagator(lg, bounds, D, K, mode="nccl", device=device)
    trainer = PartitionedTrainer(prop, model._table[r0:r1].detach().to(device).contiguous(), nur, lr=args.lr)
    best_recall, best_ndcg, best_iter = [0, 0, 0], [0, 0, 0], [0, 0]
    for epoch in range(args.epochs):
        train_dataset.ng_sample()
        users, items, labels = (torch.from_numpy(a) for a in train_dataset.arrays())
        users_d, items_d = users.to(device), items.to(device)
        labels_d = labels.to(device=device, dtype=torch.float32)
        total = torch.zeros((), dtype=torch.float64, device=device)
        for idx in epoch_batches(users.numel(), BATCH):
            idx = idx.to(device)
            total += trainer.step(users_d[idx], items_d[idx], labels_d[idx]).double().reshape(())
        if rank == 0:
            print("%d,%.5f" % (epoch, float(total.item())))
        with torch.no_grad():
            table = trainer.gather_table(prop.propagate(trainer.W))
        if rank == 0:
            ret = batch_test.test(_GatheredTables(table, nur), dataset.testRatings, dataset.testNegatives)
            print("Rec:  Epoch %d : recall=[%.4f, %.4f, %.4f],  ndcg=[%.4f, %.4f, %.4f]" % (
                epoch, ret["recall"][0], ret["recall"][1], ret["recall"][2], ret["ndcg"][0], ret["ndcg"][1],
                ret["ndcg"][2]))
            if ret["recall"][0] > best_recall[0]:
                best_recall, best_iter[0] = ret["recall"], epoch
            if ret["ndcg"][0] > best_ndcg[0]:
                best_ndcg, best_iter[1] = ret["ndcg"], epoch
    if rank == 0:
        print("--- Train Best ---")
        print("Rec:  recall=[%.4f, %.4f, %.4f],  ndcg=[%.4f, %.4f, %.4f]" % (
            best_recall[0], best_recall[1], best_recall[2], best_ndcg[0], best_ndcg[1], best_ndcg[2]))
    prop.close()
    dist.destroy_process_group()


def main(argv=None):
    import os

    args = parse_args_r(argv)
    if int(os.environ.get("WORLD_SIZE", "1")) > 1:
        if not torch.cuda.is_available():
            raise SystemExit("spex_b200.main_rec needs B200s (sm_100a); there is no CPU fallback")
        return main_distributed(args)
    utils.set_seed(args.seed)
    if not torch.cuda.is_available():
        raise SystemExit("spex_b200.main_rec needs a B200 (sm_100a); there is no CPU fallback")
    device = torch.device("cuda", int(args.cuda_id))
    torch.cuda.set_device(device)
    dataset = dataloader.Loader(args)
    train_dataset = dataloader.LightTrainData(dataset.rec_train_data, dataset.m_item, dataset.train_mat)
    Recmodel = LightGCN(args, dataset).to(device)
    optimizer = FusedAdam(Recmodel.parameters(), lr=args.lr)
    from . import ops

    ops.enable_persistent_workspaces(True)   # reuse the [N, D] scratch tables of the step (ops._Workspaces)
    best_recall, best_ndcg, best_iter = [0, 0, 0], [0, 0, 0], [0, 0]
    try:
        for epoch in range(args.epochs):
            start = time.time()
            Train(train_dataset, Recmodel, epoch, optimizer, device)
            best_recall, best_ndcg, best_iter = Test(dataset, Recmodel, epoch, best_recall, best_ndcg, best_iter)
            _ = time.time() - start
    finally:
        ops.enable_persistent_workspaces(False)
    print("--- Train Best ---")
    print("Rec:  recall=[%.4f, %.4f, %.4f],  ndcg=[%.4f, %.4f, %.4f]" % (
        best_recall[0], best_recall[1], best_recall[2], best_ndcg[0], best_ndcg[1], best_ndcg[2]))


if __name__ == "__main__":
    main()
