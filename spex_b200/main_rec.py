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
`--test_mode fullrank` (single GPU) replaces the sampled 99+1 Test() by a full ranking of every item with the
training items masked, Recall/NDCG@[10, 20, 50] computed on the device; the printed lines keep their format.
`--loss bpr` trains upstream LightGCN's BPR loss instead of the reference's BCE: an epoch is ceil(n_train / bpr_batch)
steps of bpr_batch (user, positive, negative) triples drawn on the device, each step minimising
loss + decay * reg (LightGCN.bpr_loss); the printed lines keep their format.
"""
from __future__ import annotations

import time

import numpy as np
import torch

from . import batch_test, dataloader, ops, utils
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


def bpr_epoch_steps(n_train: int, batch: int):
    """Triples per step of one BPR epoch: ceil(n_train / batch) steps that together draw n_train triples."""
    return [min(batch, n_train - s) for s in range(0, n_train, batch)]


def bpr_triples(icsr, n_user_rows: int, m_items: int, n: int):
    """n (user, positive, negative) triples on the device from the training-interaction CSR `icsr` (rowptr, col:
    user rows over item ids, item offset 0).  The sampler's seed is drawn from torch's default CPU generator, so a
    seeded run - or every rank of a distributed one - draws the same triples."""
    from .model import dropout_seed

    rp, col = icsr
    return dataloader.uniform_sample_bpr_device(rp, col, 0, m_items, n_user_rows, n, seed=dropout_seed())


def TrainBPR(dataset, recommend_model, epoch, optimizer, decay, batch):
    """One BPR epoch: per step a fresh batch of triples, model.bpr_loss, loss + decay * reg, backward, Adam."""
    recommend_model.train()
    icsr = recommend_model.train_mask_csr()
    total = torch.zeros((), dtype=torch.float64, device=icsr[0].device)
    for n in bpr_epoch_steps(int(np.asarray(dataset.trainUser).size), batch):
        users, pos, neg = bpr_triples(icsr, recommend_model.n_user_rows, recommend_model.num_items, n)
        optimizer.zero_grad(set_to_none=True)
        loss, reg = recommend_model.bpr_loss(users, pos, neg)
        loss = loss + decay * reg
        loss.backward()
        total += loss.detach().double()
        optimizer.step()
    total_loss = float(total.item())
    print("%d,%.5f" % (epoch, total_loss))
    return total_loss


def fullrank_test(Recmodel, testRatings, Ks=batch_test.Ks):
    """Full-ranking Recall / NDCG at Ks of every user in testRatings, training items masked: {'recall', 'ndcg':
    float64 [len(Ks)]} like batch_test.test().  One ShardedEvaluator (one GPU) over computer() and the training
    mask; the metrics are computed on the device (dist.ShardedEvaluator.evaluate)."""
    from .dist import ShardedEvaluator
    from .graph import truth_csr

    users = np.fromiter(testRatings.keys(), dtype=np.int64, count=len(testRatings))
    all_users, all_items = Recmodel.computer()
    mrp, mcol = Recmodel.train_mask_csr()
    ev = ShardedEvaluator(all_users, all_items, mrp, mcol, k=max(Ks), scorer=ops.default_precision(all_items.shape[1]))
    trp, tcol = truth_csr(users, testRatings)
    ret = ev.evaluate(torch.from_numpy(users).to(all_items.device), trp, tcol, Ks)
    return {"recall": ret["recall"], "ndcg": ret["ndcg"]}


def Test(dataset, Recmodel, epoch, best_recall, best_ndcg, best_iter, test_mode="sampled"):
    Recmodel = Recmodel.eval()
    with torch.no_grad():
        if test_mode == "fullrank":
            ret = fullrank_test(Recmodel, dataset.testRatings)
        else:
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
    visited in the single-GPU order, rank 0 prints the reference's lines.  Edge dropout runs with the
    device mask (`--dropout 2`): every rank makes the dropped values of its own rows, the same edges a
    one-GPU run with the same --seed drops.  `--loss bpr`: every rank samples the one-GPU run's triples
    (same interaction CSR, same seeds) and runs PartitionedTrainer.bpr_step."""
    import os

    import torch.distributed as dist

    from . import ops
    from .dist import PartitionedPropagator, PartitionedTrainer
    from .graph import partition_rows_by_nnz

    if args.dropout not in (0, 2):
        # the reference's mask is one torch.rand(nnz) stream over the whole graph: every rank would need all of
        # it and the global transpose map
        raise SystemExit(f"--dropout {args.dropout} is not supported with torchrun: use --dropout 2, the device "
                         "mask, which every rank generates for its own rows")
    if getattr(args, "test_mode", "sampled") != "sampled":
        raise SystemExit("--test_mode fullrank is not supported with torchrun: run it on one GPU")
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
    lg = ops.DeviceGraph.from_host(host.row_block(r0, r1, transposed_values=bool(args.dropout)), device, D_hint=D)
    prop = PartitionedPropagator(lg, bounds, D, K, mode="nccl", device=device)
    bpr = getattr(args, "loss", "bce") == "bpr"
    trainer = PartitionedTrainer(prop, model._table[r0:r1].detach().to(device).contiguous(), nur, lr=args.lr,
                                 keep_prob=args.keepprob if args.dropout else None,
                                 decay=getattr(args, "decay", 1e-4))
    if bpr:
        rp, col = dataset.getInteractionCSR()
        icsr = (torch.as_tensor(rp, dtype=torch.int64).to(device), torch.as_tensor(col, dtype=torch.int32).to(device))
    best_recall, best_ndcg, best_iter = [0, 0, 0], [0, 0, 0], [0, 0]
    for epoch in range(args.epochs):
        total = torch.zeros((), dtype=torch.float64, device=device)
        if bpr:
            for n in bpr_epoch_steps(int(dataset.trainUser.size), getattr(args, "bpr_batch", 2048)):
                total += trainer.bpr_step(*bpr_triples(icsr, nur, model.num_items, n)).double().reshape(())
        else:
            train_dataset.ng_sample()
            users, items, labels = (torch.from_numpy(a) for a in train_dataset.arrays())
            users_d, items_d = users.to(device), items.to(device)
            labels_d = labels.to(device=device, dtype=torch.float32)
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
            if getattr(args, "loss", "bce") == "bpr":
                TrainBPR(dataset, Recmodel, epoch, optimizer, getattr(args, "decay", 1e-4),
                         getattr(args, "bpr_batch", 2048))
            else:
                Train(train_dataset, Recmodel, epoch, optimizer, device)
            best_recall, best_ndcg, best_iter = Test(dataset, Recmodel, epoch, best_recall, best_ndcg, best_iter,
                                                     getattr(args, "test_mode", "sampled"))
            _ = time.time() - start
    finally:
        ops.enable_persistent_workspaces(False)
    print("--- Train Best ---")
    print("Rec:  recall=[%.4f, %.4f, %.4f],  ndcg=[%.4f, %.4f, %.4f]" % (
        best_recall[0], best_recall[1], best_recall[2], best_ndcg[0], best_ndcg[1], best_ndcg[2]))


if __name__ == "__main__":
    main()
