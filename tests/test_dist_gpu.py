"""Row-partitioned propagation on real GPUs (needs >= 2 devices, skipped otherwise): the NCCL
all-gather exchange and the fused SpMM + P2P push exchange (the Y exchange of spex_spmm_layer_f32's
epilogue, spex_push_rows_f32_ex) against the single-GPU kernel on the same graph.  Same row partition as the
reference's serial folds (/root/reference/LightGCN_SPEX/code/utility1/dataloader.py:167-177)."""
import os
import socket

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from helpers import random_graph

pytestmark = pytest.mark.gpu


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _worker(rank, world, port, q):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    torch.cuda.set_device(rank)
    dev = torch.device("cuda", rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
    try:
        from spex_b200 import ops
        from spex_b200.dist import PartitionedPropagator
        from spex_b200.graph import build_norm_adj, partition_rows_by_nnz

        nu, m, D, K = 5000, 3000, 64, 3
        u, i = random_graph(nu, m, 120000, 21, hub_items=3, hub_degree=2500)
        g = build_norm_adj(u, i, nu + 1, m)
        N = g.n_rows
        full = ops.DeviceGraph(torch.from_numpy(g.rowptr).to(dev), torch.from_numpy(g.col).to(dev),
                               torch.from_numpy(g.val).to(dev), N)
        torch.manual_seed(0)
        E = (torch.randn(N, D) * 0.1).to(dev)
        want = ops.propagate_mean(E, full, K)
        bounds = partition_rows_by_nnz(g.rowptr, world)
        r0, r1 = bounds[rank], bounds[rank + 1]
        lo, hi = int(g.rowptr[r0]), int(g.rowptr[r1])
        lg = ops.DeviceGraph((full.rowptr[r0: r1 + 1] - lo).contiguous(), full.col[lo:hi].clone(),
                             full.val[lo:hi].clone(), N, None, full.seg_len, row_offset=r0)
        res = {}
        modes = [("nccl", "nccl"), ("push", "push"), ("push", "copy"), ("push", "nccl")]
        try:   # NVLS multicast needs an NVSwitch box
            probe = PartitionedPropagator(lg, bounds, D, K, mode="mcast", device=dev)
            probe.close()
            modes += [("mcast", "mcast"), ("mcast", "nccl")]
        except RuntimeError as e:
            res["mcast_unavailable"] = (True, True, ["layer3", "e0_exchange", str(e)])
        for mode, e0 in modes:
            prop = PartitionedPropagator(lg, bounds, D, K, mode=mode, device=dev)
            prop.e0_exchange = e0
            a = prop.propagate(E[r0:r1].clone())
            b = prop.propagate(E[r0:r1].clone())   # buffers are reusable, result reproducible
            prop.timing = []
            c = prop.propagate(E[r0:r1].clone())
            phases = [n for n, _ in prop.phase_ms()]
            # a sweep over different tables, each announced one call ahead (published to the peers by the
            # background kernel during the previous call's last layer), then an unannounced call
            ok_ring = True
            # (both ways of publishing: from the last layer's own epilogue, and from the side-stream kernel)
            for fuse in ((True, False) if prop.can_prefetch() else ()):
                prop.fuse_publish = fuse
                tabs = [E[r0:r1].clone(), (E[r0:r1] * 2.0 - 0.5).clone(), (E[r0:r1] * -1.0).clone(), E[r0:r1].clone()]
                outs = [prop.propagate(t, next_E0_local=tabs[j + 1] if j + 1 < len(tabs) else tabs[1])
                        for j, t in enumerate(tabs)]
                stale = prop.propagate(tabs[0])           # the announced table was tabs[1]: must be ignored
                d1 = prop.propagate(tabs[1].clone())
                d2 = prop.propagate(tabs[2].clone())
                ok_ring = ok_ring and (torch.equal(outs[0], a) and torch.equal(outs[3], a) and torch.equal(stale, a)
                                       and torch.equal(outs[1], d1) and torch.equal(outs[2], d2))
            prop.close()
            res[f"{mode}/{e0}"] = (bool(torch.equal(a, want[r0:r1])),
                                   bool(torch.equal(a, b) and torch.equal(a, c) and ok_ring), phases)
        # a width that takes the generic-D kernel (ADVICE r1: its epilogue ignored the multicast table)
        D2 = 48
        E2 = (torch.randn(N, D2, generator=torch.Generator().manual_seed(1)) * 0.1).to(dev)
        want2 = ops.propagate_mean(E2, full, K)
        for mode in [m for m, e in modes if m == e and m != "nccl"]:
            prop = PartitionedPropagator(lg, bounds, D2, K, mode=mode, device=dev)
            a2 = prop.propagate(E2[r0:r1].clone())
            prop.close()
            res[f"{mode}/D48"] = (bool(torch.equal(a2, want2[r0:r1])), True, ["layer3", "e0_exchange"])
        q.put((rank, res))
    finally:
        dist.destroy_process_group()


def test_partitioned_propagation_matches_single_gpu():
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    world = 2
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_worker, args=(r, world, port, q)) for r in range(world)]
    for p in procs:
        p.start()
    out = [q.get(timeout=300) for _ in range(world)]
    for p in procs:
        p.join(60)
        assert p.exitcode == 0
    for rank, res in out:
        for key, (exact, reproducible, phases) in res.items():
            # the row partition does not change any row's summation order: bit-identical
            assert exact and reproducible, (rank, key)
            assert "layer3" in phases and "e0_exchange" in phases


def _train_worker(rank, world, port, q):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    torch.cuda.set_device(rank)
    dev = torch.device("cuda", rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
    try:
        from helpers import make_args
        from spex_b200 import ops
        from spex_b200.dataloader import SyntheticDataset
        from spex_b200.dist import PartitionedPropagator, PartitionedTrainer, ShardedEvaluator
        from spex_b200.graph import partition_rows_by_nnz
        from spex_b200.model import LightGCN
        from spex_b200.optim import FusedAdam

        # single-GPU reference on THIS rank: the drop-in model + FusedAdam, three steps
        ds = SyntheticDataset(400, 250, 6000, seed=4)
        torch.manual_seed(2020)
        model = LightGCN(make_args(), ds).to(dev)
        W0 = model._table.detach().clone()
        opt = FusedAdam(model.parameters(), lr=1e-2)
        rng = np.random.default_rng(0)
        batches, ref_losses = [], []
        for _ in range(3):
            users = torch.from_numpy(rng.integers(0, ds.n_users, 256)).to(dev)
            users[:40] = users[0]
            items = torch.from_numpy(rng.integers(0, ds.m_items, 256)).to(dev)
            labels = torch.from_numpy(rng.integers(0, 2, 256)).float().to(dev)
            batches.append((users, items, labels))
            model.train()
            opt.zero_grad(set_to_none=True)
            loss = model(users, items, labels, flag=0)
            loss.backward()
            opt.step()
            ref_losses.append(float(loss))
        W_ref = model._table.detach().clone()
        # partitioned run over the ranks
        full = model.device_graph()
        g_host = ds.getCSR()
        N, D, K = full.n_rows, 64, 3
        bounds = partition_rows_by_nnz(g_host.rowptr, world)
        r0, r1 = bounds[rank], bounds[rank + 1]
        lo, hi = int(g_host.rowptr[r0]), int(g_host.rowptr[r1])
        lg = ops.DeviceGraph((full.rowptr[r0: r1 + 1] - lo).contiguous(), full.col[lo:hi].clone(),
                             full.val[lo:hi].clone(), N, None, full.seg_len, row_offset=r0)
        res = {}
        for mode in ("nccl", "push"):
            prop = PartitionedPropagator(lg, bounds, D, K, mode=mode, device=dev)
            if mode == "push":
                prop.e0_exchange = "push"
            tr = PartitionedTrainer(prop, W0[r0:r1].clone(), ds.n_users + 1, lr=1e-2)
            losses = [float(tr.step(*b)) for b in batches]
            werr = float((tr.W - W_ref[r0:r1]).abs().max() / W_ref.abs().max())
            res[mode] = (losses[0] == ref_losses[0], max(abs(a - b) / abs(b) for a, b in zip(losses, ref_losses)), werr)
            prop.close()
        # receptive-field forward of the partitioned trainer (layers restricted to the rows the batch depends on,
        # fused exchange of the restricted rows): a graph large enough for the restriction to engage; weights
        # after three Adam steps bit-equal to the unrestricted partitioned trainer, and to the single-GPU model
        ds2 = SyntheticDataset(20000, 8000, 150000, seed=8)
        torch.manual_seed(11)
        model2 = LightGCN(make_args(), ds2).to(dev)
        W20 = model2._table.detach().clone()
        opt2 = FusedAdam(model2.parameters(), lr=1e-2)
        b2 = []
        for _ in range(3):
            u2 = torch.from_numpy(rng.integers(0, ds2.n_users, 48)).to(dev)
            i2 = torch.from_numpy(rng.integers(0, ds2.m_items, 48)).to(dev)
            l2 = torch.from_numpy(rng.integers(0, 2, 48)).float().to(dev)
            b2.append((u2, i2, l2))
            model2.train()
            opt2.zero_grad(set_to_none=True)
            lo2 = model2(u2, i2, l2, flag=0)
            lo2.backward()
            opt2.step()
        W2_ref = model2._table.detach().clone()
        full2 = model2.device_graph()
        gh2 = ds2.getCSR()
        N2 = full2.n_rows
        bounds2 = partition_rows_by_nnz(gh2.rowptr, world)
        a0, a1 = bounds2[rank], bounds2[rank + 1]
        lo_, hi_ = int(gh2.rowptr[a0]), int(gh2.rowptr[a1])
        lg2 = ops.DeviceGraph((full2.rowptr[a0: a1 + 1] - lo_).contiguous(), full2.col[lo_:hi_].clone(),
                              full2.val[lo_:hi_].clone(), N2, None, 32, row_offset=a0)   # seg_len 32: long rows too
        got = {}
        for rf in (False, True):
            prop = PartitionedPropagator(lg2, bounds2, D, K, mode="push", device=dev)
            prop.e0_exchange = "push"
            tr = PartitionedTrainer(prop, W20[a0:a1].clone(), ds2.n_users + 1, lr=1e-2)
            tr.receptive_field = rf
            if rf:
                S2 = torch.unique(torch.cat([b2[0][0], b2[0][1] + ds2.n_users + 1]))
                sets = prop.receptive_sets(S2)
                engaged = sets[K] is not None and sets[K - 1] is not None
            ls = [float(tr.step(*b)) for b in b2]
            torch.cuda.synchronize()
            got[rf] = (ls, tr.W.clone())
            prop.close()
        werr2 = float((got[True][1] - W2_ref[a0:a1]).abs().max() / W2_ref.abs().max())
        res["receptive"] = (engaged, got[True][0] == got[False][0], bool(torch.equal(got[True][1], got[False][1])), werr2)
        # evaluation sharded by user against the single-GPU ranking
        model.eval()
        users_all = torch.arange(ds.n_users, device=dev)
        i_ref, v_ref = model.rank_topk(users_all, k=20, precision="f16")
        au, ai = model.computer()
        mrp, mcol = model.train_mask_csr()
        ev = ShardedEvaluator(au, ai, mrp, mcol, k=20)
        idx, val, (a, b) = ev.rank_topk(users_all)
        same = bool(torch.equal(idx, i_ref[a:b]) and torch.equal(val, v_ref[a:b]))
        tu = np.array([u for u in range(ds.n_users) if u in ds.testRatings for _ in ds.testRatings[u]], np.int64)
        ti = np.array([i for u in range(ds.n_users) if u in ds.testRatings for i in ds.testRatings[u]], np.int64)
        from spex_b200 import metrics
        from spex_b200.graph import build_interaction_csr
        trp, tcol = build_interaction_csr(tu, ti, ds.n_users, ds.m_items)
        mm = ev.evaluate(users_all, trp, tcol, [20])
        r1g, n1g = metrics.fullrank_recall_ndcg(i_ref.cpu().numpy(), trp, tcol, 20)
        res["eval"] = (same, abs(mm["recall"][0] - float(r1g.mean())), abs(mm["ndcg"][0] - float(n1g.mean())))
        q.put((rank, res))
    finally:
        dist.destroy_process_group()


def test_partitioned_training_and_sharded_eval_match_single_gpu():
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    world = 2
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_train_worker, args=(r, world, port, q)) for r in range(world)]
    for p in procs:
        p.start()
    out = [q.get(timeout=300) for _ in range(world)]
    for p in procs:
        p.join(60)
        assert p.exitcode == 0
    for rank, res in out:
        for mode in ("nccl", "push"):
            first_equal, lerr, werr = res[mode]
            assert first_equal, (rank, mode)             # same arithmetic on the assembled rows: bit-equal loss
            assert lerr < 1e-5 and werr < 1e-5, (rank, mode, lerr, werr)
        engaged, same_loss, same_w, werr2 = res["receptive"]
        assert engaged and same_loss and same_w and werr2 < 1e-5, (rank, res["receptive"])
        same, dr, dn = res["eval"]
        assert same and dr < 1e-12 and dn < 1e-12, (rank, res["eval"])
