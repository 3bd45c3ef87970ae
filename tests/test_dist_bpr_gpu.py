"""BPR training on GPUs: PartitionedTrainer.bpr_step (one process per GPU) against LightGCN.bpr_loss + decay * reg +
FusedAdam on one GPU, and `main_rec --loss bpr`.

The partitioned backward sums the powers of A^T where the one-GPU backward nests them (dist.py), so after the first
step the two agree to rounding, not bit for bit - the bar of the BCE trainer: the first loss bit-equal, losses and
weights within 1e-5 after three steps.  Within the partitioned trainer the fused tail (the L2 gradient added in the
Adam epilogue) and the unfused one (added in the last layer's Z, then spex_adam_f32) are bit-equal, and so are the
receptive field on and off.  World 2 needs two devices and is skipped below that."""
import os
import re
import shutil
import socket
import subprocess
import sys

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from helpers import make_args

pytestmark = pytest.mark.gpu

KP = 0.3
DECAY = 1e-2
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _batches(ds, dev, rng, B=256, steps=3):
    out = []
    for _ in range(steps):
        users = torch.from_numpy(rng.integers(0, ds.n_users, B))
        pos = torch.from_numpy(rng.integers(0, ds.m_items, B))
        neg = torch.from_numpy(rng.integers(0, ds.m_items, B))
        users[:40] = users[0]                    # a user row many times
        pos[30:60] = pos[30]                     # an item row as positive and as negative, in overlapping samples
        neg[50:80] = pos[30]
        users[100:110], pos[100:110], neg[100:110] = users[0], pos[30], pos[30]   # one row per role, repeated
        out.append(tuple(t.to(dev) for t in (users, pos, neg)))
    return out


def _one_gpu(ds, dev, batches, D=64, keep_prob=None, seed=500):
    from spex_b200.model import LightGCN
    from spex_b200.optim import FusedAdam

    torch.manual_seed(2020)
    kw = dict(recdim=D) if keep_prob is None else dict(recdim=D, dropout=2, keepprob=keep_prob)
    model = LightGCN(make_args(**kw), ds).to(dev)
    W0 = model._table.detach().clone()
    opt = FusedAdam(model.parameters(), lr=1e-2)
    model.train()
    torch.manual_seed(seed)
    losses = []
    for b in batches:
        opt.zero_grad(set_to_none=True)
        loss, reg = model.bpr_loss(*b)
        total = loss + DECAY * reg
        total.backward()
        opt.step()
        losses.append(float(total))
    return W0, losses, model._table.detach().clone()


def _train(rank, world, dev, res):
    from spex_b200 import ops
    from spex_b200.dataloader import SyntheticDataset
    from spex_b200.dist import PartitionedPropagator, PartitionedTrainer
    from spex_b200.graph import partition_rows_by_nnz

    rng = np.random.default_rng(0)
    ds = SyntheticDataset(400, 250, 6000, 4)
    batches = _batches(ds, dev, rng)
    host = ds.getCSR()
    bounds = partition_rows_by_nnz(host.rowptr, world)
    r0, r1 = bounds[rank], bounds[rank + 1]
    lg = ops.DeviceGraph.from_host(host.row_block(r0, r1, transposed_values=True), dev)

    def run(W0, D, mode, keep_prob, fused_tail=True, seed=500, bs=batches, part=(lg, bounds, ds), rf=True):
        graph, bnd, data = part
        a, b = bnd[rank], bnd[rank + 1]
        prop = PartitionedPropagator(graph, bnd, D, 3, mode=mode, device=dev)
        if mode == "push":
            prop.e0_exchange = "push"
        tr = PartitionedTrainer(prop, W0[a:b].clone(), data.n_users + 1, lr=1e-2, keep_prob=keep_prob,
                                fused_tail=fused_tail, decay=DECAY)
        tr.receptive_field = rf
        torch.manual_seed(seed)
        ls = [float(tr.bpr_step(*b)) for b in bs]
        torch.cuda.synchronize()
        prop.close()
        return ls, tr.W.clone()

    def compare(key, got, ref):
        (ls, W), (ref_ls, W_ref) = got, ref
        werr = float((W - W_ref[r0:r1]).abs().max() / W_ref.abs().max())
        lerr = max(abs(a - b) / abs(b) for a, b in zip(ls, ref_ls))
        res[key] = (ls[0] == ref_ls[0], lerr, werr)

    for keep_prob in (None, KP):
        W0, ref_ls, W_ref = _one_gpu(ds, dev, batches, keep_prob=keep_prob)
        for mode in ("nccl", "push"):
            got = run(W0, 64, mode, keep_prob)
            compare(f"train/kp{keep_prob}/{mode}", got, (ref_ls, W_ref))
            if mode == "push":    # the L2 gradient in the Adam epilogue = in Z followed by spex_adam_f32
                unfused = run(W0, 64, mode, keep_prob, fused_tail=False)
                res[f"fused_tail/kp{keep_prob}"] = got[0] == unfused[0] and torch.equal(got[1], unfused[1])
    W0, ref_ls, W_ref = _one_gpu(ds, dev, batches, D=48)
    compare("train/D48/nccl", run(W0, 48, "nccl", None), (ref_ls, W_ref))
    # receptive field on and off: bit-identical (a graph large enough for the restriction to engage)
    ds2 = SyntheticDataset(20000, 8000, 150000, 8)
    host2 = ds2.getCSR()
    bounds2 = partition_rows_by_nnz(host2.rowptr, world)
    lg2 = ops.DeviceGraph.from_host(host2.row_block(bounds2[rank], bounds2[rank + 1], transposed_values=True), dev,
                                    seg_len=32)
    torch.manual_seed(11)
    from spex_b200.model import LightGCN

    W2 = LightGCN(make_args(), ds2)._table.detach().clone().to(dev)
    b2 = _batches(ds2, dev, rng, B=48)
    prop = PartitionedPropagator(lg2, bounds2, 64, 3, mode="push", device=dev)
    u, p_, n_ = b2[0]
    sets = prop.receptive_sets(torch.unique(torch.cat([u, p_ + ds2.n_users + 1, n_ + ds2.n_users + 1])))
    engaged = sets[3] is not None and sets[2] is not None
    prop.close()
    on = run(W2, 64, "push", KP, seed=900, bs=b2, part=(lg2, bounds2, ds2), rf=True)
    off = run(W2, 64, "push", KP, seed=900, bs=b2, part=(lg2, bounds2, ds2), rf=False)
    res["receptive"] = engaged and on[0] == off[0] and torch.equal(on[1], off[1])


def _worker(rank, world, port, q):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    torch.cuda.set_device(rank)
    dev = torch.device("cuda", rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
    try:
        res = {}
        try:
            _train(rank, world, dev, res)
        except Exception:   # reported, not hung: the parent waits on the queue
            import traceback

            res["error"] = traceback.format_exc()
        q.put((rank, res))
    finally:
        dist.destroy_process_group()


@pytest.mark.parametrize("world", [1, 2])
def test_partitioned_bpr_matches_single_gpu(world):
    if torch.cuda.device_count() < world:
        pytest.skip(f"needs {world} GPUs")
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_worker, args=(r, world, port, q)) for r in range(world)]
    for p in procs:
        p.start()
    out = [q.get(timeout=900) for _ in range(world)]
    for p in procs:
        p.join(60)
        assert p.exitcode == 0
    for rank, res in out:
        assert "error" not in res, (rank, res.get("error"))
        for key, v in res.items():
            if key.startswith("train/"):
                first_equal, lerr, werr = v
                assert first_equal, (rank, key)          # same rows, same loss kernel: bit-equal first loss
                assert lerr < 1e-5 and werr < 1e-5, (rank, key, lerr, werr)
            else:
                assert v, (rank, key)


# ---- the entry point -------------------------------------------------------------------------------------------
@pytest.fixture()
def tiny_root(tmp_path):
    shutil.copytree(os.path.join(ROOT, "tests", "golden", "tiny"), tmp_path / "tiny")
    return str(tmp_path)


_ARGS = ["--dataset", "tiny", "--epochs", "2", "--seed", "2020", "--loss", "bpr", "--bpr_batch", "64", "--lr", "0.01"]


def _lines(out):
    return [l for l in out.splitlines() if re.fullmatch(r"\d+,\d+\.\d{5}", l) or l.startswith("Rec:  ")]


def test_main_rec_bpr_prints_reference_lines(tiny_root, capsys):
    from spex_b200 import main_rec

    runs = []
    for _ in range(2):
        main_rec.main(_ARGS + ["--data_path", tiny_root])
        runs.append(capsys.readouterr().out)
    lines = _lines(runs[0])
    epoch_lines = [l for l in lines if "," in l and not l.startswith("Rec")]
    rec_lines = [l for l in lines if l.startswith("Rec:  Epoch ")]
    assert len(epoch_lines) == 2 and len(rec_lines) == 2
    assert re.fullmatch(r"Rec:  Epoch \d+ : recall=\[\d\.\d{4}, \d\.\d{4}, \d\.\d{4}\],  ndcg=\[\d\.\d{4}, \d\.\d{4}, "
                        r"\d\.\d{4}\]", rec_lines[0])
    assert "--- Train Best ---" in runs[0]
    assert float(epoch_lines[1].split(",")[1]) < float(epoch_lines[0].split(",")[1])
    assert _lines(runs[1]) == lines                      # one --seed, one run


def test_main_rec_bpr_torchrun_prints_the_one_gpu_lines(tiny_root, capsys):
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    from spex_b200 import main_rec

    main_rec.main(_ARGS + ["--data_path", tiny_root])
    one = _lines(capsys.readouterr().out)
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nproc-per-node", "2", "-m",
                        "spex_b200.main_rec"] + _ARGS + ["--data_path", tiny_root],
                       cwd=ROOT, capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stderr[-3000:]
    assert _lines(r.stdout) == one
