"""Edge dropout with the counter-based device mask (--dropout 2, spex_edge_dropout_f32).

The mask is a contract: edge (r, c) is kept iff int(u + keep_prob) != 0 in fp32, with u the top 24 bits of
SplitMix64(seed ^ (r << 32 | c)) scaled to [0, 1).  The numpy replica below is written from that definition alone;
the CPU tests check its statistics, the GPU tests check the kernel against it bit for bit and the model against the
oracle on the replicated mask."""
import os

import numpy as np
import pytest
import torch

from helpers import make_args, oracle_graph, random_graph, rel_err
from oracle import lightgcn_oracle as O


def splitmix64(x):
    x = np.asarray(x, dtype=np.uint64)
    x = x + np.uint64(0x9E3779B97F4A7C15)
    x = (x ^ (x >> np.uint64(30))) * np.uint64(0xBF58476D1CE4E5B9)
    x = (x ^ (x >> np.uint64(27))) * np.uint64(0x94D049BB133111EB)
    return x ^ (x >> np.uint64(31))


def mask_u(seed, rows, cols):
    """u in [0, 1) of every edge (global row, column; bit 31 of the column ignored), float32."""
    r = np.asarray(rows, dtype=np.int64).astype(np.uint64)
    c = (np.asarray(cols, dtype=np.int64) & 0x7FFFFFFF).astype(np.uint64)
    h = splitmix64(np.uint64(seed) ^ ((r << np.uint64(32)) | c))
    return (h >> np.uint64(40)).astype(np.float32) * np.float32(2.0 ** -24)


def mask_keep(seed, rows, cols, keep_prob):
    return (mask_u(seed, rows, cols) + np.float32(keep_prob)).astype(np.int32) != 0


def _pairs(n, seed):
    rng = np.random.default_rng(seed)
    return rng.integers(0, 15_000_000, n), rng.integers(0, 15_000_000, n)


# ---- CPU: the replica and the statistics of the mask -------------------------------------------------------------
def test_splitmix64_is_the_standard_finaliser():
    # first outputs of the SplitMix64 generator seeded with 0 (state advances by the golden gamma)
    g = 0x9E3779B97F4A7C15
    got = splitmix64(np.array([0, g, (2 * g) & (2 ** 64 - 1)], dtype=np.uint64))
    assert [hex(int(v)) for v in got] == ["0xe220a8397b1dcdaf", "0x6e789e6aa1b965f4", "0x6c45d188009454f"]


@pytest.mark.parametrize("kp", [0.3, 0.6])
def test_kept_fraction_is_keep_prob(kp):
    n = 2_000_000
    r, c = _pairs(n, 1)
    frac = mask_keep(12345, r, c, kp).mean()
    assert abs(frac - kp) < 5 * np.sqrt(kp * (1 - kp) / n), frac


@pytest.mark.parametrize("kp", [0.3, 0.6])
def test_both_directions_are_independent_draws(kp):
    n = 2_000_000
    r, c = _pairs(n, 2)
    both = (mask_keep(777, r, c, kp) & mask_keep(777, c, r, kp)).mean()
    p = kp * kp
    assert abs(both - p) < 5 * np.sqrt(p * (1 - p) / n), both


def test_keep_prob_one_keeps_everything():
    r, c = _pairs(2_000_000, 3)
    assert mask_keep(9, r, c, 1.0).all()


def test_same_seed_same_mask_other_seed_other_mask():
    r, c = _pairs(200_000, 4)
    a = mask_keep(2020, r, c, 0.5)
    assert np.array_equal(a, mask_keep(2020, r, c, 0.5))
    assert (a != mask_keep(2021, r, c, 0.5)).mean() > 0.4


def test_hot_bit_is_ignored_by_the_replica():
    r, c = _pairs(1000, 5)
    assert np.array_equal(mask_u(1, r, c), mask_u(1, r, c | (1 << 31)))


# ---- GPU -------------------------------------------------------------------------------------------------------
def _edges(g):
    """(global rows, columns without the hot flag) of a DeviceGraph, numpy int64 in CSR order."""
    rp = g.rowptr.cpu().numpy()
    rows = np.repeat(np.arange(g.n_rows, dtype=np.int64), np.diff(rp)) + g.row_offset
    return rows, g.col.cpu().numpy().astype(np.int64) & 0x7FFFFFFF


def _weighted_graph(dev):
    """Hub items (rows longer than a warp's chunk), the empty padding-user row and duplicate pairs (weight 3)."""
    from spex_b200 import ops
    from spex_b200.graph import build_norm_adj

    nu, m = 5000, 400
    u, i = random_graph(nu, m, 40000, 31, hub_items=3, hub_degree=3000)
    u = np.concatenate([u, u[::7], u[::7]])
    i = np.concatenate([i, i[::7], i[::7]])
    g = ops.DeviceGraph.from_host(build_norm_adj(u, i, nu + 1, m), dev)
    assert int(g.rowptr[nu + 1] - g.rowptr[nu]) == 0            # padding user
    assert int((g.rowptr[1:] - g.rowptr[:-1]).max()) > 2048     # hub rows span several chunks
    return g


@pytest.mark.gpu
@pytest.mark.parametrize("kp", [0.3, 0.6, 1.0])
def test_same_bits_as_the_host_mask_path(cuda_device, kp):
    g = _weighted_graph(cuda_device)
    vals = g.val.cpu()
    tpos = g.tpos.cpu()
    assert not torch.equal(vals, vals[tpos])   # weighted: tpos mode is required
    seed = 0x1234_5678_9ABC
    val, valT = g.device_dropout_values(seed, kp)
    rows, cols = _edges(g)
    keep = torch.from_numpy(mask_keep(seed, rows, cols, kp))
    assert torch.equal(val, g.dropout_values(keep, kp))
    assert torch.equal(valT, g.transposed_values(val))
    if kp < 1:
        assert abs(float(keep.float().mean()) - kp) < 0.02


def _symmetric_device_graph(dev, nu=3000, m=700, n=30000):
    from spex_b200 import synthetic

    keys = synthetic.generate_interactions(nu, m, n, seed=7, device=dev)
    g, _, _ = synthetic.build_norm_adj_device(keys, nu, m, seg_len=256)
    return g


@pytest.mark.gpu
def test_no_tpos_mode_on_bit_symmetric_values(cuda_device):
    from spex_b200 import ops
    from spex_b200.graph import CSRGraph, transpose_positions

    g = _symmetric_device_graph(cuda_device)
    assert g.tpos is None and g.values_symmetric
    host = CSRGraph(g.n_rows, g.n_cols, g.rowptr.cpu().numpy(), g.clean_col().cpu().numpy(), g.val.cpu().numpy())
    tpos = torch.from_numpy(transpose_positions(host)).to(cuda_device)
    assert torch.equal(g.val, g.val[tpos])
    gt = ops.DeviceGraph(g.rowptr, g.col, g.val, g.n_cols, tpos, g.seg_len)
    for kp in (0.3, 1.0):
        a = g.device_dropout_values(99, kp)
        b = gt.device_dropout_values(99, kp)
        assert torch.equal(a[0], b[0]) and torch.equal(a[1], b[1])
    bare = ops.DeviceGraph(g.rowptr, g.col, g.val, g.n_cols, None, g.seg_len)
    with pytest.raises(RuntimeError, match="transpose map"):
        bare.device_dropout_values(99, 0.3)


@pytest.mark.gpu
def test_hot_bit_changes_no_output(cuda_device):
    from spex_b200 import ops

    g = _weighted_graph(cuda_device)
    col = g.col.clone()
    col[::3] |= torch.tensor(-(2 ** 31), dtype=torch.int32, device=cuda_device)
    gh = ops.DeviceGraph(g.rowptr, col, g.val, g.n_cols, g.tpos, g.seg_len, col_hot=True)
    a = g.device_dropout_values(5, 0.4)
    b = gh.device_dropout_values(5, 0.4)
    assert torch.equal(a[0], b[0]) and torch.equal(a[1], b[1])


@pytest.mark.gpu
def test_row_block_generates_its_own_rows(cuda_device):
    from spex_b200 import ops
    from spex_b200.graph import build_norm_adj

    nu, m = 5000, 400
    u, i = random_graph(nu, m, 40000, 32, hub_items=2, hub_degree=3000)
    host = build_norm_adj(u, i, nu + 1, m)    # unit weights, no duplicates: values symmetric bit for bit
    full = ops.DeviceGraph.from_host(host, cuda_device)
    val, valT = full.device_dropout_values(42, 0.3)
    for r0, r1 in ((0, 1200), (nu - 10, nu + 150), (nu + 1, nu + 1 + m)):   # users, across the padding row, items
        blk = ops.DeviceGraph.from_host(host.row_block(r0, r1), cuda_device)
        assert blk.row_offset == r0 and blk.tpos is None
        blk.values_symmetric = True
        bv, bvt = blk.device_dropout_values(42, 0.3)
        lo, hi = int(host.rowptr[r0]), int(host.rowptr[r1])
        assert torch.equal(bv, val[lo:hi]) and torch.equal(bvt, valT[lo:hi])


def _small_model(dev, **kw):
    from spex_b200.dataloader import SyntheticDataset
    from spex_b200.model import LightGCN

    ds = SyntheticDataset(400, 250, 6000, seed=4)
    torch.manual_seed(2020)
    model = LightGCN(make_args(**kw), ds)
    ref_w = (model.embedding_user.weight.detach().clone(), model.embedding_item.weight.detach().clone())
    A = oracle_graph(ds.trainUser, ds.trainItem, ds.n_users + 1, ds.m_items)
    return ds, model.to(dev), ref_w, A


@pytest.mark.gpu
def test_model_matches_oracle_on_the_replicated_mask(cuda_device):
    from spex_b200.model import dropout_seed

    ds, model, (uw, iw), A = _small_model(cuda_device, dropout=2, keepprob=0.3)
    users = torch.arange(64) % ds.n_users
    items = torch.arange(64) % ds.m_items
    labels = torch.arange(64) % 2
    torch.manual_seed(77)
    seed = dropout_seed()
    A = A.coalesce()
    idx = A.indices().numpy()
    u = torch.from_numpy(mask_u(seed, idx[0], idx[1]))
    Adrop = O.dropout_graph(A, 0.3, rand=u)
    uw.requires_grad_(True)
    iw.requires_grad_(True)
    ru, ri = O.computer(uw, iw, Adrop, 3)
    ref = torch.nn.BCEWithLogitsLoss()(O.gamma(ru, ri, users, items), labels.float())
    ref.backward()
    model.train()
    torch.manual_seed(77)
    loss = model(users.to(cuda_device), items.to(cuda_device), labels.to(cuda_device), flag=0)
    loss.backward()
    assert abs(float(loss) - float(ref)) <= 1e-5 * abs(float(ref))
    assert rel_err(model.embedding_user.weight.grad, uw.grad) < 1e-5
    assert rel_err(model.embedding_item.weight.grad, iw.grad) < 1e-5


@pytest.mark.gpu
def test_receptive_field_step_same_bits_with_device_dropout(cuda_device):
    from spex_b200 import ops
    from spex_b200.dataloader import SyntheticDataset
    from spex_b200.model import LightGCN

    ds = SyntheticDataset(20000, 8000, 150000, seed=8)
    torch.manual_seed(2020)
    model = LightGCN(make_args(dropout=2, keepprob=0.7), ds).to(cuda_device)
    model.train()
    rng = np.random.default_rng(4)
    ops.enable_persistent_workspaces(True)
    try:
        for step in range(2):
            B = 48
            users = torch.from_numpy(rng.integers(0, ds.n_users, B)).to(cuda_device)
            items = torch.from_numpy(rng.integers(0, ds.m_items, B)).to(cuda_device)
            labels = torch.from_numpy(rng.integers(0, 2, B)).to(cuda_device)
            res = {}
            for rf in (False, True):
                model.receptive_field = rf
                model.zero_grad(set_to_none=True)
                torch.manual_seed(100 + step)            # same mask seed in both runs
                loss = model(users, items, labels, flag=0)
                loss.backward()
                res[rf] = (loss.detach().clone(), model.embedding_user.weight.grad.clone(),
                           model.embedding_item.weight.grad.clone())
            for a, b in zip(res[True], res[False]):
                assert torch.equal(a, b)
    finally:
        model.receptive_field = True
        ops.enable_persistent_workspaces(False)


@pytest.mark.gpu
def test_seeded_runs_reproduce_and_eval_does_no_dropout(cuda_device):
    ds, model, _, _ = _small_model(cuda_device, dropout=2, keepprob=0.3)
    users = (torch.arange(64) % ds.n_users).to(cuda_device)
    items = (torch.arange(64) % ds.m_items).to(cuda_device)
    labels = (torch.arange(64) % 2).to(cuda_device)
    model.train()
    losses = []
    for s in (5, 5, 6):
        torch.manual_seed(s)
        with torch.no_grad():
            losses.append(model(users, items, labels, flag=0))
    assert torch.equal(losses[0], losses[1])
    assert not torch.equal(losses[0], losses[2])
    g = model.device_graph()
    a, _ = g.device_dropout_values(5, 0.3)
    b, _ = g.device_dropout_values(6, 0.3)
    assert not torch.equal(a, b)
    _, plain, _, _ = _small_model(cuda_device, dropout=0, keepprob=0.3)
    model.eval()
    plain.eval()
    with torch.no_grad():
        assert torch.equal(model(users, items, None, flag=1), plain(users, items, None, flag=1))


@pytest.mark.gpu
def test_bad_arguments_are_rejected(cuda_device):
    from spex_b200 import _capi
    from spex_b200._capi import ptr

    g = _symmetric_device_graph(cuda_device, 300, 100, 2000)
    out = torch.empty_like(g.val)
    fn = _capi.lib.spex_edge_dropout_f32
    BAD = -1

    def run(rowptr=ptr(g.rowptr), col=ptr(g.col), val=ptr(g.val), n_rows=g.n_rows, row_offset=0, kp=0.5,
            val_out=ptr(out)):
        return fn(rowptr, col, val, None, n_rows, row_offset, 1, kp, val_out, None, None)

    assert run() == 0
    for kp in (0.0, 1.5, float("nan"), -0.3):
        assert run(kp=kp) == BAD, kp
    assert run(rowptr=None) == BAD and run(col=None) == BAD and run(val=None) == BAD and run(val_out=None) == BAD
    assert run(n_rows=-1) == BAD and run(row_offset=-1) == BAD
    assert run(n_rows=0) == 0
    torch.cuda.synchronize()
    keep = torch.from_numpy(mask_keep(1, *_edges(g), 0.5)).to(cuda_device)
    assert torch.equal(out != 0, keep)   # val_out only (valT_out NULL); every value of the graph is > 0


# ---- GPU, BASELINE.json configs[3] (10 M users x 5 M items, 2e9 edges) --------------------------------------------
SCALE = float(os.environ.get("SPEX_FULLSIZE_SCALE", "1.0"))


@pytest.mark.gpu
def test_full_size_kept_fraction_and_sampled_edges(cuda_device):
    from spex_b200 import synthetic

    free, _ = torch.cuda.mem_get_info()
    if free < 60e9 * SCALE:
        pytest.skip("needs ~60 GB of free HBM")
    nu, m, ni = int(10_000_000 * SCALE), int(5_000_000 * SCALE), int(1_000_000_000 * SCALE)
    keys = synthetic.generate_interactions(nu, m, ni, seed=2020, device=cuda_device)
    g, _, _ = synthetic.build_norm_adj_device(keys, nu, m)
    del keys
    g.mark_hot_columns(64)
    kp, seed = 0.3, 0xC0FFEE
    val, valT = g.device_dropout_values(seed, kp)
    n = g.nnz
    kept = int((val != 0).sum())
    assert abs(kept / n - kp) < 5 * (kp * (1 - kp) / n) ** 0.5, kept / n
    gen = torch.Generator(device=cuda_device).manual_seed(3)
    pos = torch.randint(0, n, (1_000_000,), device=cuda_device, generator=gen)
    rows = torch.searchsorted(g.rowptr, pos, right=True) - 1
    cols = (g.col[pos] & 0x7FFFFFFF).long()
    rows_np, cols_np = rows.cpu().numpy(), cols.cpu().numpy()
    fwd = torch.from_numpy(mask_keep(seed, rows_np, cols_np, kp)).to(cuda_device)
    bwd = torch.from_numpy(mask_keep(seed, cols_np, rows_np, kp)).to(cuda_device)
    kpt = torch.full((1,), kp, device=cuda_device)   # a device tensor: IEEE division, as the kernel's
    assert torch.equal(val[pos], (g.val[pos] * fwd.float()) / kpt)
    assert torch.equal(valT[pos], (g.val[pos] * bwd.float()) / kpt)
    del val, valT, g
    torch.cuda.empty_cache()
