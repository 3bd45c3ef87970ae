"""Receptive-field training step (spex_spmm_csr_rows_f32, ops._PropagateMeanRows): restricting every layer to
the rows a mini-batch depends on must not change a single bit of what the batch sees - its rows of the layer
mean, the loss, and the gradient of the whole embedding table - against the full computer() of
LightGCN_SPEX/code/utility1/model.py:66-97 + main_rec.py:34-35, which stays the semantics."""
import numpy as np
import pytest
import torch

from helpers import make_args, oracle_graph, random_graph, rel_err
from oracle import lightgcn_oracle as O

pytestmark = pytest.mark.gpu


def _graph(dev, seg_len, nu=20000, m=8000, n_inter=120000, hubs=6, hub_degree=900):
    from spex_b200 import ops
    from spex_b200.graph import build_norm_adj

    u, i = random_graph(nu, m, n_inter, 21, hub_items=hubs, hub_degree=hub_degree)
    return ops.DeviceGraph.from_host(build_norm_adj(u, i, nu + 1, m), dev, seg_len=seg_len), nu + 1, m


@pytest.mark.parametrize("blocked", [False, True])
def test_row_subset_layer_is_bit_identical_on_both_plan_shapes(cuda_device, blocked, monkeypatch):
    """One layer on a row list (short rows, long rows through their segments, an empty row) = the same rows of
    the full layer; the rows outside the list are left untouched.  Both long-row plans."""
    from spex_b200 import ops

    if blocked:   # column-blocked segment list, forced on a small table
        monkeypatch.setattr(ops.DeviceGraph, "L2_WINDOW_BYTES", 64 * 1024)
        monkeypatch.setattr(ops.DeviceGraph, "MIN_CB_COLS", 64)
        monkeypatch.setattr(ops.DeviceGraph, "HUB_EDGES_PER_BLOCK", 4)
    g, nur, m = _graph(cuda_device, seg_len=32)
    assert g.n_long > 0 and (g.n_hub_seg > 0) == blocked
    N, D = nur + m, 64
    torch.manual_seed(3)
    X = torch.randn(N, D, device=cuda_device)
    add = torch.randn(N, D, device=cuda_device)
    Yf, Zf = torch.empty_like(X), torch.empty_like(X)
    ops.spmm(g, X, Y=Yf, addend=add, addend_scale=1.0, Z=Zf, z_scale=0.25)
    gen = torch.Generator().manual_seed(5)
    rows = torch.randperm(N, generator=gen)[:3000]
    long_ids = g.long_rows[:4].long().cpu()
    rows = torch.unique(torch.cat([rows, long_ids, torch.tensor([nur - 1])])).to(cuda_device)   # + hubs + padding user
    sub = g.row_subset(rows)
    assert sub[1] is not None and sub[1].numel() >= 4
    Y = torch.full_like(X, 7.0)
    Z = torch.full_like(X, 7.0)
    ops.spmm_rows(g, X, sub, Y=Y, addend=add, addend_scale=1.0, Z=Z, z_scale=0.25)
    assert torch.equal(Y[rows], Yf[rows]) and torch.equal(Z[rows], Zf[rows])
    other = torch.ones(N, dtype=torch.bool, device=cuda_device)
    other[rows] = False
    assert bool((Y[other] == 7.0).all()) and bool((Z[other] == 7.0).all())
    # D = 32 / 128 take the same path
    for D2 in (32, 128):
        X2 = torch.randn(N, D2, device=cuda_device)
        Yf2 = ops.spmm(g, X2)
        Y2 = torch.zeros_like(X2)
        ops.spmm_rows(g, X2, sub, Y=Y2)
        assert torch.equal(Y2[rows], Yf2[rows])


@pytest.mark.parametrize("blocked", [False, True])
@pytest.mark.parametrize("frac", [0.002, 0.08, 0.6])
def test_sparse_input_mask_is_bit_identical(cuda_device, blocked, frac, monkeypatch):
    """x_nonzero: a table that is zero outside a marked row set gives the same bits whether the zero rows are
    gathered (dense layer) or skipped (masked kernels) - all rows and a row subset, D = 64 / 32 / 128, ragged
    tails, long rows, both long-row plans, from almost empty to mostly full masks."""
    from spex_b200 import ops

    if blocked:
        monkeypatch.setattr(ops.DeviceGraph, "L2_WINDOW_BYTES", 64 * 1024)
        monkeypatch.setattr(ops.DeviceGraph, "MIN_CB_COLS", 64)
        monkeypatch.setattr(ops.DeviceGraph, "HUB_EDGES_PER_BLOCK", 4)
    g, nur, m = _graph(cuda_device, seg_len=32)
    N = nur + m
    gen = torch.Generator().manual_seed(int(frac * 1000))
    nzrows = torch.randperm(N, generator=gen)[: max(int(N * frac), 3)].to(cuda_device)
    mask = ops.nonzero_mask(N, nzrows)
    for D in (64, 32, 128):
        torch.manual_seed(D)
        X = torch.zeros(N, D, device=cuda_device)
        X[nzrows] = torch.randn(nzrows.numel(), D, device=cuda_device)
        add = torch.randn(N, D, device=cuda_device)
        Zd = torch.empty_like(X)
        ops.spmm(g, X, addend=add, Z=Zd, z_scale=0.5)
        Zm = torch.empty_like(X)
        ops.spmm_rows(g, X, None, addend=add, Z=Zm, z_scale=0.5, x_nonzero=mask)
        assert torch.equal(Zm, Zd)
        rows = torch.unique(torch.cat([torch.randperm(N, generator=gen)[:2000], g.long_rows[:3].long().cpu()])).to(cuda_device)
        Zs = torch.full_like(X, 3.0)
        ops.spmm_rows(g, X, g.row_subset(rows), addend=add, Z=Zs, z_scale=0.5, x_nonzero=mask)
        assert torch.equal(Zs[rows], Zd[rows])


@pytest.mark.parametrize("K", [1, 2, 3])
@pytest.mark.parametrize("expand_all", [False, True])
def test_propagate_mean_rows_bit_identical(cuda_device, K, expand_all, monkeypatch):
    """Rows S of the layer mean and the full gradient dE0, receptive-field path vs full path: torch.equal.
    expand_all lifts the neighbour-set limit so that every layer (not only the last two) is restricted."""
    from spex_b200 import ops

    if expand_all:
        monkeypatch.setattr(ops, "EXPAND_MAX_EDGE_FRAC", 0.5)
        monkeypatch.setattr(ops, "SUBSET_MAX_EDGE_FRAC", 0.9)
    g, nur, m = _graph(cuda_device, seg_len=32)
    N, D = nur + m, 64
    torch.manual_seed(9)
    E_full = torch.randn(N, D, device=cuda_device, requires_grad=True)
    E_rows = E_full.detach().clone().requires_grad_(True)
    gen = torch.Generator().manual_seed(K)
    S = torch.cat([torch.randint(0, nur - 1, (24,), generator=gen),
                   nur + torch.randint(0, m, (72,), generator=gen), torch.tensor([nur + 2])]).to(cuda_device)
    R = ops.receptive_rows(g, torch.unique(S), K)
    assert R[K] is not None                      # the last layer is always restricted here
    if expand_all and K >= 2:
        assert R[1] is not None
    w = torch.randn(S.numel(), D, device=cuda_device)
    out_f = ops.propagate_mean(E_full, g, K)
    (out_f[S] * w).sum().backward()
    out_r = ops.propagate_mean(E_rows, g, K, rows_needed=S)
    assert torch.equal(out_r[S], out_f[S])
    # backward contract: gradient zero outside S (what the loss kernels produce)
    gdense = torch.zeros(N, D, device=cuda_device)
    gdense.index_add_(0, S, w)
    out_r.backward(gdense)
    assert torch.equal(E_rows.grad, E_full.grad)


@pytest.mark.parametrize("loss_kind", ["bce", "bpr", "bce_dropout"])
def test_model_training_step_same_bits_as_full_computer(cuda_device, loss_kind):
    """LightGCN.forward(flag=0) / bpr_loss in training mode with and without the receptive-field path: same loss
    bits, same gradient bits, persistent workspaces on (two steps: the zero tables are re-used), and the result
    still matches the oracle's autograd."""
    from spex_b200 import ops
    from spex_b200.dataloader import SyntheticDataset
    from spex_b200.model import LightGCN

    ds = SyntheticDataset(20000, 8000, 150000, seed=8)
    kw = dict(dropout=1, keepprob=0.7) if loss_kind == "bce_dropout" else {}
    torch.manual_seed(2020)
    model = LightGCN(make_args(**kw), ds).to(cuda_device)
    model.train()
    rng = np.random.default_rng(4)
    ops.enable_persistent_workspaces(True)
    try:
        for step in range(2):
            B = 48
            users = torch.from_numpy(rng.integers(0, ds.n_users, B)).to(cuda_device)
            a = torch.from_numpy(rng.integers(0, ds.m_items, B)).to(cuda_device)
            b = torch.from_numpy(rng.integers(0, ds.m_items, B)).to(cuda_device)
            labels = torch.from_numpy(rng.integers(0, 2, B)).to(cuda_device)
            res = {}
            for rf in (False, True):
                model.receptive_field = rf
                model.zero_grad(set_to_none=True)
                torch.manual_seed(100 + step)            # same dropout mask in both runs
                if loss_kind == "bpr":
                    l, r = model.bpr_loss(users, a, b)
                    loss = l + 1e-2 * r
                else:
                    loss = model(users, a, labels, flag=0)
                loss.backward()
                res[rf] = (loss.detach().clone(), model.embedding_user.weight.grad.clone(),
                           model.embedding_item.weight.grad.clone())
            assert torch.equal(res[True][0], res[False][0])
            assert torch.equal(res[True][1], res[False][1])
            assert torch.equal(res[True][2], res[False][2])
        if loss_kind == "bce":
            A = oracle_graph(ds.trainUser, ds.trainItem, ds.n_users + 1, ds.m_items)
            uw = model.embedding_user.weight.detach().cpu().clone().requires_grad_(True)
            iw = model.embedding_item.weight.detach().cpu().clone().requires_grad_(True)
            ref = O.bce_forward(uw, iw, A, 3, users.cpu(), a.cpu(), labels.cpu())
            ref.backward()
            assert abs(float(res[True][0]) - float(ref)) <= 1e-5 * abs(float(ref))
            assert rel_err(res[True][1], uw.grad) < 1e-5 and rel_err(res[True][2], iw.grad) < 1e-5
    finally:
        model.receptive_field = True
        ops.enable_persistent_workspaces(False)
