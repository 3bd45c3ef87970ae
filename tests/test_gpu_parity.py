"""GPU parity: the CUDA path (through the C-ABI, via spex_b200.ops / model) against the CPU oracle
on the same seeded inputs.  Tolerances: 1e-5 relative for fp32 propagation / losses / gradients
(north_star), exact index agreement modulo score ties for top-k, 1e-2 for bf16 scoring."""
import numpy as np
import pytest
import torch

from helpers import check_topk_against_scores, make_args, oracle_graph, random_graph, rel_err
from oracle import lightgcn_oracle as O

pytestmark = pytest.mark.gpu

TOL = 1e-5


def _dev_graph(u, i, nur, m, dev, seg_len=1024):
    from spex_b200 import ops
    from spex_b200.graph import build_norm_adj

    return ops.DeviceGraph.from_host(build_norm_adj(u, i, nur, m), dev, seg_len=seg_len)


@pytest.mark.parametrize("D", [64, 32, 128, 20, 256])
@pytest.mark.parametrize("seg_len", [1024, 32])
def test_spmm_matches_sparse_mm(cuda_device, D, seg_len):
    from spex_b200 import ops

    nu, m = 700, 400
    u, i = random_graph(nu, m, 9000, 11, hub_items=3, hub_degree=500)
    A = oracle_graph(u, i, nu + 1, m)
    g = _dev_graph(u, i, nu + 1, m, cuda_device, seg_len)
    if seg_len == 32:
        assert g.n_long > 0
    torch.manual_seed(0)
    X = torch.randn(nu + 1 + m, D)
    ref = torch.sparse.mm(A, X)
    Y = ops.spmm(g, X.to(cuda_device))
    assert rel_err(Y, ref) < TOL
    # empty rows (the padding user) stay exactly zero
    assert float(Y[nu].abs().max()) == 0.0
    # fused epilogue: Z = (addend*2 + A.X) * 0.25, Y written too
    add = torch.randn_like(X)
    Z = torch.empty_like(X, device=cuda_device)
    Y2 = torch.empty_like(Z)
    ops.spmm(g, X.to(cuda_device), Y=Y2, addend=add.to(cuda_device), addend_scale=2.0, Z=Z, z_scale=0.25)
    assert torch.equal(Y2, Y)
    assert rel_err(Z, (add * 2 + ref) * 0.25) < TOL


@pytest.mark.parametrize("D", [64, 32, 128])
def test_spmm_16_byte_aligned_table_takes_the_128_bit_kernels(cuda_device, D):
    """A table that is only 16-byte aligned (the ABI's minimum) cannot use the 256-bit gathers: the library falls
    back to the 128-bit kernels.  Same result as the 32-byte aligned table to fp32 rounding (the two kernels sum a
    row in different fixed orders), both within tolerance of torch.sparse.mm, and each bit-reproducible."""
    from spex_b200 import ops

    nu, m = 700, 400
    u, i = random_graph(nu, m, 9000, 11, hub_items=3, hub_degree=500)
    A = oracle_graph(u, i, nu + 1, m)
    g = _dev_graph(u, i, nu + 1, m, cuda_device, 32)
    N = nu + 1 + m
    torch.manual_seed(1)
    X = torch.randn(N, D)
    ref = torch.sparse.mm(A, X)
    big = torch.empty(N * D + 4, device=cuda_device)
    Xu = big[4:].view(N, D)
    Xu.copy_(X)
    assert Xu.data_ptr() % 32 == 16
    Xa = X.to(cuda_device)
    assert Xa.data_ptr() % 32 == 0
    Yu, Ya = ops.spmm(g, Xu), ops.spmm(g, Xa)
    assert rel_err(Yu, ref) < TOL and rel_err(Ya, ref) < TOL
    assert rel_err(Yu, Ya) < 1e-6
    assert torch.equal(ops.spmm(g, Xu), Yu) and torch.equal(ops.spmm(g, Xa), Ya)


@pytest.mark.parametrize("seg_len", [32, 256])
def test_spmm_column_blocked_long_rows(cuda_device, seg_len, monkeypatch):
    """Long rows cut at column-block boundaries and launched block-major (the L2-window path used
    on tables far larger than L2), forced here on a small graph."""
    from spex_b200 import ops

    monkeypatch.setattr(ops.DeviceGraph, "L2_WINDOW_BYTES", 16 * 1024)
    monkeypatch.setattr(ops.DeviceGraph, "MIN_CB_COLS", 48)
    monkeypatch.setattr(ops.DeviceGraph, "HUB_EDGES_PER_BLOCK", 10)   # hubs blocked, the rest fixed-length
    nu, m, D = 900, 500, 64
    u, i = random_graph(nu, m, 12000, 13, hub_items=4, hub_degree=700)
    A = oracle_graph(u, i, nu + 1, m)
    g = _dev_graph(u, i, nu + 1, m, cuda_device, seg_len)
    assert g.seg_start is not None and g.n_long > 0 and g.n_seg > g.n_long and g.n_hub > 0
    if seg_len == 32:
        assert g.n_hub < g.n_long   # mixed plan: blocked hubs + fixed-length mid rows
    # every edge of every long row is covered exactly once, segments never exceed seg_len
    cnt = g.seg_count.cpu().numpy()
    assert cnt.max() <= seg_len and cnt.min() >= 1
    deg = (g.rowptr[1:] - g.rowptr[:-1])[g.long_rows.long()].cpu().numpy()
    segptr = g.long_segptr.cpu().numpy()
    per_row = np.add.reduceat(cnt[g.row_seg.cpu().numpy()], segptr[:-1])
    assert np.array_equal(per_row, deg)
    torch.manual_seed(0)
    X = torch.randn(nu + 1 + m, D)
    ref = torch.sparse.mm(A, X)
    Y = ops.spmm(g, X.to(cuda_device))
    assert rel_err(Y, ref) < TOL
    assert torch.equal(Y, ops.spmm(g, X.to(cuda_device)))
    E = X * 0.1
    ru, ri = O.computer(E[: nu + 1], E[nu + 1:], A, 3)
    out = ops.propagate_mean(E.to(cuda_device), g, 3)
    assert rel_err(out, torch.cat([ru, ri])) < TOL


@pytest.mark.parametrize("seg_len", [32, 1024])
def test_hot_column_flags_give_bit_identical_results(cuda_device, seg_len):
    """Bit 31 of col flags hot table rows (L2 evict_last gathers): a cache hint only, so results
    are bit-identical to the unflagged graph."""
    from spex_b200 import ops

    nu, m, D = 900, 500, 64
    u, i = random_graph(nu, m, 12000, 17, hub_items=4, hub_degree=700)
    g0 = _dev_graph(u, i, nu + 1, m, cuda_device, seg_len)
    g1 = _dev_graph(u, i, nu + 1, m, cuda_device, seg_len)
    n_hot = g1.mark_hot_columns(D, budget_bytes=16 * 1024)
    assert 0 < n_hot <= 2 * (16 * 1024 // 256) and g1.col_hot
    assert (g1.col < 0).any() and torch.equal(g1.clean_col(), g0.col)
    torch.manual_seed(0)
    X = torch.randn(nu + 1 + m, D, device=cuda_device)
    assert torch.equal(ops.spmm(g1, X), ops.spmm(g0, X))
    E = X * 0.1
    assert torch.equal(ops.propagate_mean(E, g1, 3), ops.propagate_mean(E, g0, 3))
    A = g1.to_sparse_coo()
    assert int(A.indices()[1].max()) < nu + 1 + m


def test_spmm_rejects_a_plan_without_segment_list_or_with_unknown_flags(cuda_device):
    """spex_long_plan has one segment list and one flag bit (SPEX_PLAN_COL_HOTBIT): a plan with long rows but no
    seg_start / seg_count / row_seg, or with any other flag bit set, is refused with SPEX_E_BADARG before a launch."""
    import ctypes

    from spex_b200 import _capi, ops

    nu, m, D = 700, 400, 64
    u, i = random_graph(nu, m, 9000, 11, hub_items=3, hub_degree=500)
    g = _dev_graph(u, i, nu + 1, m, cuda_device, 32)
    assert g.n_long > 0
    X = torch.randn(g.n_cols, D, device=cuda_device)
    Y = torch.empty(g.n_rows, D, device=cuda_device)
    g.plan(D)

    def run(plan):
        rc = _capi.lib.spex_spmm_csr_f32(_capi.ptr(g.rowptr), _capi.ptr(g.col), _capi.ptr(g.val), _capi.ptr(X),
                                         g.n_rows, D, _capi.ptr(Y), None, 1.0, None, 1.0, ctypes.byref(plan),
                                         _capi.stream_ptr())
        torch.cuda.synchronize()
        return rc

    assert run(_capi.LongPlan.from_buffer_copy(g._plan_struct)) == 0
    for flag in (2, 4, 1 << 30):
        bad = _capi.LongPlan.from_buffer_copy(g._plan_struct)
        bad.flags |= flag
        assert run(bad) == -1, flag                      # SPEX_E_BADARG
    for field in ("seg_start", "seg_count", "row_seg"):
        bad = _capi.LongPlan.from_buffer_copy(g._plan_struct)
        setattr(bad, field, None)
        assert run(bad) == -1, field


@pytest.mark.parametrize("K", [0, 1, 2, 3, 4])
def test_propagate_mean_and_determinism(cuda_device, K):
    from spex_b200 import ops

    nu, m, D = 500, 300, 64
    u, i = random_graph(nu, m, 7000, 5, hub_items=2, hub_degree=400)
    A = oracle_graph(u, i, nu + 1, m)
    g = _dev_graph(u, i, nu + 1, m, cuda_device, seg_len=64)
    torch.manual_seed(1)
    E = torch.randn(nu + 1 + m, D) * 0.1
    ru, ri = O.computer(E[: nu + 1], E[nu + 1:], A, K)
    out = ops.propagate_mean(E.to(cuda_device), g, K)
    assert rel_err(out, torch.cat([ru, ri])) < TOL
    out2 = ops.propagate_mean(E.to(cuda_device), g, K)
    assert torch.equal(out, out2), "propagation must be bit-reproducible (no atomics)"


@pytest.mark.parametrize("dropout", [False, True])
def test_propagate_backward(cuda_device, dropout):
    from spex_b200 import ops

    nu, m, D, K = 300, 200, 64, 3
    u, i = random_graph(nu, m, 4000, 9)
    A = oracle_graph(u, i, nu + 1, m)
    g = _dev_graph(u, i, nu + 1, m, cuda_device)
    torch.manual_seed(2)
    E = (torch.randn(nu + 1 + m, D) * 0.1).requires_grad_(True)
    W = torch.randn(nu + 1 + m, D)
    val = valT = None
    Aref = A
    if dropout:
        rand = torch.rand(A._nnz())
        Aref = O.dropout_graph(A, 0.6, rand)
        keep = (rand + 0.6).int().bool()
        val = g.dropout_values(keep, 0.6)
        valT = g.transposed_values(val)
    ru, ri = O.computer(E[: nu + 1], E[nu + 1:], Aref, K)
    (torch.cat([ru, ri]) * W).sum().backward()
    Ed = E.detach().to(cuda_device).requires_grad_(True)
    out = ops.propagate_mean(Ed, g, K, val, valT)
    assert rel_err(out, torch.cat([ru, ri])) < TOL
    (out * W.to(cuda_device)).sum().backward()
    assert rel_err(Ed.grad, E.grad) < TOL


def _small_model(cuda_device, **kw):
    from spex_b200.dataloader import SyntheticDataset
    from spex_b200.model import LightGCN

    ds = SyntheticDataset(400, 250, 6000, seed=4)
    torch.manual_seed(2020)
    model = LightGCN(make_args(**kw), ds)
    ref_w = (model.embedding_user.weight.detach().clone(), model.embedding_item.weight.detach().clone())
    A = oracle_graph(ds.trainUser, ds.trainItem, ds.n_users + 1, ds.m_items)
    return ds, model.to(cuda_device), ref_w, A


def test_model_forward_backward_bce(cuda_device):
    ds, model, (uw, iw), A = _small_model(cuda_device)
    rng = np.random.default_rng(0)
    B = 256
    users = torch.from_numpy(rng.integers(0, ds.n_users, B))
    users[:40] = users[0]  # heavy duplicates: exercises the segmented scatter
    items = torch.from_numpy(rng.integers(0, ds.m_items, B))
    items[100:130] = items[100]
    labels = torch.from_numpy(rng.integers(0, 2, B))
    uw.requires_grad_(True)
    iw.requires_grad_(True)
    ref = O.bce_forward(uw, iw, A, 3, users, items, labels)
    ref.backward()
    model.train()
    loss = model(users.to(cuda_device), items.to(cuda_device), labels.to(cuda_device), flag=0)
    loss.backward()
    assert abs(float(loss) - float(ref)) <= TOL * abs(float(ref))
    assert rel_err(model.embedding_user.weight.grad, uw.grad) < TOL
    assert rel_err(model.embedding_item.weight.grad, iw.grad) < TOL
    # flag=1 returns the logits
    model.eval()
    with torch.no_grad():
        g1 = model(users.to(cuda_device), items.to(cuda_device), None, flag=1)
        ru, ri = O.computer(uw.detach(), iw.detach(), A, 3)
    assert rel_err(g1, O.gamma(ru, ri, users, items)) < TOL


def test_model_dropout_matches_reference_mask(cuda_device):
    ds, model, (uw, iw), A = _small_model(cuda_device, dropout=1, keepprob=0.3)
    users = torch.arange(64) % ds.n_users
    items = torch.arange(64) % ds.m_items
    labels = (torch.arange(64) % 2)
    torch.manual_seed(77)
    Adrop = O.dropout_graph(A, 0.3)
    uw.requires_grad_(True)
    iw.requires_grad_(True)
    ru, ri = O.computer(uw, iw, Adrop, 3)
    ref = torch.nn.BCEWithLogitsLoss()(O.gamma(ru, ri, users, items), labels.float())
    ref.backward()
    model.train()
    torch.manual_seed(77)
    loss = model(users.to(cuda_device), items.to(cuda_device), labels.to(cuda_device), flag=0)
    loss.backward()
    assert abs(float(loss) - float(ref)) <= TOL * abs(float(ref))
    assert rel_err(model.embedding_user.weight.grad, uw.grad) < TOL
    assert rel_err(model.embedding_item.weight.grad, iw.grad) < TOL


def test_model_bpr_loss(cuda_device):
    ds, model, (uw, iw), A = _small_model(cuda_device)
    rng = np.random.default_rng(1)
    B = 512
    users = torch.from_numpy(rng.integers(0, ds.n_users, B))
    pos = torch.from_numpy(rng.integers(0, ds.m_items, B))
    neg = torch.from_numpy(rng.integers(0, ds.m_items, B))
    uw.requires_grad_(True)
    iw.requires_grad_(True)
    rl, rr = O.bpr_loss(uw, iw, A, 3, users, pos, neg)
    (rl + 1e-2 * rr).backward()
    model.train()
    l, r = model.bpr_loss(users.to(cuda_device), pos.to(cuda_device), neg.to(cuda_device))
    (l + 1e-2 * r).backward()
    assert abs(float(l) - float(rl)) <= TOL * abs(float(rl))
    assert abs(float(r) - float(rr)) <= TOL * abs(float(rr))
    assert rel_err(model.embedding_user.weight.grad, uw.grad) < TOL
    assert rel_err(model.embedding_item.weight.grad, iw.grad) < TOL


def test_adam_matches_torch(cuda_device):
    from spex_b200 import ops

    torch.manual_seed(3)
    n = 64 * 1001 + 3
    p0 = torch.randn(n)
    p_ref = p0.clone().requires_grad_(True)
    opt = torch.optim.Adam([p_ref], lr=1e-3)
    p = p0.to(cuda_device)
    m = torch.zeros_like(p)
    v = torch.zeros_like(p)
    for step in range(1, 4):
        g = torch.randn(n)
        p_ref.grad = g.clone()
        opt.step()
        ops.adam_step(p, g.to(cuda_device), m, v, 1e-3, 0.9, 0.999, 1e-8, step)
    assert rel_err(p, p_ref) < 1e-6


def test_sampled_test_matches_reference_semantics(cuda_device):
    from spex_b200 import batch_test

    ds, model, (uw, iw), A = _small_model(cuda_device)
    model.eval()
    got = batch_test.test(model, ds.testRatings, ds.testNegatives)
    ru, ri = O.computer(uw, iw, A, 3)
    want = O.test_sampled(ru, ri, ds.testRatings, ds.testNegatives)
    # scores agree to 1e-5; rankings can differ only at near-ties, so allow a few users to move
    n = len(ds.testRatings)
    assert np.abs(got["recall"] - want["recall"]).max() <= 3.0 / n
    assert np.abs(got["ndcg"] - want["ndcg"]).max() <= 3.0 / n


def test_rating_and_topk_fp32(cuda_device):
    ds, model, (uw, iw), A = _small_model(cuda_device)
    model.eval()
    ru, ri = O.computer(uw, iw, A, 3)
    users = np.arange(0, ds.n_users, 3)
    rating = model.getUsersRating(torch.from_numpy(users).to(cuda_device))
    ref = O.users_rating(ru, ri, torch.from_numpy(users))
    assert rel_err(rating, ref) < TOL
    rp, col = ds.getInteractionCSR()
    masked = [col[rp[u]: rp[u + 1]] for u in users]
    scores = torch.matmul(ru[users].double(), ri.double().t()).numpy()
    for k in (1, 20, 128):
        idx, val = model.rank_topk(users, k=k, precision="fp32")
        check_topk_against_scores(idx, val, scores, k, masked, atol=1e-6)
    # determinism + tie-break by ascending id on exact ties (duplicate item rows)
    from spex_b200 import ops

    I2 = torch.cat([ri[:50], ri[:50]]).to(cuda_device)
    idx, val = ops.score_topk_f32(ru.to(cuda_device), I2, torch.arange(10), 100)
    idx = idx.cpu().numpy()
    for r in range(10):
        pairs = idx[r].reshape(50, 2)
        assert (pairs[:, 1] == pairs[:, 0] + 50).all()


def test_topk_bf16_tensor_core(cuda_device):
    from spex_b200 import ops

    torch.manual_seed(5)
    n_u, m, D = 300, 5000, 64
    U = (torch.randn(n_u, D) * 0.3).bfloat16().float()
    I = (torch.randn(m, D) * 0.3).bfloat16().float()
    users = torch.arange(n_u)
    rng = np.random.default_rng(2)
    mu = rng.integers(0, n_u, 6000)
    mi = rng.integers(0, m, 6000)
    from spex_b200.graph import build_interaction_csr

    rp, col = build_interaction_csr(mu, mi, n_u, m)
    masked = [col[rp[u]: rp[u + 1]] for u in range(n_u)]
    scores = torch.matmul(U.double(), I.double().t()).numpy()
    Ud, Id = U.to(cuda_device), I.to(cuda_device)
    Ib, m_pad = ops.pack_bf16(Id, None, ops.TC_ITEM_MULTIPLE)
    Ub, b_pad = ops.pack_bf16(Ud, users.to(cuda_device), ops.TC_USER_MULTIPLE)
    rpd = torch.from_numpy(rp).to(cuda_device)
    cold = torch.from_numpy(col).to(cuda_device)
    for k in (1, 20, 50, ops.TC_MAX_K):
        idx, val = ops.score_topk_bf16(Ub, n_u, b_pad, Ib, m, m_pad, k, users.to(cuda_device), rpd, cold)
        torch.cuda.synchronize()
        # inputs are exactly representable in bf16, so only the accumulation order differs
        check_topk_against_scores(idx, val, scores, k, masked, atol=1e-4)
    # agreement with the exact fp32 scorer on the same inputs (identical modulo near-ties)
    i32, v32 = ops.score_topk_f32(Ud, Id, users, 20, rpd, cold)
    i16, v16 = ops.score_topk_bf16(Ub, n_u, b_pad, Ib, m, m_pad, 20, users.to(cuda_device), rpd, cold)
    assert float((v32 - v16).abs().max()) < 1e-4
    assert float((i32 == i16).float().mean()) > 0.99


def test_topk_bf16_ties_and_duplicates(cuda_device):
    """Exact score ties (duplicated and all-zero item rows, spread over both column halves of the
    256-item stages) are broken by ascending item id, exactly like the fp32 scorer."""
    from spex_b200 import ops

    torch.manual_seed(11)
    n_u, m, D = 130, 3000, 64
    U = (torch.randn(n_u, D) * 0.3).bfloat16().float()
    base = (torch.randn(40, D) * 0.3).bfloat16().float()
    I = base[torch.randint(0, 40, (m,))].clone()      # every item row is one of 40 vectors
    I[::7] = 0.0                                       # and every 7th is all-zero (score 0)
    Ud, Id = U.to(cuda_device), I.to(cuda_device)
    users = torch.arange(n_u, device=cuda_device)
    Ib, m_pad = ops.pack_bf16(Id, None, ops.TC_ITEM_MULTIPLE)
    Ub, b_pad = ops.pack_bf16(Ud, users, ops.TC_USER_MULTIPLE)
    scores = torch.matmul(U.double(), I.double().t())
    for k in (5, 20, 50):
        i16, v16 = ops.score_topk_bf16(Ub, n_u, b_pad, Ib, m, m_pad, k, users, None, None)
        # reference order: score descending, then item id ascending (stable sort on -score)
        order = torch.sort(-scores, dim=1, stable=True).indices[:, :k]
        ref_v = torch.gather(scores, 1, order)
        got_v = torch.gather(scores, 1, i16.cpu().long())
        assert torch.allclose(got_v, ref_v, atol=1e-5), k            # same score multiset per rank
        tie_free = (ref_v[:, :-1] - ref_v[:, 1:]).abs() > 1e-4
        # within a run of equal scores the ids must ascend
        ids = i16.cpu().long()
        assert bool(((ids[:, 1:] > ids[:, :-1]) | tie_free).all()), k
        # the lowest ids of a tied group win: identical to the stable order on every row whose
        # top-(k+1) scores are either exactly tied (identical item rows) or clearly apart
        top = -torch.sort(-scores, dim=1, stable=True).values[:, : k + 1]
        gap = top[:, :-1] - top[:, 1:]
        clean = ~((gap > 1e-9) & (gap < 1e-4)).any(dim=1)
        assert int(clean.sum()) > n_u // 2
        assert torch.equal(ids[clean], order[clean]), k


def test_model_rank_topk_bf16_vs_fp32(cuda_device):
    ds, model, (uw, iw), A = _small_model(cuda_device)
    model.eval()
    users = np.arange(ds.n_users)
    i32, v32 = model.rank_topk(users, k=20, precision="fp32")
    i16, v16 = model.rank_topk(users, k=20, precision="bf16")
    # bf16 scoring: 1e-2 relative on scores (north_star); sets mostly agree
    scale = float(v32.abs().max())
    assert float((v32 - v16).abs().max()) <= 1e-2 * scale
    same = [(len(set(a.tolist()) & set(b.tolist())) / 20.0) for a, b in zip(i32.cpu().numpy(), i16.cpu().numpy())]
    assert np.mean(same) > 0.9


def test_expert_gate_and_ngcf_epilogue(cuda_device):
    from spex_b200 import ops

    torch.manual_seed(6)
    n, D = 1000, 64
    e0, e1 = torch.randn(n, D), torch.randn(n, D)
    W = torch.randn(2 * D, 2) * 0.1
    ref = O.expert_gate(e0, e1, W)
    got = ops.expert_gate(e0.to(cuda_device), e1.to(cuda_device), W.to(cuda_device))
    assert rel_err(got, ref) < TOL
    nu, m = 300, 200
    u, i = random_graph(nu, m, 4000, 9)
    A = oracle_graph(u, i, nu + 1, m)
    g = _dev_graph(u, i, nu + 1, m, cuda_device)
    ego = torch.randn(nu + 1 + m, D) * 0.1
    W1, W2 = torch.randn(D, D) * 0.1, torch.randn(D, D) * 0.1
    b1, b2 = torch.randn(D) * 0.1, torch.randn(D) * 0.1
    r_out, r_norm = O.ngcf_layer(A, ego, W1, b1, W2, b2, 0.2)
    side = ops.spmm(g, ego.to(cuda_device))
    norm = torch.empty(nu + 1 + m, 128, device=cuda_device)
    out = ops.ngcf_epilogue(ego.to(cuda_device), side, W1.to(cuda_device), b1.to(cuda_device),
                            W2.to(cuda_device), b2.to(cuda_device), 0.2, norm=norm[:, 64:], norm_stride=128)
    assert rel_err(out, r_out) < TOL
    assert rel_err(norm[:, 64:], r_norm) < 1e-5


def test_cpu_tensor_is_rejected():
    from spex_b200 import ops

    with pytest.raises(RuntimeError):
        ops.rating_dense(torch.zeros(4, 64), torch.zeros(4, 64), torch.zeros(1, dtype=torch.long))


@pytest.mark.parametrize("loss", ["bce", "bpr"])
def test_large_batch_sorted_scatter_matches_scan_and_oracle(cuda_device, loss, monkeypatch):
    """Batches beyond 2048 entries take the sorted segmented scatter (stable radix sort of (row, position)
    + one warp per run): gradients bit-identical to the duplicate-scan form and <= 1e-5 from the oracle;
    with the persistent workspaces the dense gradient table is zero-filled once and only the touched
    rows are cleared between steps."""
    from spex_b200 import ops

    ds, model, (uw, iw), A = _small_model(cuda_device)
    rng = np.random.default_rng(7)
    B = 6000                                            # 400 users x 250 items: heavy duplicates
    users = torch.from_numpy(rng.integers(0, ds.n_users, B))
    pos = torch.from_numpy(rng.integers(0, ds.m_items, B))
    neg = torch.from_numpy(rng.integers(0, ds.m_items, B))
    labels = torch.from_numpy(rng.integers(0, 2, B))
    uw.requires_grad_(True)
    iw.requires_grad_(True)
    if loss == "bce":
        ref = O.bce_forward(uw, iw, A, 3, users, pos, labels)
        ref.backward()
    else:
        rl, rr = O.bpr_loss(uw, iw, A, 3, users, pos, neg)
        (rl + 1e-2 * rr).backward()

    def run():
        model.zero_grad(set_to_none=True)
        model.train()
        if loss == "bce":
            l = model(users.to(cuda_device), pos.to(cuda_device), labels.to(cuda_device), flag=0)
            l.backward()
        else:
            l, r = model.bpr_loss(users.to(cuda_device), pos.to(cuda_device), neg.to(cuda_device))
            (l + 1e-2 * r).backward()
        return (model.embedding_user.weight.grad.detach().clone(), model.embedding_item.weight.grad.detach().clone())

    gu_sorted, gi_sorted = run()
    assert rel_err(gu_sorted, uw.grad) < TOL and rel_err(gi_sorted, iw.grad) < TOL
    # the scan form (no workspace) must give the same bits
    monkeypatch.setattr(ops, "_scatter_workspace", lambda total, device: (None, 0))
    gu_scan, gi_scan = run()
    monkeypatch.undo()
    assert torch.equal(gu_sorted, gu_scan) and torch.equal(gi_sorted, gi_scan)
    # persistent workspaces: three steps in a row give the same gradients (rows are cleared in between)
    ops.enable_persistent_workspaces(True)
    try:
        for _ in range(3):
            gu_p, gi_p = run()
            assert torch.equal(gu_p, gu_sorted) and torch.equal(gi_p, gi_sorted)
        # a different (small, scan-form) batch in between must not leave stale rows behind
        small = slice(0, 300)
        users_b, pos_b, neg_b, labels_b = users, pos, neg, labels
        users, pos, neg, labels = users[small], pos[small], neg[small], labels[small]
        run()
        users, pos, neg, labels = users_b, pos_b, neg_b, labels_b
        gu_p, gi_p = run()
        assert torch.equal(gu_p, gu_sorted) and torch.equal(gi_p, gi_sorted)
    finally:
        ops.enable_persistent_workspaces(False)
