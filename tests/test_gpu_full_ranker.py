"""ops.FullRanker, the one host dispatcher of full ranking (item pack once, user blocks, scorer call), and the
callers that go through it: LightGCN.rank_topk and dist.ShardedEvaluator (here with no process group, world
size 1)."""
import numpy as np
import pytest
import torch


def _tables(dev, D, n_u=300, m=3000, seed=3):
    from spex_b200.graph import build_interaction_csr

    g = torch.Generator().manual_seed(seed)
    U = (torch.randn(n_u, D, generator=g) * 0.3).to(dev)
    I = (torch.randn(m, D, generator=g) * 0.3).to(dev)
    rng = np.random.default_rng(seed)
    rp, col = build_interaction_csr(rng.integers(0, n_u, 4000), rng.integers(0, m, 4000), n_u, m)
    return U, I, torch.from_numpy(rp).to(dev), torch.from_numpy(col).to(dev)


def _direct(ops, precision, U, I, users, k, rp, col):
    """The scorer calls as the callers made them before FullRanker: every user in one call."""
    m, D = I.shape
    if precision == "f16":
        Ih, m_pad, imeta = ops.pack_f16(I, None, ops.TC_ITEM_MULTIPLE)
        Uh, b_pad, umeta = ops.pack_f16(U, users, ops.TC_USER_MULTIPLE)
        return ops.score_topk_f16(Uh, umeta, users.numel(), b_pad, Ih, imeta, m, m_pad, D, k, users, rp, col)
    if precision == "bf16":
        Ib, m_pad = ops.pack_bf16(I, None, ops.TC_ITEM_MULTIPLE)
        Ub, b_pad = ops.pack_bf16(U, users, ops.TC_USER_MULTIPLE)
        return ops.score_topk_bf16(Ub, users.numel(), b_pad, Ib, m, m_pad, k, users, rp, col)
    return ops.score_topk_f32(U, I, users, k, rp, col)


def _same_bits(a, b):
    return a.shape == b.shape and torch.equal(a.view(torch.int32), b.view(torch.int32))


@pytest.mark.gpu
@pytest.mark.parametrize("precision,D", [("f16", 64), ("f16", 128), ("bf16", 64), ("fp32", 64), ("fp32", 40)])
def test_full_ranker_matches_direct_scorer_calls(cuda_device, precision, D):
    from spex_b200 import ops

    U, I, rp, col = _tables(cuda_device, D)
    users = torch.randperm(U.shape[0], generator=torch.Generator().manual_seed(1)).to(cuda_device)
    i_ref, v_ref = _direct(ops, precision, U, I, users, 20, rp, col)
    ranker = ops.FullRanker(I, precision)
    for block in (200, None):            # 200: two blocks, neither a multiple of 128 users
        idx, val = ranker.topk(U, users, 20, rp, col, user_block=block)
        torch.cuda.synchronize()
        assert _same_bits(idx, i_ref) and _same_bits(val, v_ref), (precision, D, block)
    # no mask, and an empty user list
    i0, v0 = _direct(ops, precision, U, I, users, 7, None, None)
    idx, val = ranker.topk(U, users, 7, user_block=128)
    assert _same_bits(idx, i0) and _same_bits(val, v0)
    idx, val = ranker.topk(U, users[:0], 7)
    assert idx.shape == (0, 7) and val.shape == (0, 7)


@pytest.mark.gpu
@pytest.mark.parametrize("precision", ["f16", "bf16", "fp32"])
def test_sharded_evaluator_on_one_gpu_matches_model(cuda_device, precision):
    from spex_b200 import batch_test
    from spex_b200.dist import ShardedEvaluator
    from spex_b200.graph import build_interaction_csr
    from test_gpu_parity import _small_model

    ds, model, _, _ = _small_model(cuda_device)
    model.eval()
    users = np.arange(ds.n_users)
    i_ref, v_ref = model.rank_topk(users, k=20, precision=precision)
    au, ai = model.computer()
    mrp, mcol = model.train_mask_csr()
    ev = ShardedEvaluator(au, ai, mrp, mcol, k=20, scorer=precision)
    assert ev.world == 1 and ev.scorer == precision          # random tables: the f16 probe keeps the filter
    users_d = torch.from_numpy(users).to(cuda_device)
    for block in (148 * 2 * 128 * 4, 96):
        idx, val, (lo, hi) = ev.rank_topk(users_d, block=block)
        assert (lo, hi) == (0, ds.n_users)
        assert _same_bits(idx, i_ref) and _same_bits(val, v_ref), block
    # Recall/NDCG@20: the evaluator's one-all-reduce sums against batch_test.test_fullrank
    truth = {int(u): list(ds.testRatings[u]) for u in users if u in ds.testRatings}
    tu = np.array([u for u in users for _ in truth.get(int(u), [])], np.int64)
    ti = np.array([i for u in users for i in truth.get(int(u), [])], np.int64)
    trp, tcol = build_interaction_csr(tu, ti, ds.n_users, ds.m_items)
    got = ev.recall_ndcg(users_d, trp, tcol)
    ref = batch_test.test_fullrank(model, users, truth, k=20, precision=precision)
    assert got["users"] == ds.n_users
    assert abs(got["recall"] - ref["recall"]) < 1e-12 and abs(got["ndcg"] - ref["ndcg"]) < 1e-12, (got, ref)


@pytest.mark.parametrize("precision,D,exc", [("f16", 32, RuntimeError), ("f16", 96, RuntimeError),
                                             ("bf16", 128, RuntimeError), ("fp16", 64, ValueError),
                                             ("int8", 64, ValueError)])
def test_full_ranker_rejects_precision_and_dim(precision, D, exc):
    """The precision is checked against D before anything is packed (no GPU needed)."""
    from spex_b200 import ops

    with pytest.raises(exc):
        ops.FullRanker(torch.zeros(16, D), precision)
