"""Full-ranking rank of held-out pairs (spex_rank_pairs_f16 / spex_rank_pairs_f32, FullRanker.ranks) and the metrics
built on it (FullRanker.rank_metrics), against exact float64 ranks, the top-k lists and FullRanker.evaluate.

The rank of pair (u, t) is the number of items outside u's mask, other than t, that come before t under (score
descending, id ascending).  Dyadic small-integer tables make every score exact in every precision, so there the
ranks must equal the float64 ranks exactly, ties by id included; random tables are checked against a float64
bracket wide enough for operand rounding.
"""
import numpy as np
import pytest
import torch

from test_epinion2_golden import ep2_root  # noqa: F401  (module fixture: the epinion2 dataset on disk)
from test_gpu_ranking_edges import _dyadic, _mask_csr

pytestmark = pytest.mark.gpu

CASES = [("f16", 64), ("f16", 128), ("fp32", 64), ("fp32", 48)]


def _masks(rng, n_users, m):
    """A few masked items per user; every fourth user has an empty row."""
    return {u: [] if u % 4 == 0 else list(rng.integers(0, m, rng.integers(1, 8))) for u in range(n_users)}


def _device_mask(masks, n_users, dev):
    rp, col = _mask_csr(masks, n_users)
    return torch.from_numpy(rp).to(dev), torch.from_numpy(col).to(dev)


def _exact_ranks(S, users, items, masks):
    """float64 ranks: items outside the mask, other than t, with (score, -id) above (s_t, -t)."""
    out = np.empty(len(users), np.int64)
    ids = np.arange(S.shape[1])
    for p, (u, t) in enumerate(zip(users, items)):
        s = S[u]
        above = (s > s[t]) | ((s == s[t]) & (ids < t))
        above[t] = False
        above[list(masks.get(int(u), []))] = False
        out[p] = int(above.sum())
    return out


def _ranker(I, precision, dev, probe=False):
    from spex_b200 import ops

    return ops.FullRanker(I.to(dev), precision, probe=probe)


@pytest.mark.parametrize("precision,D", CASES)
@pytest.mark.parametrize("P", [1, 127, 129, 901])
@pytest.mark.parametrize("m", [1, 127, 128, 129, 3000])
def test_ranks_exact_on_dyadic_tables(cuda_device, precision, D, P, m):
    """Exact ties everywhere (small integers), masks with empty rows, held-out items that are masked, users that
    repeat, and - for m not a multiple of 128 - the zero-padded last tile, whose columns score 0."""
    gen = torch.Generator().manual_seed(P * 7 + m)
    rng = np.random.default_rng(P + m)
    n_users = 300
    U, I = _dyadic(gen, n_users, D, -2), _dyadic(gen, m, D, -3)
    masks = _masks(rng, n_users, m)
    users = rng.integers(0, n_users, P)
    items = rng.integers(0, m, P)
    rp, col = _device_mask(masks, n_users, cuda_device)
    got = _ranker(I, precision, cuda_device).ranks(U.to(cuda_device), torch.from_numpy(users),
                                                   torch.from_numpy(items), rp, col)
    S = U.double().numpy() @ I.double().numpy().T
    assert got.dtype == torch.int32 and got.shape == (P,)
    np.testing.assert_array_equal(got.cpu().numpy(), _exact_ranks(S, users, items, masks))


@pytest.mark.parametrize("precision,D", CASES)
@pytest.mark.parametrize("P,m", [(1, 1), (127, 129), (129, 127), (901, 3000), (129, 128)])
def test_ranks_in_float64_bracket(cuda_device, precision, D, P, m):
    """Random tables: each rank lies in [#items above s_t + delta, #items at or above s_t - delta] (unmasked, t
    excluded), delta covering the rounding of the operands to fp16 (or of the fp32 sums)."""
    rng = np.random.default_rng(3 * P + m)
    n_users = 200
    U = rng.standard_normal((n_users, D)).astype(np.float32)
    I = rng.standard_normal((m, D)).astype(np.float32)
    masks = _masks(rng, n_users, m)
    users = rng.integers(0, n_users, P)
    items = rng.integers(0, m, P)
    rp, col = _device_mask(masks, n_users, cuda_device)
    got = _ranker(torch.from_numpy(I), precision, cuda_device).ranks(
        torch.from_numpy(U).to(cuda_device), torch.from_numpy(users), torch.from_numpy(items), rp, col).cpu().numpy()
    S = U.astype(np.float64) @ I.astype(np.float64).T
    rel = 2.0 ** -9 if precision == "f16" else D * 2.0 ** -22
    for p, (u, t) in enumerate(zip(users, items)):
        delta = rel * np.linalg.norm(U[u]) * np.linalg.norm(I, axis=1).max() + 1e-30
        ok = np.ones(m, bool)
        ok[t] = False
        ok[list(masks.get(int(u), []))] = False
        lo = int(((S[u] > S[u, t] + delta) & ok).sum())
        hi = int(((S[u] >= S[u, t] - delta) & ok).sum())
        assert lo <= got[p] <= hi, (p, lo, got[p], hi)


@pytest.mark.parametrize("precision,D,k", [("f16", 64, 512), ("f16", 128, 512), ("fp32", 64, 128), ("fp32", 48, 128)])
def test_ranks_are_topk_positions(cuda_device, precision, D, k):
    """A pair whose item is in topk(k) has rank == its position; every other unmasked item has rank >= k."""
    rng = np.random.default_rng(D + k)
    n_users, m = 300, 3000
    U = torch.from_numpy(rng.standard_normal((n_users, D)).astype(np.float32)).to(cuda_device)
    I = torch.from_numpy(rng.standard_normal((m, D)).astype(np.float32))
    masks = _masks(rng, n_users, m)
    rp, col = _device_mask(masks, n_users, cuda_device)
    r = _ranker(I, precision, cuda_device)
    users = torch.arange(n_users)
    idx, _ = r.topk(U, users, k, rp, col)
    idx = idx.cpu().numpy()
    pu = np.repeat(np.arange(n_users), 6)
    pt = rng.integers(0, m, pu.size)
    pt[0::6] = idx[:, 0]
    pt[1::6] = idx[:, k // 2]
    pt[2::6] = idx[:, k - 1]
    got = r.ranks(U, torch.from_numpy(pu), torch.from_numpy(pt), rp, col).cpu().numpy()
    for p, (u, t) in enumerate(zip(pu, pt)):
        pos = np.flatnonzero(idx[u] == t)
        if pos.size:
            assert got[p] == pos[0], (p, u, t)
        elif t not in masks.get(int(u), []):
            assert got[p] >= k, (p, u, t)


@pytest.mark.parametrize("precision,D", CASES)
def test_edges(cuda_device, precision, D):
    """Duplicated item rows (exact ties broken by id); a held-out item with a negative score and m = 130 (the
    padded columns of the last tile score 0 and must not count); a masked held-out item; a mask with items above
    and below t."""
    gen = torch.Generator().manual_seed(5)
    m = 130
    I = _dyadic(gen, m, D, -3)
    I[10:20] = I[50]                                         # eleven identical rows
    U = _dyadic(gen, 4, D, -2)
    U[3] = -U[3]
    S = U.double().numpy() @ I.double().numpy().T
    t_neg = int(np.argsort(S[3])[5])                         # a low (negative) score
    assert S[3, t_neg] < 0
    order = np.argsort(-S[2], kind="stable")
    t_mid = int(order[60])
    masks = {0: [], 1: [15, 16, 50, 129], 2: [int(order[3]), int(order[100]), t_mid], 3: list(range(0, 128, 9))}
    users = np.array([0, 0, 0, 1, 1, 2, 2, 3, 3])
    items = np.array([15, 50, 19, 15, 17, t_mid, int(order[61]), t_neg, 129])
    rp, col = _device_mask(masks, 4, cuda_device)
    got = _ranker(I, precision, cuda_device).ranks(U.to(cuda_device), torch.from_numpy(users),
                                                   torch.from_numpy(items), rp, col).cpu().numpy()
    np.testing.assert_array_equal(got, _exact_ranks(S, users, items, masks))


@pytest.mark.parametrize("D", [64, 128])
def test_band_items_inside_the_filter_margin(cuda_device, D):
    """The adversarial items of test_gpu_ranking_edges.py (exact score just above the decoys', fp16 filter value
    below it) and the decoys themselves: every one falls inside the band around a decoy's score, so the ranks
    come from the exact re-score."""
    u = np.full(D, 2.0 ** -6)
    u[:16] = 1.0
    adv = np.full(D, 15 * 2.0 ** -9)
    adv[:16] = 1.0
    adv[14] = 1.0 + 7 * 2.0 ** -10
    s_adv = float(u @ adv)
    q = int(np.ceil((s_adv - 16.0) * 1024)) - 1
    dec = np.zeros(D)
    dec[:16] = 1.0 + (q // 16) * 2.0 ** -10
    dec[: q % 16] += 2.0 ** -10
    m, n_dec, n_adv = 128 * 8 + 37, 200, 50
    I = np.zeros((m, D))
    I[:, :16] = -1.0
    I[:n_dec] = dec
    adv_ids = 400 + 12 * np.arange(n_adv)
    I[adv_ids] = adv
    U = np.tile(u, (3, 1)) * np.array([1.0, 0.5, 0.25])[:, None]
    users = np.array([0, 0, 1, 1, 2, 2, 0])
    items = np.array([0, 199, 57, int(adv_ids[0]), int(adv_ids[49]), 1000, 1036])
    got = _ranker(torch.from_numpy(I).float(), "f16", cuda_device).ranks(
        torch.from_numpy(U).float().to(cuda_device), torch.from_numpy(users), torch.from_numpy(items)).cpu().numpy()
    np.testing.assert_array_equal(got, _exact_ranks(U @ I.T, users, items, {}))
    assert got[0] == n_adv and got[1] == n_adv + 199 and got[3] == 0


def _truth(rng, n_users, m, multi):
    """{position: sorted held-out items}: one per user, or 0-5 with empty rows."""
    rows = {}
    for b in range(n_users):
        n = 1 if not multi else int(rng.integers(0, 6))
        rows[b] = sorted(set(rng.integers(0, m, n).tolist()))
    rp = np.zeros(n_users + 1, np.int64)
    rp[1:] = np.cumsum([len(rows[b]) for b in range(n_users)])
    col = np.array([i for b in range(n_users) for i in rows[b]], np.int32)
    return rows, rp, col


@pytest.mark.parametrize("precision,D,kmax", [("f16", 64, 512), ("f16", 128, 512), ("fp32", 64, 128),
                                              ("fp32", 48, 128)])
@pytest.mark.parametrize("multi", [False, True])
def test_rank_metrics_equal_evaluate(cuda_device, precision, D, kmax, multi):
    rng = np.random.default_rng(D + kmax + multi)
    n_users, m = 1500, 4000
    U = torch.from_numpy(rng.standard_normal((n_users, D)).astype(np.float32)).to(cuda_device)
    I = torch.from_numpy(rng.standard_normal((m, D)).astype(np.float32))
    masks = _masks(rng, n_users, m)
    rp, col = _device_mask(masks, n_users, cuda_device)
    users = torch.from_numpy(rng.permutation(n_users))
    _, trp, tcol = _truth(rng, n_users, m, multi)
    r = _ranker(I, precision, cuda_device)
    cut = [1, 10, 20, 50, kmax]
    ev = r.evaluate(U, users, cut, trp, tcol, rp, col)
    rm = r.rank_metrics(U, users, cut, trp, tcol, rp, col)
    for key in ("recall", "precision", "hit"):
        np.testing.assert_array_equal(rm[key], ev[key], err_msg=key)
    np.testing.assert_allclose(rm["ndcg"], ev["ndcg"], rtol=0, atol=1e-12)
    assert rm["users"] == n_users


def _np_metrics(ranks, trp, tcol, users, masks, m, cutoffs):
    """Host formula of rank_metrics from float64 ranks."""
    disc = 1.0 / np.log2(np.arange(2, max(cutoffs) + 2))
    idcg = np.concatenate([[0.0], np.cumsum(disc)])
    B = len(trp) - 1
    rec, prec, ndcg, hit = (np.zeros(len(cutoffs)) for _ in range(4))
    mrr = auc = 0.0
    for b in range(B):
        T = tcol[trp[b]: trp[b + 1]]
        R = ranks[trp[b]: trp[b + 1]]
        M = set(int(x) for x in masks.get(int(users[b]), []))
        live = np.array([int(t) not in M for t in T], bool)
        lr = np.sort(R[live])
        for c, K in enumerate(cutoffs):
            h = lr[lr < K]
            if T.size:
                rec[c] += h.size / T.size
                ndcg[c] += (disc[h].sum() / idcg[min(T.size, K)]) if h.size else 0.0
            prec[c] += h.size / K
            hit[c] += h.size > 0
        if lr.size:
            mrr += 1.0 / (1.0 + lr[0])
        n_neg = m - len(M) - live.sum()
        if T.size:
            a = [(1.0 - (r - (lr < r).sum()) / n_neg if n_neg > 0 else 1.0) if lv else 0.0 for r, lv in zip(R, live)]
            auc += np.mean(a)
    return {"recall": rec / B, "precision": prec / B, "ndcg": ndcg / B, "hit": hit / B, "mrr": mrr / B,
            "auc": auc / B}


@pytest.mark.parametrize("precision,D", CASES)
def test_mrr_auc_and_large_cutoffs_match_numpy(cuda_device, precision, D):
    """Dyadic tables (ranks exact in every precision), multi-item truth with empty and masked entries, cutoffs up
    to 1000 and m: every metric equals the float64 host formula."""
    gen = torch.Generator().manual_seed(D)
    rng = np.random.default_rng(D + 1)
    n_users, m = 400, 3000
    U, I = _dyadic(gen, n_users, D, -2), _dyadic(gen, m, D, -3)
    masks = _masks(rng, n_users, m)
    users = rng.permutation(n_users)
    rows, trp, tcol = _truth(rng, n_users, m, True)
    for b in range(0, n_users, 7):                            # some held-out items are masked
        if rows[b]:
            masks[int(users[b])] = sorted(set(masks[int(users[b])]) | {rows[b][0]})
    rp, col = _device_mask(masks, n_users, cuda_device)
    cut = [1, 10, 1000, m]
    rm = _ranker(I, precision, cuda_device).rank_metrics(U.to(cuda_device), torch.from_numpy(users), cut, trp, tcol,
                                                         rp, col)
    S = U.double().numpy() @ I.double().numpy().T
    pu = np.repeat(users, np.diff(trp))
    ref = _np_metrics(_exact_ranks(S, pu, tcol, masks), trp, tcol, users, masks, m, cut)
    for key in ("recall", "precision", "hit", "ndcg"):
        np.testing.assert_allclose(rm[key], ref[key], rtol=0, atol=1e-12, err_msg=key)
    assert abs(rm["mrr"] - ref["mrr"]) < 1e-12 and abs(rm["auc"] - ref["auc"]) < 1e-12, (rm, ref)


def test_rank_metrics_on_epinion2_match_fullrank_test(cuda_device, ep2_root):
    """All 3 185 epinion2 test users with the golden weights: rank_metrics at Ks equals main_rec.fullrank_test."""
    from test_epinion2_golden import _gpu_model

    from spex_b200 import batch_test, main_rec, ops
    from spex_b200.graph import truth_csr

    ds, model = _gpu_model(ep2_root, cuda_device)
    model.eval()
    ref = main_rec.fullrank_test(model, ds.testRatings)
    users = np.fromiter(ds.testRatings.keys(), dtype=np.int64, count=len(ds.testRatings))
    assert users.size == 3185
    all_users, all_items = model.computer()
    mrp, mcol = model.train_mask_csr()
    trp, tcol = truth_csr(users, ds.testRatings)
    r = ops.FullRanker(all_items, ops.default_precision(all_items.shape[1]), probe=True)
    got = r.rank_metrics(all_users, torch.from_numpy(users).to(cuda_device), batch_test.Ks, trp, tcol, mrp, mcol,
                         probe_users=torch.arange(all_users.shape[0], device=cuda_device))
    np.testing.assert_allclose(got["recall"], ref["recall"], rtol=0, atol=1e-12)
    np.testing.assert_allclose(got["ndcg"], ref["ndcg"], rtol=0, atol=1e-12)
    rk = model.item_ranks(users[:64], [ds.testRatings[int(u)][0] for u in users[:64]])
    assert rk.shape == (64,) and rk.dtype == torch.int32


def test_degenerate_table_goes_to_fp32_and_stays_in_bracket(cuda_device):
    """Almost parallel item rows: the probe sends the rank query to fp32, whose ranks meet the float64 bracket."""
    rng = np.random.default_rng(9)
    D, m, n_users = 64, 2000, 64
    base = rng.standard_normal(D)
    I = (base[None, :] + 1e-3 * rng.standard_normal((m, D))).astype(np.float32)
    U = (base[None, :] + 0.3 * rng.standard_normal((n_users, D))).astype(np.float32)
    Ud = torch.from_numpy(U).to(cuda_device)
    r = _ranker(torch.from_numpy(I), "f16", cuda_device, probe=True)
    users = torch.arange(n_users)
    assert r.scorer_for(None, Ud, users.to(cuda_device)) == "fp32"
    items = rng.integers(0, m, n_users)
    got = r.ranks(Ud, users, torch.from_numpy(items)).cpu().numpy()
    S = U.astype(np.float64) @ I.astype(np.float64).T
    for p, t in enumerate(items):
        delta = D * 2.0 ** -22 * np.linalg.norm(U[p]) * np.linalg.norm(I, axis=1).max()
        ok = np.arange(m) != t
        assert ((S[p] > S[p, t] + delta) & ok).sum() <= got[p] <= ((S[p] >= S[p, t] - delta) & ok).sum()


@pytest.mark.parametrize("precision", ["f16", "fp32"])
def test_ranks_deterministic_permutation_and_blocks(cuda_device, monkeypatch, precision):
    from spex_b200 import ops

    rng = np.random.default_rng(11)
    n_users, m, D, P = 500, 5000, 64, 3000
    U = torch.from_numpy(rng.standard_normal((n_users, D)).astype(np.float32)).to(cuda_device)
    I = torch.from_numpy(rng.standard_normal((m, D)).astype(np.float32))
    masks = _masks(rng, n_users, m)
    rp, col = _device_mask(masks, n_users, cuda_device)
    users = torch.from_numpy(rng.integers(0, n_users, P))
    items = torch.from_numpy(rng.integers(0, m, P))
    r = _ranker(I, precision, cuda_device)
    a = r.ranks(U, users, items, rp, col)
    assert torch.equal(a, r.ranks(U, users, items, rp, col))
    perm = torch.from_numpy(rng.permutation(P))
    assert torch.equal(a[perm.to(cuda_device)], r.ranks(U, users[perm], items[perm], rp, col))
    truth_rp = np.arange(n_users + 1, dtype=np.int64)
    truth_col = rng.integers(0, m, n_users).astype(np.int32)
    base = r.rank_metrics(U, torch.arange(n_users), [5, 50], truth_rp, truth_col, rp, col)
    for blk in (128, 1000):
        monkeypatch.setattr(ops, "RANK_PAIR_BLOCK", blk)
        assert torch.equal(a, r.ranks(U, users, items, rp, col)), blk
        got = r.rank_metrics(U, torch.arange(n_users), [5, 50], truth_rp, truth_col, rp, col)
        for key in ("recall", "precision", "ndcg", "hit"):
            assert np.array_equal(got[key], base[key]), (blk, key)
        assert got["mrr"] == base["mrr"] and got["auc"] == base["auc"]


def test_rejections_launch_nothing(cuda_device):
    from spex_b200 import _capi, ops
    from spex_b200._capi import lib, ptr

    dev = cuda_device
    D, P, m = 64, 130, 300
    Uh = torch.zeros(256 * D, dtype=torch.float16, device=dev)
    Ih = torch.zeros(384 * D, dtype=torch.float16, device=dev)
    meta = torch.ones(4, device=dev)
    items = torch.zeros(P, dtype=torch.int32, device=dev)
    out = torch.empty(P, dtype=torch.int32, device=dev)
    rp = torch.zeros(2, dtype=torch.int64, device=dev)
    cl = torch.zeros(1, dtype=torch.int32, device=dev)
    U = torch.zeros(4, D, device=dev)
    users = torch.zeros(P, dtype=torch.int64, device=dev)

    def f16(D=D, P_pad=256, m_pad=384, mrp=None, mcol=None, o=out):
        return lib.spex_rank_pairs_f16(ptr(Uh), ptr(Ih), D, None, None, ptr(items), P, P_pad, m, m_pad, ptr(meta),
                                       ptr(mrp), ptr(mcol), ptr(o), None)

    def f32(D=D, mrp=None, mcol=None, o=out):
        return lib.spex_rank_pairs_f32(ptr(U), ptr(U), D, ptr(users), ptr(items), P, 4, ptr(mrp), ptr(mcol), ptr(o),
                                       None)

    n0 = _capi.launch_count()
    assert f16(D=48) == -2 and f16(D=96) == -2 and f32(D=6) == -2 and f32(D=516) == -2
    assert f16(P_pad=200) == -1 and f16(m_pad=320) == -1
    assert f16(mrp=rp) == -1 and f16(mcol=cl) == -1 and f32(mrp=rp) == -1 and f32(mcol=cl) == -1
    assert f16(o=None) == -1 and f32(o=None) == -1
    assert _capi.launch_count() == n0
    r = ops.FullRanker(torch.zeros(m, D, device=dev), "fp32")
    with pytest.raises(ValueError, match="item ids"):
        r.ranks(U, torch.zeros(2, dtype=torch.int64), torch.tensor([0, m]))
    with pytest.raises(ValueError, match="item ids"):
        r.ranks(U, torch.zeros(1, dtype=torch.int64), torch.tensor([-1]))
    with pytest.raises(ValueError, match="bf16"):
        ops.FullRanker(torch.zeros(m, 64, device=dev), "bf16").ranks(U, users[:1], items[:1])
    assert _capi.launch_count() == n0


@pytest.mark.parametrize("precision,D", CASES)
def test_repeated_mask_ids_are_excluded_once(cuda_device, precision, D):
    """A mask row may repeat an id: the ranks and every metric equal those of the de-duplicated row."""
    gen = torch.Generator().manual_seed(21)
    rng = np.random.default_rng(21)
    n_users, m = 64, 700
    U, I = _dyadic(gen, n_users, D, -2), _dyadic(gen, m, D, -3)
    masks = _masks(rng, n_users, m)
    rows = [sorted(list(masks[u]) + list(masks[u])[:2]) for u in range(n_users)]   # first ids twice
    rp_dup = np.zeros(n_users + 1, np.int64)
    rp_dup[1:] = np.cumsum([len(r) for r in rows])
    col_dup = np.array([i for r in rows for i in r], np.int32)
    assert col_dup.size > sum(len(set(r)) for r in rows)
    dup = (torch.from_numpy(rp_dup).to(cuda_device), torch.from_numpy(col_dup).to(cuda_device))
    uniq = _device_mask(masks, n_users, cuda_device)
    r = _ranker(I, precision, cuda_device)
    Ud = U.to(cuda_device)
    users = np.repeat(np.arange(n_users), 4)
    items = rng.integers(0, m, users.size)
    a = r.ranks(Ud, torch.from_numpy(users), torch.from_numpy(items), *dup)
    b = r.ranks(Ud, torch.from_numpy(users), torch.from_numpy(items), *uniq)
    assert torch.equal(a, b)
    S = U.double().numpy() @ I.double().numpy().T
    np.testing.assert_array_equal(a.cpu().numpy(), _exact_ranks(S, users, items, masks))
    _, trp, tcol = _truth(rng, n_users, m, True)
    x = r.rank_metrics(Ud, torch.arange(n_users), [1, 10, m], trp, tcol, *dup)
    y = r.rank_metrics(Ud, torch.arange(n_users), [1, 10, m], trp, tcol, *uniq)
    for key in ("recall", "precision", "ndcg", "hit"):
        assert np.array_equal(x[key], y[key]), key
    assert x["mrr"] == y["mrr"] and x["auc"] == y["auc"]


def test_rank_metrics_rejections_launch_nothing(cuda_device):
    """spex_rank_metrics refuses bad cutoffs, half a mask and a mask without users before launching anything."""
    import ctypes as C

    from spex_b200 import _capi, ops
    from spex_b200._capi import lib, ptr

    dev = cuda_device
    B, m = 4, 100
    ranks = torch.zeros(B, dtype=torch.int32, device=dev)
    trp = torch.arange(B + 1, dtype=torch.int64, device=dev)
    tcol = torch.zeros(B, dtype=torch.int32, device=dev)
    users = torch.arange(B, dtype=torch.int64, device=dev)
    mrp = torch.zeros(B + 1, dtype=torch.int64, device=dev)
    mcol = torch.zeros(1, dtype=torch.int32, device=dev)
    disc = torch.ones(m, dtype=torch.float64, device=dev)
    idcg = torch.ones(m + 1, dtype=torch.float64, device=dev)
    cs = torch.zeros(1, 9, 4, dtype=torch.float64, device=dev)
    ce = torch.zeros(1, 4, dtype=torch.float64, device=dev)

    def call(cuts, users=users, mrp=None, mcol=None, m_items=m):
        cut = (C.c_int32 * len(cuts))(*cuts)
        return lib.spex_rank_metrics(ptr(ranks), B, ptr(trp), ptr(tcol), ptr(users), ptr(mrp), ptr(mcol), m_items,
                                     cut, len(cuts), ptr(disc), ptr(idcg), ptr(cs), ptr(ce), None)

    n0 = _capi.launch_count()
    assert call(list(range(1, 10))) == -5                      # n_cut > 8
    assert call([10, 5]) == -1 and call([5, 5]) == -1          # not strictly ascending
    assert call([0]) == -1 and call([m + 1]) == -1             # outside [1, m]
    assert call([5], m_items=0) == -1
    assert call([5], mrp=mrp) == -1 and call([5], mcol=mcol) == -1   # half a mask
    assert call([5], users=None, mrp=mrp, mcol=mcol) == -1     # a mask without users
    assert _capi.launch_count() == n0
    r = ops.FullRanker(torch.zeros(m, 48, device=dev), "fp32")
    with pytest.raises(ValueError, match="m_items"):
        r.rank_metrics(torch.zeros(B, 48, device=dev), users, [5, m + 1], trp, tcol)
    with pytest.raises(ValueError, match="ascending"):
        r.rank_metrics(torch.zeros(B, 48, device=dev), users, [5, 5], trp, tcol)
    assert _capi.launch_count() == n0
