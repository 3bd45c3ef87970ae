"""Full-ranking Recall / precision / NDCG / hit rate on the device (spex_fullrank_metrics, FullRanker.evaluate,
ShardedEvaluator.evaluate, main_rec --test_mode fullrank) against the float64 host formula
metrics.fullrank_recall_ndcg."""
import ctypes as C
import re
import shutil

import numpy as np
import pytest
import torch

from spex_b200 import graph, metrics

SPEX_E_BADARG, SPEX_E_TOOBIG = -1, -5


# ---------------------------------------------------------------------------------------------------------------
# host reference
def _host_metrics(topk, rp, col, cutoffs):
    """[B, n_cut, 4] (recall, precision, ndcg, hit): recall / ndcg from metrics.fullrank_recall_ndcg, hits by
    np.isin as there."""
    B = topk.shape[0]
    out = np.zeros((B, len(cutoffs), 4))
    for j, K in enumerate(cutoffs):
        rec, ndcg = metrics.fullrank_recall_ndcg(topk, rp, col, K)
        hits = np.array([np.isin(topk[u, :K], col[rp[u]: rp[u + 1]]).sum() if rp[u + 1] > rp[u] else 0
                         for u in range(B)], dtype=np.float64)
        out[:, j] = np.stack([rec, hits / K, ndcg, (hits > 0).astype(np.float64)], axis=1) if B else 0
    return out


def _case(B, k, seed):
    """Distinct ids per row (as every scorer returns), -1 padding on every 7th row; truth rows cycle through:
    empty, longer than k, hits planted at ranks 0 and k - 1, duplicate ids, a few random ids."""
    rng = np.random.default_rng(seed)
    m = 2 * k + 40
    topk = np.stack([rng.permutation(m)[:k] for _ in range(B)]).astype(np.int32) if B else np.zeros((0, k), np.int32)
    for u in range(0, B, 7):
        topk[u, k - int(rng.integers(1, k + 1)):] = -1
    rows = []
    for u in range(B):
        kind = (u + (B == 1) * 2) % 5
        if kind == 0:
            t = []
        elif kind == 1:
            t = rng.choice(m, size=k + 7, replace=False).tolist()
        elif kind == 2:
            t = [int(x) for x in (topk[u, 0], topk[u, k - 1]) if x >= 0] + rng.integers(0, m, 2).tolist()
        elif kind == 3:
            x = int(topk[u, min(3, k - 1)]) if topk[u, min(3, k - 1)] >= 0 else 0
            t = [x, x, x, int(rng.integers(0, m))]
        else:
            t = rng.integers(0, m, int(rng.integers(1, 6))).tolist()
        rows.append(np.sort(np.asarray(t, np.int64)))
    rp = np.zeros(B + 1, np.int64)
    rp[1:] = np.cumsum([r.size for r in rows]) if B else []
    col = np.concatenate(rows).astype(np.int64) if B and rp[-1] else np.zeros(0, np.int64)
    return topk, rp, col


def _device_metrics(dev, topk, rp, col, cutoffs):
    from spex_b200 import ops
    from spex_b200._capi import call, ptr, stream_ptr

    B, k = topk.shape
    n_cut = len(cutoffs)
    t = torch.from_numpy(topk).to(dev)
    trp = torch.from_numpy(rp).to(dev)
    tcol = torch.from_numpy(col.astype(np.int32) if col.size else np.zeros(1, np.int32)).to(dev)
    disc, idcg = (torch.from_numpy(a).to(dev) for a in ops.rank_discounts(k))
    n_chunks = (B + ops.METRICS_CHUNK - 1) // ops.METRICS_CHUNK
    pu = torch.full((B, n_cut, 4), -7.0, dtype=torch.float64, device=dev)
    cs = torch.empty(n_chunks, n_cut, 4, dtype=torch.float64, device=dev)
    sums = torch.full((n_cut, 4), -7.0, dtype=torch.float64, device=dev)
    call("spex_fullrank_metrics", ptr(t), B, k, ptr(trp), ptr(tcol), (C.c_int32 * n_cut)(*cutoffs), n_cut,
         ptr(disc), ptr(idcg), ptr(pu), ptr(cs), stream_ptr())
    call("spex_fullrank_metrics_reduce", ptr(cs), n_chunks, n_cut, ptr(sums), stream_ptr())
    return pu.cpu().numpy(), cs.cpu().numpy(), sums.cpu().numpy()


@pytest.mark.gpu
@pytest.mark.parametrize("k,cutoff_sets", [(1, [[1]]), (20, [[20], [1, 5, 10, 20]]), (50, [[10, 20, 50]]),
                                           (64, [[1, 2, 3, 4, 8, 16, 32, 64], [33, 63]]),
                                           (100, [[10, 20, 50, 100], [64, 99]]), (512, [[1, 100, 511, 512]])])
@pytest.mark.parametrize("B", [0, 1, 2500])
def test_kernel_matches_host_formula(cuda_device, k, cutoff_sets, B):
    topk, rp, col = _case(B, k, seed=B * 1000 + k)
    for cutoffs in cutoff_sets:
        got, cs, sums = _device_metrics(cuda_device, topk, rp, col, cutoffs)
        ref = _host_metrics(topk, rp, col, cutoffs)
        assert got.shape == ref.shape
        for j in (0, 1, 3):                      # recall, precision, hit: bit-equal
            assert np.array_equal(got[..., j], ref[..., j]), (k, cutoffs, j)
        assert np.abs(got[..., 2] - ref[..., 2]).max(initial=0.0) <= 1e-13, (k, cutoffs)
        # chunk sums are the per-chunk sums of the per-user values, the totals their ascending sum
        for c in range(cs.shape[0]):
            assert np.allclose(cs[c], got[c * 1024: (c + 1) * 1024].sum(0), rtol=1e-14, atol=1e-12)
        want = np.zeros_like(sums)
        for c in range(cs.shape[0]):
            want += cs[c]
        assert np.array_equal(sums, want)


def _eval_tables(dev, n_u=5000, m=3000, D=64, seed=5):
    from spex_b200.graph import build_interaction_csr

    g = torch.Generator().manual_seed(seed)
    U = (torch.randn(n_u, D, generator=g) * 0.3).to(dev)
    I = (torch.randn(m, D, generator=g) * 0.3).to(dev)
    rng = np.random.default_rng(seed)
    mrp, mcol = build_interaction_csr(rng.integers(0, n_u, 40000), rng.integers(0, m, 40000), n_u, m)
    users = rng.permutation(n_u)[: n_u - 37]
    truth = {int(u): rng.integers(0, m, int(rng.integers(0, 5))).tolist() for u in users[::2]}
    trp, tcol = graph.truth_csr(users, truth)
    return U, I, torch.from_numpy(mrp).to(dev), torch.from_numpy(mcol).to(dev), users, trp, tcol


@pytest.mark.gpu
@pytest.mark.parametrize("precision", ["f16", "bf16", "fp32"])
def test_evaluate_is_deterministic_and_independent_of_the_user_block(cuda_device, precision):
    from spex_b200 import ops

    U, I, mrp, mcol, users, trp, tcol = _eval_tables(cuda_device)
    ranker = ops.FullRanker(I, precision)
    res = []
    for _ in range(2):
        for block in (1024, 3072, None):
            res.append(ranker.evaluate(U, users, [5, 10, 20, 50], trp, tcol, mrp, mcol, user_block=block,
                                       per_user=True))
    for r in res[1:]:
        assert r["users"] == res[0]["users"] == users.size
        for name in ops.METRIC_NAMES:
            assert np.array_equal(r[name], res[0][name]), name
        assert torch.equal(r["per_user"], res[0]["per_user"])
    # the means are those of the per-user values, which are the host formula on the ranking
    idx, _ = ranker.topk(U, users, 50, mrp, mcol)
    ref = _host_metrics(idx.cpu().numpy(), trp, tcol, [5, 10, 20, 50])
    pu = res[0]["per_user"].cpu().numpy()
    assert np.array_equal(pu[..., [0, 1, 3]], ref[..., [0, 1, 3]])
    assert np.abs(pu[..., 2] - ref[..., 2]).max() <= 1e-13
    assert np.allclose(res[0]["recall"], ref[..., 0].mean(0), rtol=0, atol=1e-14)


@pytest.mark.gpu
@pytest.mark.parametrize("precision", ["f16", "bf16", "fp32"])
def test_sharded_evaluate_matches_recall_ndcg_and_test_fullrank(cuda_device, precision):
    from spex_b200 import batch_test
    from spex_b200.dist import ShardedEvaluator
    from test_gpu_parity import _small_model

    ds, model, _, _ = _small_model(cuda_device)
    model.eval()
    users = np.arange(ds.n_users)
    au, ai = model.computer()
    mrp, mcol = model.train_mask_csr()
    ev = ShardedEvaluator(au, ai, mrp, mcol, k=20, scorer=precision)
    assert ev.scorer == precision
    truth = {int(u): list(ds.testRatings[u]) for u in users if u in ds.testRatings}
    trp, tcol = graph.truth_csr(users, truth)
    users_d = torch.from_numpy(users).to(cuda_device)
    got = ev.evaluate(users_d, trp, tcol, [20])
    ref = batch_test.test_fullrank(model, users, truth, k=20, precision=precision)
    assert got["users"] == ds.n_users
    assert abs(got["recall"][0] - ref["recall"]) < 1e-12 and abs(got["ndcg"][0] - ref["ndcg"]) < 1e-12
    wide = [64, 100] if precision == "f16" else []          # f16 at k = 100: the wide kernel
    for cutoffs in ([10, 20, 50], wide):
        if not cutoffs:
            continue
        got = ev.evaluate(users_d, trp, tcol, cutoffs)
        for j, K in enumerate(cutoffs):
            ref = batch_test.test_fullrank(model, users, truth, k=K, precision=precision)
            assert abs(got["recall"][j] - ref["recall"]) < 1e-12, (precision, K)
            assert abs(got["ndcg"][j] - ref["ndcg"]) < 1e-12, (precision, K)


@pytest.mark.gpu
def test_cutoffs_are_prefixes_of_one_ranking(cuda_device):
    from spex_b200 import ops

    U, I, mrp, mcol, users, trp, tcol = _eval_tables(cuda_device, n_u=3000, m=2000, D=40, seed=9)
    ranker = ops.FullRanker(I, "fp32")
    cutoffs = [1, 7, 20, 50]
    one = ranker.evaluate(U, users, cutoffs, trp, tcol, mrp, mcol, per_user=True)
    for j, K in enumerate(cutoffs):
        sep = ranker.evaluate(U, users, [K], trp, tcol, mrp, mcol, per_user=True)
        assert torch.equal(one["per_user"][:, j], sep["per_user"][:, 0]), K
        for name in ops.METRIC_NAMES:
            assert one[name][j] == sep[name][0], (K, name)


def test_rejections_launch_nothing():
    """Every bad argument is refused before a launch (no GPU needed: nothing reaches the device)."""
    from spex_b200 import _capi, ops

    lib = _capi.lib
    fake = C.c_void_p(1 << 20)                  # never dereferenced: every call below is refused first
    n0 = ops.launch_count()

    def run(k, cuts, n_cut=None, B=4, topk=fake, chunk=fake, disc=fake):
        n = len(cuts) if n_cut is None else n_cut
        return lib.spex_fullrank_metrics(topk, B, k, fake, fake, (C.c_int32 * max(len(cuts), 1))(*cuts), n, disc,
                                         fake, None, chunk, None)

    assert run(513, [10]) == SPEX_E_TOOBIG
    assert run(64, list(range(1, 10))) == SPEX_E_TOOBIG
    assert run(20, [10, 10]) == SPEX_E_BADARG
    assert run(20, [10, 5]) == SPEX_E_BADARG
    assert run(20, [0, 5]) == SPEX_E_BADARG
    assert run(20, [5, 21]) == SPEX_E_BADARG
    assert run(0, [1]) == SPEX_E_BADARG
    assert run(20, [], n_cut=0) == SPEX_E_BADARG
    assert run(20, [5], B=-1) == SPEX_E_BADARG
    assert run(20, [5], topk=None) == SPEX_E_BADARG
    assert run(20, [5], chunk=None) == SPEX_E_BADARG
    assert run(20, [5], disc=None) == SPEX_E_BADARG
    assert lib.spex_fullrank_metrics(fake, 4, 20, fake, fake, None, 1, fake, fake, None, fake, None) == SPEX_E_BADARG
    assert lib.spex_fullrank_metrics_reduce(fake, 3, 9, fake, None) == SPEX_E_TOOBIG
    assert lib.spex_fullrank_metrics_reduce(fake, 3, 2, None, None) == SPEX_E_BADARG
    assert lib.spex_fullrank_metrics_reduce(None, 3, 2, fake, None) == SPEX_E_BADARG
    assert lib.spex_fullrank_metrics_reduce(fake, -1, 2, fake, None) == SPEX_E_BADARG
    assert ops.launch_count() == n0
    for bad in ([], [5, 5], [0, 3], list(range(1, 10))):
        with pytest.raises(ValueError):
            ops.check_cutoffs(bad)


@pytest.mark.gpu
def test_evaluate_rejects_unsorted_truth(cuda_device):
    from spex_b200 import ops

    U, I, mrp, mcol, users, trp, tcol = _eval_tables(cuda_device, n_u=600, m=500)
    ranker = ops.FullRanker(I, "fp32")
    r = int(np.nonzero(np.diff(trp) >= 2)[0][0])
    bad = tcol.copy()
    bad[trp[r]: trp[r + 1]] = bad[trp[r]: trp[r + 1]][::-1]
    assert bad[trp[r]] > bad[trp[r + 1] - 1]
    n0 = ops.launch_count()
    with pytest.raises(ValueError, match="sorted"):
        ranker.evaluate(U, users, [10], trp, bad, mrp, mcol)
    with pytest.raises(ValueError, match="rowptr"):
        ranker.evaluate(U, users, [10], trp[:-1], tcol, mrp, mcol)
    with pytest.raises(ValueError):
        ranker.evaluate(U, users, [10, 10], trp, tcol, mrp, mcol)
    assert ops.launch_count() == n0
    # an empty user list, and users none of which has held-out items
    e = ranker.evaluate(U, users[:0], [10], np.zeros(1, np.int64), np.zeros(0, np.int32))
    assert e["users"] == 0 and e["recall"].tolist() == [0.0]
    z = ranker.evaluate(U, users[:5], [3, 10], np.zeros(6, np.int64), np.zeros(0, np.int32))
    assert z["users"] == 5 and all(z[n].tolist() == [0.0, 0.0] for n in ops.METRIC_NAMES)


def test_discounts_and_truth_csr_on_the_host():
    from spex_b200 import ops

    disc, idcg = ops.rank_discounts(512)
    for k in (1, 20, 50, 512):          # the expressions of metrics.fullrank_recall_ndcg, prefixes of k = 512
        d = 1.0 / np.log2(np.arange(2, k + 2))
        cum = np.concatenate([[0.0], np.cumsum(d)])
        assert np.array_equal(disc[:k], d) and np.array_equal(idcg[: k + 1], cum)
    rp, col = graph.truth_csr([7, 3, 9, 4], {3: [5, 2, 5], 4: [1], 8: [6]})
    assert rp.tolist() == [0, 0, 2, 2, 3] and col.tolist() == [2, 5, 1]
    rp, col = graph.truth_csr([1, 2], {})
    assert rp.tolist() == [0, 0, 0] and col.size == 0


def test_test_mode_flag_keeps_the_reference_namespace():
    from spex_b200.lg_parser import parse_args_r

    assert not hasattr(parse_args_r([]), "test_mode")
    assert parse_args_r(["--test_mode", "fullrank"]).test_mode == "fullrank"
    assert parse_args_r(["--test_mode", "sampled"]).test_mode == "sampled"
    with pytest.raises(SystemExit):
        parse_args_r(["--test_mode", "other"])


@pytest.mark.gpu
def test_main_rec_fullrank_test_mode(tmp_path, capsys, monkeypatch):
    import os

    from spex_b200 import batch_test, main_rec, ops

    shutil.copytree(os.path.join(os.path.dirname(__file__), "golden", "tiny"), tmp_path / "tiny")
    seen = []
    orig = main_rec.Test

    def spy(dataset, Recmodel, epoch, *a, **kw):
        out = orig(dataset, Recmodel, epoch, *a, **kw)
        # the reference at the same weights: the host metrics of test_fullrank on the scorer the evaluator picks
        # (its probe samples all users; test_fullrank's, through rank_topk, the test users)
        au, ai = Recmodel.computer()
        users = np.fromiter(dataset.testRatings.keys(), np.int64)
        ranker = ops.FullRanker(ai, ops.default_precision(ai.shape[1]), probe=True)
        prec = ranker.scorer_for(max(batch_test.Ks), au, torch.arange(au.shape[0], device=au.device))
        if prec == "f16":
            assert ranker.scorer_for(max(batch_test.Ks), au, torch.from_numpy(users).to(au.device)) == "f16"
        seen.append([batch_test.test_fullrank(Recmodel, users, dataset.testRatings, k=K, precision=prec)
                     for K in batch_test.Ks])
        return out

    monkeypatch.setattr(main_rec, "Test", spy)
    main_rec.main(["--dataset", "tiny", "--data_path", str(tmp_path), "--epochs", "2", "--seed", "2020",
                   "--test_mode", "fullrank"])
    out = capsys.readouterr().out.splitlines()
    rec_lines = [l for l in out if l.startswith("Rec:  Epoch ")]
    assert len(rec_lines) == 2 and len(seen) == 2
    for line, ref in zip(rec_lines, seen):
        assert re.fullmatch(r"Rec:  Epoch \d+ : recall=\[\d\.\d{4}, \d\.\d{4}, \d\.\d{4}\],  ndcg=\[\d\.\d{4}, \d\.\d{4}, \d\.\d{4}\]", line)
        want = "recall=[%.4f, %.4f, %.4f],  ndcg=[%.4f, %.4f, %.4f]" % (
            *(r["recall"] for r in ref), *(r["ndcg"] for r in ref))
        assert line.endswith(want), (line, want)
    assert "--- Train Best ---" in out
