"""spex_score_topk_f16_wide: the fp16-accumulator tensor-core scorer for 1 <= k <= 512, whose per-row candidate
buffers live in a caller-owned workspace, against the exact float64 top-k of test_gpu_ranking_edges.py (dyadic
integer tables: every summation order gives the same bits), and the public callers that route k > 64 to it."""
import numpy as np
import pytest
import torch

from test_epinion2_golden import ep2_root  # noqa: F401  (module fixture: the epinion2 dataset on disk)
from test_gpu_ranking_edges import (SENT_IDX, SENT_VAL, _assert_exact, _dyadic, _mask_csr, _operands, _pack,
                                    _random_masks, _reference, _round_up)

pytestmark = pytest.mark.gpu

KS = [1, 65, 100, 128, 129, 256, 511, 512]


def _cap(k):
    return (2 * k + 64 + 31) // 32 * 32


def _wide(U, I, users, k, masks=None, pass_ids=True, extra_cta=False, dev=None):
    """The wide scorer on host tables (as _score of test_gpu_ranking_edges.py): (idx, val, reference)."""
    from spex_b200 import ops

    B, D, m = users.numel(), U.shape[1], I.shape[0]
    Ud, Id, ud = U.to(dev), I.to(dev), users.to(dev)
    rp = col = None
    if masks is not None:
        rp_h, col_h = _mask_csr(masks, U.shape[0])
        rp, col = torch.from_numpy(rp_h).to(dev), torch.from_numpy(col_h).to(dev)
    mask_rows = users.numpy() if pass_ids else np.arange(B)
    masked = [masks.get(int(r), []) if masks is not None else [] for r in mask_rows]
    b_pad = _round_up(B, 128) + (128 if extra_cta else 0)
    m_pad = _round_up(m, 128)
    out_i = torch.full((b_pad, k), SENT_IDX, dtype=torch.int32, device=dev)
    out_v = torch.full((b_pad, k), SENT_VAL, dtype=torch.float32, device=dev)
    Uh, umeta = _pack("f16", Ud, ud, b_pad, D)
    Ih, imeta = _pack("f16", Id, None, m_pad, D)
    ops.score_topk_f16_wide(Uh, umeta, B, b_pad, Ih, imeta, m, m_pad, D, k, ud if pass_ids else None, rp, col,
                            out_i, out_v)
    scores = _operands(U[users], umeta.cpu()) @ _operands(I, imeta.cpu()).t()
    torch.cuda.synchronize()
    assert bool((out_i[B:] == SENT_IDX).all()) and bool((out_v[B:] == SENT_VAL).all()), "a padded row wrote output"
    return out_i[:B], out_v[:B], _reference(scores, masked, k)


# ---- 1. bit-exact against float64 --------------------------------------------------------------------------------
@pytest.mark.parametrize("D", [64, 128])
@pytest.mark.parametrize("k", KS)
def test_wide_bit_exact(cuda_device, D, k):
    gen = torch.Generator().manual_seed(D * 1000 + k)
    rng = np.random.default_rng(k)
    n_u = 200
    # several buffer compactions per row (m > 2 cap), masks on both sides of 16/128/256, permuted ids, a padded CTA
    m = 2 * _cap(k) + 37
    users = torch.randperm(n_u, generator=gen)[:129]
    masks = _random_masks(rng, n_u, m, max_per_row=30)
    U, I = _dyadic(gen, n_u, D, exp=-3), _dyadic(gen, m, D, exp=2)
    _assert_exact(*_wide(U, I, users, k, masks, extra_cta=True, dev=cuda_device), (D, k, "compactions"))
    # NULL user ids, and duplicated ones
    _assert_exact(*_wide(U, I, torch.arange(130), k, masks, pass_ids=False, dev=cuda_device), (D, k, "null ids"))
    dup = torch.randint(0, 40, (131,), generator=gen)
    idx, val, ref = _wide(U, I, dup, k, masks, dev=cuda_device)
    _assert_exact(idx, val, ref, (D, k, "dup ids"))
    first = {int(u): b for b, u in reversed(list(enumerate(dup.tolist())))}
    assert all(torch.equal(idx[b], idx[first[u]]) for b, u in enumerate(dup.tolist()))
    # one item tile
    I1 = _dyadic(gen, 100, D, exp=0)
    _assert_exact(*_wide(U, I1, users, k, _random_masks(rng, n_u, 100), dev=cuda_device), (D, k, "one tile"))
    # all scores negative, m not a multiple of 128 and, for k > 1, m < k: padded items must never appear and the
    # slots past the unmasked items are -1 / -inf
    mneg = max(k // 2 + 5, 7) if k > 1 else 133
    Up = _dyadic(gen, n_u, D, exp=-2, lo=1, hi=8)
    In = _dyadic(gen, mneg, D, exp=1, lo=-8, hi=-1)
    idx, val, ref = _wide(Up, In, users, k, _random_masks(rng, n_u, mneg), dev=cuda_device)
    assert int(idx.max()) < mneg
    n_valid = (ref[0] >= 0).sum(axis=1)
    ids, vals = idx.cpu().numpy(), val.cpu().numpy()
    for b in range(ids.shape[0]):
        assert (ids[b, n_valid[b]:] == -1).all() and np.isneginf(vals[b, n_valid[b]:]).all()
    _assert_exact(idx, val, ref, (D, k, "negative"))


# ---- 2. every score ties ------------------------------------------------------------------------------------------
@pytest.mark.parametrize("D", [64, 128])
@pytest.mark.parametrize("k", [65, 512])
def test_wide_all_ties(cuda_device, D, k):
    """Every item row identical: each overflow takes the exact compaction form, which must keep exactly k entries
    (lowest ids) and terminate; the output is the unmasked ids in ascending order."""
    gen = torch.Generator().manual_seed(k + D)
    rng = np.random.default_rng(D)
    n_u, m = 150, 4 * _cap(k) + 11
    U = _dyadic(gen, n_u, D, exp=-1)
    I = _dyadic(gen, 1, D, exp=0).expand(m, D).contiguous()
    users = torch.arange(n_u)
    masks = _random_masks(rng, n_u, m, max_per_row=40)
    idx, val, ref = _wide(U, I, users, k, masks, dev=cuda_device)
    _assert_exact(idx, val, ref, (D, k))
    for b in range(0, n_u, 7):
        skip = set(masks[b])
        assert idx[b].tolist() == [i for i in range(m) if i not in skip][:k]


# ---- 3. the filter margin at k > 64 -------------------------------------------------------------------------------
@pytest.mark.parametrize("D", [64, 128])
@pytest.mark.parametrize("k", [100, 300])
def test_wide_filter_margin_adversarial(cuda_device, D, k):
    """The construction of test_f16_filter_margin_adversarial with more decoys than the wide buffer holds, so the
    threshold rises (exact compactions of the tied decoys) before the adversarial items arrive: none of the k true
    top items may be dropped."""
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
    assert s_adv - 2.0 ** -9 < float(u @ dec) < s_adv
    n_dec, n_adv = 2 * _cap(k) + 100, k + 20
    adv_ids = n_dec + 100 + 12 * np.arange(n_adv)
    m = int(adv_ids[-1]) + 37
    I = np.zeros((m, D))
    I[:, :16] = -1.0
    I[:n_dec] = dec
    I[adv_ids] = adv
    n_u = 130
    U = np.tile(u, (n_u, 1)) * (2.0 ** -(np.arange(n_u) % 3))[:, None]
    U, I = torch.from_numpy(U).float(), torch.from_numpy(I).float()
    idx, val, ref = _wide(U, I, torch.arange(n_u), k, dev=cuda_device)
    assert (ref[0] == adv_ids[:k]).all()
    _assert_exact(idx, val, ref, (D, k))


# ---- 4. prefix property and agreement with the fp32 scorer on random tables ---------------------------------------
def _random_tables(D, n_u, m, seed):
    gen = torch.Generator().manual_seed(seed)
    U = torch.randn(n_u, D, generator=gen)
    I = torch.randn(m, D, generator=gen) * (6.0 / (m + D)) ** 0.5
    n = I[1::3].shape[0]
    I[0: 3 * n: 3] = I[1::3]                                # duplicated rows: exact ties
    return U, I


@pytest.mark.parametrize("D", [64, 128])
def test_wide_prefix_and_fp32_agreement(cuda_device, D):
    from spex_b200 import ops

    dev = cuda_device
    n_u, m = 2048, 100_003
    U, I = _random_tables(D, n_u, m, seed=D)
    rng = np.random.default_rng(D)
    masks = _random_masks(rng, n_u, m, max_per_row=50)
    rp_h, col_h = _mask_csr(masks, n_u)
    rp, col = torch.from_numpy(rp_h).to(dev), torch.from_numpy(col_h).to(dev)
    Ud, Id = U.to(dev), I.to(dev)
    users = torch.randperm(n_u, generator=torch.Generator().manual_seed(1)).to(dev)
    Ih, m_pad, imeta = ops.pack_f16(Id, None, ops.TC_ITEM_MULTIPLE)
    Uh, b_pad, umeta = ops.pack_f16(Ud, users, ops.TC_USER_MULTIPLE)
    args = (Uh, umeta, n_u, b_pad, Ih, imeta, m, m_pad, D)
    i512, v512 = ops.score_topk_f16_wide(*args, 512, users, rp, col)
    i64, v64 = ops.score_topk_f16(*args, 64, users, rp, col)
    torch.cuda.synchronize()
    assert torch.equal(i512[:, :64], i64) and torch.equal(v512[:, :64].view(torch.int32), v64.view(torch.int32))
    assert bool((v512[:, 1:] <= v512[:, :-1]).all())
    i128, v128 = ops.score_topk_f16_wide(*args, 128, users, rp, col)
    torch.cuda.synchronize()
    assert torch.equal(i512[:, :128], i128) and torch.equal(v512[:, :128].view(torch.int32), v128.view(torch.int32))
    _check_vs_fp32_on_operands(i128, v128, Ud, Id, users, umeta, imeta, rp, col)


def _check_vs_fp32_on_operands(idx, val, U, I, users, umeta, imeta, rp=None, col=None, min_same=0.99):
    """The f16 scorers return the exact top-k of the fp16 operands: spex_score_topk_f32 on the decoded operands
    gives the same ids except near-ties, and values within the FMA-order tolerance (2 D 2^-24 |u| max|v|)."""
    from spex_b200 import ops

    k, D = idx.shape[1], U.shape[1]
    uop = _operands(U, umeta).float()
    iop = _operands(I, imeta).float()
    f_i, f_v = ops.score_topk_f32(uop, iop, users, k, rp, col)
    torch.cuda.synchronize()
    tol = (2 * D * 2.0 ** -24 * uop[users].norm(dim=1) * iop.norm(dim=1).max())[:, None]
    assert bool(((val - f_v).abs() <= tol).all())
    same = idx == f_i
    assert float(same.float().mean()) > min_same, float(same.float().mean())
    # a differing id is a swap within the tolerance: its exact score is within tol of the slot's fp32 value
    bad = torch.nonzero(~same)
    if bad.numel():
        b, p = bad[:, 0], bad[:, 1]
        s = (uop[users[b]].double() * iop[idx[b, p].long()].double()).sum(1)
        assert bool(((s - f_v[b, p].double()).abs() <= 2 * tol[b, 0].double()).all())


# ---- 5. determinism -----------------------------------------------------------------------------------------------
@pytest.mark.parametrize("k", [100, 300])
def test_wide_deterministic_and_independent_of_user_block(cuda_device, k):
    from spex_b200 import ops

    dev = cuda_device
    U, I = _random_tables(64, 3000, 40_000, seed=k)
    Ud, Id = U.to(dev), I.to(dev)
    users = torch.randperm(3000, generator=torch.Generator().manual_seed(k)).to(dev)
    ranker = ops.FullRanker(Id, "f16")
    got = [ranker.topk(Ud, users, k, user_block=b) for b in (None, None, 128, 1000)]
    torch.cuda.synchronize()
    i0, v0 = got[0]
    for i, v in got[1:]:
        assert torch.equal(i, i0) and torch.equal(v.view(torch.int32), v0.view(torch.int32))


# ---- 6. argument errors launch nothing ----------------------------------------------------------------------------
def test_wide_rejections_launch_nothing(cuda_device):
    import ctypes as C

    from spex_b200 import _capi
    from spex_b200._capi import ptr

    dev = cuda_device
    buf = torch.zeros(1 << 16, dtype=torch.float32, device=dev)
    p = ptr(buf)
    users = torch.arange(128, device=dev)
    rp = torch.zeros(129, dtype=torch.int64, device=dev)
    col = torch.zeros(1, dtype=torch.int32, device=dev)
    BADARG, BADDIM, ALIGN, TOOBIG, WORKSPACE = -1, -2, -3, -5, -6
    lib, s = _capi.lib, C.c_void_p(torch.cuda.current_stream().cuda_stream)
    ws_bytes = lib.spex_score_topk_f16_wide_workspace_bytes
    assert ws_bytes(128, 100) == 128 * _cap(100) * 8 and ws_bytes(256, 512) == 256 * 1088 * 8
    assert ws_bytes(128, 0) == 0 and ws_bytes(128, 513) == 0 and ws_bytes(-128, 100) == 0
    work = torch.zeros(ws_bytes(256, 512) // 4 + 4, dtype=torch.float32, device=dev)

    def wide(D=64, B_pad=128, m_pad=128, k=100, rpp=None, colp=None, w=None, nbytes=None):
        w = ptr(work) if w is None else w
        nbytes = ws_bytes(B_pad, k) if nbytes is None else nbytes
        return lib.spex_score_topk_f16_wide(p, p, D, 128, B_pad, 128, m_pad, p, p, ptr(users), rpp, colp, k, p, p,
                                            w, nbytes, s)

    before = _capi.launch_count()
    cases = [
        (wide(k=0), TOOBIG), (wide(k=513), TOOBIG), (wide(k=-1), TOOBIG),
        (wide(w=C.c_void_p(0)), WORKSPACE), (wide(nbytes=ws_bytes(128, 100) - 8), WORKSPACE),
        (wide(k=512, nbytes=ws_bytes(128, 400)), WORKSPACE),
        (wide(w=C.c_void_p(work.data_ptr() + 8)), ALIGN),
        (wide(B_pad=192), BADARG), (wide(m_pad=130), BADARG),
        (wide(rpp=ptr(rp)), BADARG), (wide(colp=ptr(col)), BADARG),
        (wide(D=32), BADDIM), (wide(D=96), BADDIM), (wide(D=256), BADDIM),
    ]
    assert [c[0] for c in cases] == [c[1] for c in cases]
    assert _capi.launch_count() == before
    oi = torch.empty(128, 100, dtype=torch.int32, device=dev)
    ov = torch.empty(128, 100, dtype=torch.float32, device=dev)
    Uh = torch.zeros(128 * 64, dtype=torch.float16, device=dev)
    meta = torch.tensor([1.0, 1.0, 1.0, 1.0], device=dev)
    rc = lib.spex_score_topk_f16_wide(ptr(Uh), ptr(Uh), 64, 128, 128, 128, 128, ptr(meta), ptr(meta), None, None,
                                      None, 100, ptr(oi), ptr(ov), ptr(work), ws_bytes(128, 100), s)
    torch.cuda.synchronize()
    assert rc == 0 and _capi.launch_count() == before + 1              # the valid call does launch
    assert oi.tolist() == [list(range(100))] * 128                      # every score 0: ascending ids


# ---- 7. the public callers ----------------------------------------------------------------------------------------
def _train_items(model, users):
    rp, col = (t.cpu().numpy() for t in model.train_mask_csr())
    return [set(col[rp[u]: rp[u + 1]].tolist()) for u in users]


def _near_tie_agreement(i_a, v_a, i_b, v_b, rtol=2e-3):
    """Two rankings of the same table with fp16 and fp32 operands: values close, mostly the same items."""
    scale = float(v_b.abs().max())
    assert float((v_a - v_b).abs().max()) <= rtol * scale
    overlap = [len(set(a) & set(b)) / len(a) for a, b in zip(i_a.cpu().tolist(), i_b.cpu().tolist())]
    assert np.mean(overlap) > 0.95, np.mean(overlap)


def test_lightgcn_rank_topk_wide_on_epinion2(cuda_device, ep2_root):
    from test_epinion2_golden import _gpu_model

    ds, model = _gpu_model(ep2_root, cuda_device)
    model.eval()
    users = np.arange(ds.n_users)
    i100, v100 = model.rank_topk(users, k=100)
    i32, v32 = model.rank_topk(users, k=100, precision="fp32")
    _near_tie_agreement(i100, v100, i32, v32)
    w_i, w_v = model.rank_topk(users, k=100, probe=False)              # the wide kernel whatever the probe says
    _near_tie_agreement(w_i, w_v, i32, v32)
    i300, v300 = model.rank_topk(users, k=300)
    torch.cuda.synchronize()
    assert i300.shape == (ds.n_users, 300)
    assert bool((v300[:, 1:] <= v300[:, :-1]).all())
    ids = i300.cpu().numpy()
    assert ids.min() >= 0 and ids.max() < ds.m_items
    for u, row, train in zip(users, ids, _train_items(model, users)):
        assert len(set(row.tolist())) == 300 and not (set(row.tolist()) & train), u
    assert torch.equal(i300[:, :100], w_i)


def test_rank_topk_rejects_k_beyond_the_precision(cuda_device):
    from test_gpu_parity import _small_model

    _, model, _, _ = _small_model(cuda_device)
    model.eval()
    for prec, k, serves in (("bf16", 65, "f16"), ("fp32", 129, "f16"), ("f16", 513, None), ("f16", 0, None)):
        with pytest.raises(ValueError, match=prec) as e:
            model.rank_topk([0, 1, 2], k=k, precision=prec)
        assert serves is None or f"'{serves}'" in str(e.value)


def test_ngcf_rank_topk_wide_d128(cuda_device):
    import os

    from spex_b200.ngcf import build_ngcf_norm_adj
    from test_ngcf_golden import GOLD, _model

    G = dict(np.load(os.path.join(GOLD, "ngcf_epinion2.npz")))
    d = np.load(os.path.join(GOLD, "epinion2_data.npz"))
    graph = build_ngcf_norm_adj(d["train_user"], d["train_item"], int(G["n_users"]), int(G["n_items"]))
    model = _model(G, graph, cuda_device)
    model.eval()
    from spex_b200 import ops

    users = torch.arange(0, 700, device=cuda_device)
    i_w, v_w = model.rank_topk(users, k=100, probe=False)
    ua, ia = model.propagate()
    assert ua.shape[1] == 128
    # the untrained model's scores are near-ties everywhere: compare on the same fp16 operands
    _, _, umeta = ops.pack_f16(ua, users, ops.TC_USER_MULTIPLE)
    _, _, imeta = ops.pack_f16(ia, None, ops.TC_ITEM_MULTIPLE)
    _check_vs_fp32_on_operands(i_w, v_w, ua.contiguous(), ia.contiguous(), users, umeta, imeta, min_same=0.9)
    with pytest.raises(ValueError, match="fp32"):
        model.rank_topk(users, k=200, precision="fp32")


def test_sharded_evaluator_k100_matches_test_fullrank(cuda_device):
    from spex_b200 import batch_test
    from spex_b200.dist import ShardedEvaluator
    from spex_b200.graph import build_interaction_csr
    from test_gpu_parity import _small_model

    ds, model, _, _ = _small_model(cuda_device)
    model.eval()
    users = np.arange(ds.n_users)
    au, ai = model.computer()
    mrp, mcol = model.train_mask_csr()
    ev = ShardedEvaluator(au, ai, mrp, mcol, k=100, scorer="f16")
    assert ev.world == 1 and ev.scorer == "f16"
    truth = {int(u): list(ds.testRatings[u]) for u in users if u in ds.testRatings}
    tu = np.array([u for u in users for _ in truth.get(int(u), [])], np.int64)
    ti = np.array([i for u in users for i in truth.get(int(u), [])], np.int64)
    trp, tcol = build_interaction_csr(tu, ti, ds.n_users, ds.m_items)
    idx, _, _ = ev.rank_topk(torch.from_numpy(users).to(cuda_device))
    i_ref, _ = model.rank_topk(users, k=100)
    assert torch.equal(idx, i_ref)
    got = ev.evaluate(torch.from_numpy(users).to(cuda_device), trp, tcol, [100])
    ref = batch_test.test_fullrank(model, users, truth, k=100, precision="f16")
    assert got["users"] == ds.n_users
    assert abs(got["recall"][0] - ref["recall"]) < 1e-12 and abs(got["ndcg"][0] - ref["ndcg"]) < 1e-12, (got, ref)
