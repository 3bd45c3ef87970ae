"""The three full-ranking scorers at the edges of their contract, against one exact float64 top-k.

spex_score_topk_f32 (fp32 CUDA cores), spex_score_topk_bf16 (tcgen05, bf16 operands, fp32 accumulators) and
spex_score_topk_f16 (tcgen05 fp16-accumulator filter + exact fp32 re-score) promise the same output: per user the
k best unmasked items, score descending, ties by ascending item id, and -1 / -inf in the slots beyond the user's
unmasked items.

Most inputs are dyadic small-integer tables: integers in [-8, 8] times a power of two.  Every product and partial
sum is then exact in fp32 and the operands are exact in bf16 and in scaled fp16, so every summation order gives the
same bits and each scorer must return the reference exactly: ids, values and the order of the many exact ties
that small integers produce.  The cases cover what random tables never reach: the zero-padded last item tile when
every real score is negative, fewer eligible items than k, the candidate-buffer width switches (k 24/25, 56/57),
one item tile, fewer tiles than pipeline stages, NULL / permuted / duplicated user ids, padded CTAs, the fp16
filter margin at D = 128 and FullRanker's user blocks.
"""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

SENT_IDX, SENT_VAL = 0x5EED, 12345.0     # written into output rows the scorer must not touch


# ---- inputs ------------------------------------------------------------------------------------------------------
def _dyadic(gen, n, D, exp=0, lo=-8, hi=8):
    """fp32 [n, D] of integers in [lo, hi] times 2^exp."""
    return torch.randint(lo, hi + 1, (n, D), generator=gen).float() * (2.0 ** exp)


def _mask_csr(rows_items, n_rows):
    """CSR (int64 rowptr, int32 col, ascending per row) of a {row: item ids} dict."""
    rp = np.zeros(n_rows + 1, np.int64)
    cols = []
    for r in range(n_rows):
        c = np.unique(np.asarray(rows_items.get(r, []), np.int64))
        rp[r + 1] = rp[r] + c.size
        cols.append(c)
    col = np.concatenate(cols).astype(np.int32) if cols else np.zeros(0, np.int32)
    return rp, col


def _random_masks(rng, n_rows, m, max_per_row=6, boundary=True):
    """A few random masked items per row; some rows also mask the ids on both sides of 16- and 128-column
    boundaries (15/16, 127/128, 255/256) that exist in [0, m)."""
    out = {}
    for r in range(n_rows):
        ids = list(rng.integers(0, max(m, 1), rng.integers(0, max_per_row + 1)))
        if boundary and r % 3 == 0:
            ids += [i for i in (15, 16, 127, 128, 255, 256) if i < m]
        out[r] = [i for i in ids if i < m]
    return out


# ---- the reference -----------------------------------------------------------------------------------------------
def _reference(scores, masked, k):
    """Exact top-k of float64 scores [B, m]: masked items removed, score descending, ties by ascending item id
    (a stable sort on -score), then -1 / -inf up to k.  masked[b] = the item ids excluded for row b."""
    s = np.asarray(scores.numpy() if torch.is_tensor(scores) else scores, np.float64) + 0.0   # no -0.0
    B, m = s.shape
    idx = np.full((B, k), -1, np.int32)
    val = np.full((B, k), -np.inf, np.float32)
    for b in range(B):
        keep = np.ones(m, bool)
        keep[np.asarray(masked[b], np.int64)] = False
        ids = np.nonzero(keep)[0]
        order = ids[np.argsort(-s[b, ids], kind="stable")][:k]
        idx[b, : order.size] = order
        val[b, : order.size] = s[b, order]
    return idx, val


def _assert_exact(idx, val, ref, what):
    ri, rv = ref
    idx, val = idx.cpu().numpy(), val.cpu().numpy()
    assert idx.shape == ri.shape, what
    bad = np.nonzero((idx != ri).any(axis=1) | ~(val == rv).all(axis=1))[0]
    assert bad.size == 0, (what, int(bad[0]), idx[bad[0]].tolist(), ri[bad[0]].tolist(), val[bad[0]].tolist(),
                           rv[bad[0]].tolist())


# ---- the scorers -------------------------------------------------------------------------------------------------
def _pack(kind, src, rows, n_pad, D):
    """spex_pack_bf16 / spex_pack_f16 with an explicit n_pad: (packed, meta or None)."""
    from spex_b200._capi import call, ptr, stream_ptr

    n = src.shape[0] if rows is None else rows.numel()
    if kind == "bf16":
        out = torch.empty(n_pad * D, dtype=torch.bfloat16, device=src.device)
        call("spex_pack_bf16", ptr(src), ptr(rows), n, n_pad, D, ptr(out), stream_ptr())
        return out, None
    out = torch.empty(n_pad * D, dtype=torch.float16, device=src.device)
    meta = torch.empty(4, dtype=torch.float32, device=src.device)
    call("spex_pack_f16", ptr(src), ptr(rows), n, n_pad, D, ptr(out), ptr(meta), stream_ptr())
    return out, meta


def _operands(x, meta):
    """float64 values of packed fp16 operands: fp16(x * scale) / scale, scale from the pack's own meta."""
    sc = float(meta[0])
    return (x.float() * sc).half().double() / sc


def _round_up(n, q):
    return (n + q - 1) // q * q


def _score(kind, U, I, users, k, masks=None, pass_ids=True, extra_cta=False, dev=None):
    """Run one scorer on host tables U [n_u, D], I [m, D] for the rows users (int64 [B]) with the mask
    {mask row: items} (None: mask pointers NULL).  Mask row of output row b: users[b], or b when pass_ids is
    False (user_ids NULL; fp32 always passes users).  tc scorers: B_pad is the next multiple of 128 (plus one
    CTA with extra_cta) and the output rows [B, B_pad) hold a sentinel that must survive.
    Returns (idx, val, reference)."""
    from spex_b200 import ops

    B, D, m = users.numel(), U.shape[1], I.shape[0]
    Ud, Id, ud = U.to(dev), I.to(dev), users.to(dev)
    rp = col = None
    if masks is not None:
        rp_h, col_h = _mask_csr(masks, U.shape[0])
        rp, col = torch.from_numpy(rp_h).to(dev), torch.from_numpy(col_h).to(dev)
    mask_rows = users.numpy() if (pass_ids or kind == "fp32") else np.arange(B)
    masked = [masks.get(int(r), []) if masks is not None else [] for r in mask_rows]
    if kind == "fp32":
        idx, val = ops.score_topk_f32(Ud, Id, ud, k, rp, col)
        torch.cuda.synchronize()
        return idx, val, _reference(U[users].double() @ I.double().t(), masked, k)
    b_pad = _round_up(B, 128) + (128 if extra_cta else 0)
    m_pad = _round_up(m, 128)
    out_i = torch.full((b_pad, k), SENT_IDX, dtype=torch.int32, device=dev)
    out_v = torch.full((b_pad, k), SENT_VAL, dtype=torch.float32, device=dev)
    ids = ud if pass_ids else None
    if kind == "bf16":
        Ub, _ = _pack("bf16", Ud, ud, b_pad, D)
        Ib, _ = _pack("bf16", Id, None, m_pad, D)
        ops.score_topk_bf16(Ub, B, b_pad, Ib, m, m_pad, k, ids, rp, col, out_i, out_v)
        scores = U[users].bfloat16().double() @ I.bfloat16().double().t()
    else:
        Uh, umeta = _pack("f16", Ud, ud, b_pad, D)
        Ih, imeta = _pack("f16", Id, None, m_pad, D)
        ops.score_topk_f16(Uh, umeta, B, b_pad, Ih, imeta, m, m_pad, D, k, ids, rp, col, out_i, out_v)
        scores = _operands(U[users], umeta.cpu()) @ _operands(I, imeta.cpu()).t()
    torch.cuda.synchronize()
    assert bool((out_i[B:] == SENT_IDX).all()) and bool((out_v[B:] == SENT_VAL).all()), \
        f"{kind}: a padded user row wrote output"
    return out_i[:B], out_v[:B], _reference(scores, masked, k)


# (scorer, D) of the tensor-core paths
TC = [("bf16", 64), ("f16", 64), ("f16", 128)]


# ---- 1. shapes x k -----------------------------------------------------------------------------------------------
# m_items: partial 16-column block, exact tile, one tile (one TMEM buffer used), fewer tiles than stages (3-4),
# exact multiples of 128 (no padding), and 901 = 128 * (4 + 3) + 5 tiles for the ring / accumulator phases to wrap
SHAPES = [(1, 1), (1, 64), (15, 24), (15, 25), (16, 56), (16, 57), (17, 64), (17, 1), (127, 57), (128, 24),
          (128, 64), (129, 25), (129, 56), (256, 1), (256, 57), (257, 24), (257, 64), (901, 25), (901, 56),
          (901, 64), (901, 1)]


@pytest.mark.parametrize("m,k", SHAPES)
def test_shapes_and_buffer_widths_bit_exact(cuda_device, m, k):
    gen = torch.Generator().manual_seed(1000 + 7 * m + k)
    rng = np.random.default_rng(m * 100 + k)
    n_u = 200
    users = torch.randperm(n_u, generator=gen)[:129]          # two CTAs, the second with one real row
    masks = _random_masks(rng, n_u, m)
    for kind, D in TC + [("fp32", 64)]:
        U, I = _dyadic(gen, n_u, D, exp=-3), _dyadic(gen, m, D, exp=2)
        idx, val, ref = _score(kind, U, I, users, k, masks, dev=cuda_device)
        _assert_exact(idx, val, ref, (kind, D, m, k))


@pytest.mark.parametrize("m,k", [(901, 24), (901, 25), (257, 56), (901, 57), (901, 64)])
def test_exact_ties_across_tiles(cuda_device, m, k):
    """Every item row is one of five vectors, so each score ties with ~m/5 items spread over every tile: the
    top-k is the lowest ids of the best classes, on every row."""
    gen = torch.Generator().manual_seed(m + k)
    rng = np.random.default_rng(k)
    n_u = 140
    users = torch.arange(n_u)
    masks = _random_masks(rng, n_u, m, max_per_row=20)
    for kind, D in TC + [("fp32", 64)]:
        U = _dyadic(gen, n_u, D, exp=-1)
        I = _dyadic(gen, 5, D, exp=0)[torch.randint(0, 5, (m,), generator=gen)]
        idx, val, ref = _score(kind, U, I, users, k, masks, dev=cuda_device)
        _assert_exact(idx, val, ref, (kind, D, m, k))


# ---- all-negative scores: the padded items (score 0) would win if any padding check failed -----------------------
@pytest.mark.parametrize("m,k,n_masked", [(1, 1, 0), (5, 25, 2), (17, 24, 0), (129, 57, 100), (129, 64, 0),
                                          (300, 64, 250), (901, 57, 870)])
def test_all_negative_scores_never_return_padding(cuda_device, m, k, n_masked):
    gen = torch.Generator().manual_seed(m * k + 3)
    rng = np.random.default_rng(m + n_masked)
    n_u = 130
    users = torch.arange(n_u)
    masks = {r: list(rng.permutation(m)[: n_masked - (r % 3)]) for r in range(n_u)} if n_masked else None
    for kind, D in TC + [("fp32", 64)]:
        U = _dyadic(gen, n_u, D, exp=-2, lo=1, hi=8)            # positive users, negative items:
        I = _dyadic(gen, m, D, exp=1, lo=-8, hi=-1)             # every real score < 0 = a padded item's score
        idx, val, ref = _score(kind, U, I, users, k, masks, dev=cuda_device)
        ids = idx.cpu().numpy()
        assert ids.max() < m, (kind, D, "a zero-padded item was returned")
        n_valid = (ref[0] >= 0).sum(axis=1)
        for b in range(n_u):                                    # the tail: exactly -1 / -inf
            assert (ids[b, n_valid[b]:] == -1).all() and np.isneginf(val.cpu().numpy()[b, n_valid[b]:]).all()
        _assert_exact(idx, val, ref, (kind, D, m, k))


# ---- masks -------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("m,k", [(257, 25), (901, 64), (901, 1)])
def test_mask_edges(cuda_device, m, k):
    gen = torch.Generator().manual_seed(m + 11 * k)
    rng = np.random.default_rng(m)
    n_u = 160
    users = torch.randperm(n_u, generator=gen)
    masks = _random_masks(rng, n_u, m)
    masks[int(users[0])] = []                                   # empty mask row
    masks[int(users[1])] = list(range(m))                       # every item masked: the whole row is -1
    masks[int(users[2])] = [15, 16, 127, 128, 255, 256]
    masks[int(users[3])] = list(rng.permutation(m)[: min(m - 3, 300)])   # more masked items than one tile
    masks[int(users[4])] = list(range(m - k + 1))               # fewer eligible items than k
    for kind, D in TC + [("fp32", 64)]:
        U, I = _dyadic(gen, n_u, D, exp=0), _dyadic(gen, m, D, exp=-4)
        idx, val, ref = _score(kind, U, I, users, k, masks, dev=cuda_device)
        assert (idx[1].cpu() == -1).all() and torch.isneginf(val[1].cpu()).all()
        _assert_exact(idx, val, ref, (kind, D, m, k))
        idx, val, ref = _score(kind, U, I, users, k, None, dev=cuda_device)     # mask_rowptr == NULL
        _assert_exact(idx, val, ref, (kind, D, m, k, "no mask"))


# ---- users -------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("B,ids,extra_cta", [(1, "none", False), (1, "perm", True), (127, "dup", False),
                                             (128, "none", True), (128, "perm", False), (129, "dup", True),
                                             (129, "none", False)])
def test_user_ids_and_padded_ctas(cuda_device, B, ids, extra_cta):
    gen = torch.Generator().manual_seed(B + len(ids))
    rng = np.random.default_rng(B)
    n_u, m, k = 300, 301, 25
    if ids == "none":
        users = torch.arange(B)
    elif ids == "perm":
        users = torch.randperm(n_u, generator=gen)[:B]
    else:
        users = torch.randint(0, 40, (B,), generator=gen)       # duplicates
    masks = _random_masks(rng, n_u, m, max_per_row=30)
    for kind, D in TC + [("fp32", 64)]:
        U, I = _dyadic(gen, n_u, D, exp=3), _dyadic(gen, m, D, exp=-2)
        idx, val, ref = _score(kind, U, I, users, k, masks, pass_ids=(ids != "none"), extra_cta=extra_cta,
                               dev=cuda_device)
        _assert_exact(idx, val, ref, (kind, D, B, ids))
        if ids == "dup":                                        # the same user gives the same row
            first = {int(u): b for b, u in reversed(list(enumerate(users.tolist())))}
            for b, u in enumerate(users.tolist()):
                assert torch.equal(idx[b], idx[first[u]])


# ---- fp32 scorer: D and k up to its limits -----------------------------------------------------------------------
@pytest.mark.parametrize("D,k,m", [(4, 1, 5), (4, 128, 300), (20, 127, 100), (20, 64, 1000), (132, 64, 129),
                                   (132, 128, 257), (512, 1, 257), (512, 128, 1000)])
def test_fp32_dims_and_large_k(cuda_device, D, k, m):
    gen = torch.Generator().manual_seed(D * k + m)
    rng = np.random.default_rng(D)
    n_u = 45                                                    # 21 users: 3 CTAs of 8, the last one partial
    users = torch.randperm(n_u, generator=gen)[:21]
    masks = _random_masks(rng, n_u, m, max_per_row=40)
    U, I = _dyadic(gen, n_u, D, exp=-1), _dyadic(gen, m, D, exp=-1)
    idx, val, ref = _score("fp32", U, I, users, k, masks, dev=cuda_device)
    _assert_exact(idx, val, ref, (D, k, m))


# ---- determinism and argument checks -----------------------------------------------------------------------------
def test_rerun_gives_the_same_bits(cuda_device):
    """Random (not dyadic) tables: near-ties go through the compaction paths; a second call returns the same
    bits."""
    gen = torch.Generator().manual_seed(5)
    users = torch.randperm(300, generator=gen)[:257]
    masks = _random_masks(np.random.default_rng(5), 300, 3000, max_per_row=20)
    for kind, D in TC + [("fp32", 64)]:
        U, I = torch.randn(300, D, generator=gen), torch.randn(3000, D, generator=gen)
        I[::3] = I[1::3][: I[::3].shape[0]]                     # duplicated rows: exact ties
        runs = [_score(kind, U, I, users, 57, masks, dev=cuda_device)[:2] for _ in range(2)]
        (i0, v0), (i1, v1) = runs
        assert torch.equal(i0, i1) and torch.equal(v0.view(torch.int32), v1.view(torch.int32)), kind


def test_contract_rejections_launch_nothing(cuda_device):
    """Each rejected call returns its documented code from the argument check alone: no kernel is launched."""
    import ctypes as C

    from spex_b200 import _capi
    from spex_b200._capi import ptr

    dev = cuda_device
    buf = torch.zeros(1 << 16, dtype=torch.float32, device=dev)
    p = ptr(buf)
    users = torch.arange(128, device=dev)
    rp = torch.zeros(129, dtype=torch.int64, device=dev)
    col = torch.zeros(1, dtype=torch.int32, device=dev)
    BADARG, BADDIM, TOOBIG = -1, -2, -5
    lib, s = _capi.lib, C.c_void_p(torch.cuda.current_stream().cuda_stream)

    def f16(D=64, B_pad=128, m_pad=128, k=20, rpp=None, colp=None):
        return lib.spex_score_topk_f16(p, p, D, 128, B_pad, 128, m_pad, p, p, ptr(users), rpp, colp, k, p, p, s)

    def bf16(B_pad=128, m_pad=128, k=20, rpp=None, colp=None):
        return lib.spex_score_topk_bf16(p, p, 128, B_pad, 128, m_pad, ptr(users), rpp, colp, k, p, p, s)

    def f32(D=64, k=20, rpp=None, colp=None):
        return lib.spex_score_topk_f32(p, p, D, ptr(users), 128, 128, rpp, colp, k, p, p, s)

    before = _capi.launch_count()
    cases = [
        (f16(k=0), TOOBIG), (f16(k=65), TOOBIG), (f16(B_pad=192), BADARG), (f16(m_pad=130), BADARG),
        (f16(rpp=ptr(rp)), BADARG), (f16(colp=ptr(col)), BADARG), (f16(D=32), BADDIM), (f16(D=96), BADDIM),
        (f16(D=256), BADDIM),
        (bf16(k=0), TOOBIG), (bf16(k=65), TOOBIG), (bf16(B_pad=130), BADARG), (bf16(m_pad=200), BADARG),
        (bf16(rpp=ptr(rp)), BADARG), (bf16(colp=ptr(col)), BADARG),
        (f32(k=0), TOOBIG), (f32(k=129), TOOBIG), (f32(rpp=ptr(rp)), BADARG), (f32(colp=ptr(col)), BADARG),
        (f32(D=6), BADDIM), (f32(D=516), BADDIM),
    ]
    assert [c[0] for c in cases] == [c[1] for c in cases]
    assert _capi.launch_count() == before
    oi = torch.empty(128, 128, dtype=torch.int32, device=dev)
    ov = torch.empty(128, 128, dtype=torch.float32, device=dev)
    rc = lib.spex_score_topk_f32(p, p, 64, ptr(users), 128, 128, None, None, 128, ptr(oi), ptr(ov), s)
    assert rc == 0 and _capi.launch_count() == before + 1               # the valid call does launch
    torch.cuda.synchronize()


# ---- 3. pack kernels, decoded on the host ------------------------------------------------------------------------
def _decode(packed, n_pad, D):
    """Inverse of the layout of include/spex_b200.h: element (r, k) at (r/8)*(8*D) + (k/8)*64 + (r%8)*8 + k%8
    (in 16-bit elements)."""
    return packed.view(n_pad // 8, D // 8, 8, 8).permute(0, 2, 1, 3).reshape(n_pad, D)


@pytest.mark.parametrize("D", [8, 64, 128])
@pytest.mark.parametrize("gather", [False, True])
def test_pack_layouts_decode_to_rounded_inputs(cuda_device, D, gather):
    gen = torch.Generator().manual_seed(D + gather)
    n_src = 77
    x = torch.randn(n_src, D, generator=gen) * torch.exp2(torch.randint(-20, 20, (n_src, 1), generator=gen).float())
    x[3, : D // 2] = 0.0
    rows = torch.randint(0, n_src, (51,), generator=gen) if gather else None
    src = x[rows] if gather else x
    n = src.shape[0]
    n_pad = _round_up(n, 8) + 16                                # two all-padding row groups
    xd = x.to(cuda_device)
    rd = rows.to(cuda_device) if gather else None
    pb, _ = _pack("bf16", xd, rd, n_pad, D)
    ph, meta = _pack("f16", xd, rd, n_pad, D)
    torch.cuda.synchronize()
    gb = _decode(pb.cpu().view(torch.int16), n_pad, D)
    gh = _decode(ph.cpu().view(torch.int16), n_pad, D)
    assert torch.equal(gb[:n], src.bfloat16().view(torch.int16))
    sc = float(meta.cpu()[0])
    assert torch.equal(gh[:n], (src * sc).half().view(torch.int16))
    assert not gb[n:].any() and not gh[n:].any()                # padding rows are zero


def _check_meta(meta, x):
    """scale a power of two, 1/scale exact, max scaled norm in [2^6, 2^7) (the largest such scale), max norm^2."""
    sc, inv, vmax, n2 = (float(v) for v in meta)
    n2_ref = float((x.double() ** 2).sum(1).max())
    if n2_ref == 0.0:
        assert (sc, inv, vmax, n2) == (1.0, 1.0, 0.0, 0.0)
        return
    assert sc == 2.0 ** round(np.log2(sc)) and inv * sc == 1.0
    assert abs(n2 - n2_ref) <= 1e-5 * n2_ref
    assert 64.0 <= vmax < 128.0 and abs(vmax - np.sqrt(n2) * sc * 1.0001) <= 1e-5 * vmax


@pytest.mark.parametrize("D", [64, 128])
@pytest.mark.parametrize("case", ["tiny", "huge", "zero", "one_huge_row"])
def test_f16_scale_meta_and_ranking(cuda_device, D, case):
    """pack_f16's meta on tables of norm ~1e-4, ~1e4, all zero and with one row 2^27 larger than the rest (whose
    components then scale to fp16 subnormals and lose bits), and the f16 ranking against the float64 top-k of its own operands."""
    gen = torch.Generator().manual_seed(D + len(case))
    rng = np.random.default_rng(D)
    n_u, m, k = 140, 300, 25
    U, I = _dyadic(gen, n_u, D, exp=0), _dyadic(gen, m, D, exp=0)
    if case == "tiny":
        U, I = U * 2.0 ** -17, I * 2.0 ** -16
    elif case == "huge":
        U, I = U * 2.0 ** 10, I * 2.0 ** 11
    elif case == "zero":
        U = torch.zeros(n_u, D)
    else:                                                       # scale ~2^-26: the other rows' odd multiples
        U[7] = U[7] * 2.0 ** 27                                 # of 2^-26 round to multiples of 2^-24
    users = torch.arange(n_u)
    masks = _random_masks(rng, n_u, m)
    _, umeta = _pack("f16", U.to(cuda_device), users.to(cuda_device), 256, D)
    _check_meta(umeta.cpu(), U)
    if case == "one_huge_row":                                  # the other rows really lose bits to subnormals
        uop = _operands(U, umeta.cpu())
        assert bool((uop[:7] != U[:7].double()).any())
        assert bool(((U * float(umeta[0])).abs()[:7] < 2.0 ** -14).any())
    idx, val, ref = _score("f16", U, I, users, k, masks, dev=cuda_device)
    _assert_exact(idx, val, ref, (D, case))
    if case == "zero":                                          # every score 0: ids 0.. in order, minus the masked
        for b in range(n_u):
            keep = [i for i in range(m) if i not in set(masks[b])][:k]
            assert idx[b].tolist() == keep


# ---- 4. the fp16 filter margin at D = 128 ------------------------------------------------------------------------
def _f16_round(x, toward_zero):
    h = np.float16(x)
    if toward_zero and abs(float(h)) > abs(x):
        h = np.nextafter(h, np.float16(0.0))
    return float(h)


def _f16_round_down(x):
    h = np.float16(x)
    return float(np.nextafter(h, np.float16(-np.inf)) if float(h) > x else h)


def _emulated_f16_acc(u, v, toward_zero):
    """A pessimistic fp16 accumulator: the partial sum rounded to fp16 after every K = 16 MMA step (the exact
    16-term sum of a step is added first)."""
    acc = 0.0
    for d in range(0, u.size, 16):
        acc = _f16_round(acc + float(np.dot(u[d: d + 16], v[d: d + 16])), toward_zero)
    return acc


@pytest.mark.parametrize("D", [64, 128])
@pytest.mark.parametrize("k", [10, 50])
def test_f16_filter_margin_adversarial(cuda_device, D, k):
    """Items whose fp16-accumulated score loses as much as the per-K-step rounding model allows, placed just above
    the k-th exact score with decoys just below it.

    User u = (1 x16, 2^-6 ...).  An adversarial item's first K step sums to 16 + 7*2^-10 (rounds down to 16) and
    each later step adds 15*2^-11, just under half an ulp of 16, which rounds away too: after D/16 steps the fp16
    accumulator still reads 16 while the exact score is 16 + (15 D/16 - 1) 2^-11, an error of about
    (D/16 - 0.6) 2^-11 |u| Vmax.  200 decoys, exactly summed in one K step to just below the adversarial score,
    come first in id order; they fill the candidate buffer, so the filter threshold - (exact k-th score - eps),
    rounded down to fp16 - rises before the adversarial items arrive.  With a margin of 2^-9 at D = 128 that
    threshold is above 16 and every adversarial item would be dropped; the result must be the exact top-k: the
    first k adversarial items."""
    nb = D // 16
    u = np.full(D, 2.0 ** -6)
    u[:16] = 1.0
    adv = np.full(D, 15 * 2.0 ** -9)
    adv[:16] = 1.0
    adv[14] = 1.0 + 7 * 2.0 ** -10
    s_adv = float(u @ adv)
    q = int(np.ceil((s_adv - 16.0) * 1024)) - 1                 # decoy score 16 + q 2^-10, just below s_adv
    dec = np.zeros(D)
    dec[:16] = 1.0 + (q // 16) * 2.0 ** -10
    dec[: q % 16] += 2.0 ** -10
    s_dec = float(u @ dec)
    assert s_dec == 16.0 + q * 2.0 ** -10 and s_adv - 2.0 ** -9 < s_dec < s_adv
    uv = np.linalg.norm(u) * max(np.linalg.norm(adv), np.linalg.norm(dec))     # |u| Vmax
    for tz in (False, True):                                    # the construction under both rounding variants
        a = _emulated_f16_acc(u, adv, tz)
        rel = (s_adv - a) / uv
        assert a == 16.0 and (nb - 1) * 2.0 ** -11 < rel < nb * 2.0 ** -11, (tz, rel)
        # the filter threshold after the decoys, for a margin of (DK/16) 2^-11 and of 2^-9
        assert _f16_round_down(s_dec - nb * 2.0 ** -11 * uv * 1.0001) <= a
        assert (_f16_round_down(s_dec - 2.0 ** -9 * uv * 1.0001) > a) == (D == 128)
    m, n_dec, n_adv = 128 * 8 + 37, 200, 50
    I = np.zeros((m, D))
    I[:, :16] = -1.0                                            # fillers: score -16
    I[:n_dec] = dec
    adv_ids = 400 + 12 * np.arange(n_adv)                       # spread over later tiles
    I[adv_ids] = adv
    n_u = 130
    U = np.tile(u, (n_u, 1)) * (2.0 ** -(np.arange(n_u) % 3))[:, None]
    U, I = torch.from_numpy(U).float(), torch.from_numpy(I).float()
    idx, val, ref = _score("f16", U, I, torch.arange(n_u), k, dev=cuda_device)
    assert (ref[0] == adv_ids[:k]).all()                        # the operands are exact: adversarial items win
    _assert_exact(idx, val, ref, (D, k))


# ---- 5. FullRanker does not depend on user_block ------------------------------------------------------------------
@pytest.mark.parametrize("D", [64, 128])
def test_full_ranker_f16_independent_of_user_block(cuda_device, D):
    """Users whose row norms span 2^12, largest first: packed per block of 128, the later blocks would get a larger
    user scale than the call as a whole, so their small components would round differently (subnormal or not).
    The user scale belongs to the call: None, 256 and 128 give the same bits, and each row is the exact top-k of
    the operands packed for the whole call."""
    from spex_b200 import ops

    gen = torch.Generator().manual_seed(D)
    rng = np.random.default_rng(D)
    n_u, m, k = 400, 1000, 20
    U = torch.randn(n_u, D, generator=gen) * torch.exp2(-12.0 * torch.arange(n_u).float() / n_u)[:, None]
    I = _dyadic(gen, m, D, exp=-3)
    users = torch.randperm(n_u, generator=gen)[:330].sort().values     # kept in norm order: blocks differ in scale
    masks = _random_masks(rng, n_u, m, max_per_row=10)
    rp_h, col_h = _mask_csr(masks, n_u)
    dev = cuda_device
    rp, col = torch.from_numpy(rp_h).to(dev), torch.from_numpy(col_h).to(dev)
    ranker = ops.FullRanker(I.to(dev), "f16")
    got = {}
    for block in (None, 256, 128):
        got[block] = ranker.topk(U.to(dev), users.to(dev), k, rp, col, user_block=block)
    torch.cuda.synchronize()
    # the test has teeth: a per-block scale changes some operands of the later blocks
    _, meta_all = _pack("f16", U.to(dev), users.to(dev), 384, D)
    _, meta_blk = _pack("f16", U.to(dev), users[256:].to(dev), 128, D)
    assert float(meta_blk[0]) > float(meta_all[0])
    assert bool((_operands(U[users[256:]], meta_all.cpu()) != _operands(U[users[256:]], meta_blk.cpu())).any())
    for block in (256, 128):
        assert torch.equal(got[block][0], got[None][0]), block
        assert torch.equal(got[block][1].view(torch.int32), got[None][1].view(torch.int32)), block
    # exact top-k of the call's operands: ids identical wherever the float64 ranking has no near-tie at rank k,
    # values to fp32 rounding of a 64-128-term sum
    uop, iop = _operands(U[users], meta_all.cpu()), _operands(I, ranker._imeta.cpu())
    scores = (uop @ iop.t()).numpy()
    ri, rv = _reference(scores, [masks[int(u)] for u in users], k)
    idx, val = got[None][0].cpu().numpy(), got[None][1].cpu().numpy()
    tol = 2 * D * 2.0 ** -24 * (uop.norm(dim=1) * iop.norm(dim=1).max()).numpy()[:, None]
    assert (np.abs(val - rv) <= tol).all()
    same = (idx == ri).all(axis=1)
    # rows that differ must differ only by a swap of scores within the tolerance
    for b in np.nonzero(~same)[0]:
        assert np.abs(scores[b, idx[b]] - scores[b, ri[b]]).max() <= tol[b, 0], b
    assert same.mean() > 0.9
