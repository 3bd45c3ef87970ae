"""The training-step kernels of csrc/loss.cu at the edges of their contract, against float64 references.

Covered entry points: the gather -> dot -> loss forwards (spex_bce_fwd_f32, spex_bpr_fwd_f32 and ops.gather_dot /
bce_loss / bpr_loss), the deterministic scatter backward (spex_bce_bwd_ws_f32, spex_bpr_bwd_ws_f32,
spex_scatter_rows_f32) in its scan and sorted forms, spex_clear_rows_f32, spex_gather_owned_rows_f32, dense Adam
(spex_adam_f32), the expert gate and its backward, candidate scoring and ops.rating_dense.

Most inputs are dyadic small-integer tables: integers in [-8, 8] times a power of two.  Every product and every
partial sum below is then a multiple of a fixed power of two and smaller than 2^24 of those units, so it is exact in
fp32: every summation order gives the same bits, and gathers, dots and scatters must equal the float64 reference
exactly (torch.equal / np.array_equal).  Tolerances appear only where a transcendental or a division is involved,
each as a bound in ulps (u = 2^-24, the unit roundoff, is half an ulp of a value in [1, 2)):
  * sigmoid 1/(1 + expf(-x)): expf is within 2 ulp, the add and the IEEE division add 0.5 ulp each, so a weight in
    [0, 1] is within 4u of the true value; (sigma - y)/B then adds one rounding of the difference and one of the
    division by B.  Where sigma(x) is below the fp32 normal range (x < -87) expf overflows and the kernel returns 0:
    the absolute bound covers that;
  * softplus max(x, 0) + log1pf(expf(-|x|)): 4 ulps of the result (expf 2, log1pf 1, the add 0.5), or 2^-126
    absolute where the result is subnormal;
  * a mean over B terms, summed per thread in a stride of 1024 and then by a 1024-wide tree: the classical
    bound (n + 16) u sum|term| with n = ceil(B/1024) + 10 sequential additions, plus 6u per term for the
    transcendentals, plus one ulp for the division by B;
  * Adam: the moments to 2 ulps of their largest intermediate, the parameter to 1 ulp plus 4 ulps of the update
    (sqrt, the division by sqrt(1 - b2^t), + eps, m/denom, the fp32 step size and its product);
  * the expert gate: softmax weights to 8u relative, the backward's dz to 32u of |da0| + |da1|, dW to the
    fixed-order summation bound over its (rows per warp + 8 warps + CTAs) sequential additions.

The scatter cases cover what random batches do not reach: the NV = 4 instantiations (D > 128) and D with only some
lanes active (4, 20, 100, 132), the switch between the O(n^2/32) duplicate scan (up to 2048 list entries, and up to
2^18 without a workspace) and the radix-sorted form, rows whose first occurrence sits at list position 31, 32 or 33
(the 32-entry ballot chunks of the scan), one row filling the whole list, rows that only the second BPR segment
touches, alternating rows, the row window of spex_scatter_rows_f32, gscalar = NULL and cconst != 1.  Rows that no
entry targets hold a sentinel that must survive.  The refusals (workspace missing, short or misaligned; D = 0, 6, 516)
must launch nothing.  An empty batch gives a NaN loss, as torch.nn.BCEWithLogitsLoss does, and zero gradients.
"""
import ctypes as C
import math

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

SENT = 12345.0                       # written into outputs a kernel must not touch
U_RND = 2.0 ** -24                   # unit roundoff of fp32
E_BADDIM, E_WORKSPACE, E_TOOBIG = -2, -6, -5
DS = [4, 20, 64, 100, 128, 132, 256, 512]
SCATTER_DS = [4, 20, 64, 128, 132, 512]
GRID_FLOAT4 = 148 * 8 * 256          # float4 per pass of the capped grid-stride loops


# ---- helpers -----------------------------------------------------------------------------------------------------
def _capi():
    from spex_b200 import _capi

    return _capi


def _p(t):
    return None if t is None else C.c_void_p(t.data_ptr())


def _st():
    return _capi().stream_ptr()


def _dyadic(rng, shape, exp=0, lo=-8, hi=8):
    """fp32 array of integers in [lo, hi] times 2^exp."""
    return (rng.integers(lo, hi + 1, shape) * (2.0 ** exp)).astype(np.float32)


def _dev(a, dev, dtype=None):
    t = torch.from_numpy(np.ascontiguousarray(a))
    return t.to(device=dev, dtype=dtype) if dtype is not None else t.to(dev)


def _ws(total, dev):
    """(workspace, bytes) of the sorted scatter for `total` list entries; (None, 0) where the scan form runs."""
    nbytes = int(_capi().lib.spex_scatter_workspace_bytes(int(total)))
    if nbytes == 0:
        return None, 0
    return torch.empty(nbytes, dtype=torch.uint8, device=dev), nbytes


def _spacing(ref):
    """fp32 ulp at each |ref| (the subnormal step below the normal range)."""
    return np.spacing(np.abs(np.asarray(ref, np.float64)).astype(np.float32)).astype(np.float64)


def _assert_within(got, ref, tol, what):
    got, ref = np.broadcast_arrays(np.asarray(got, np.float64), np.asarray(ref, np.float64))
    assert np.isfinite(got).all(), (what, "non-finite output")
    err = np.abs(got - ref)
    tol = np.broadcast_to(np.asarray(tol, np.float64), err.shape)
    bad = np.flatnonzero((err > tol).ravel())
    assert bad.size == 0, (what, int(bad[0]), float(got.ravel()[bad[0]]), float(ref.ravel()[bad[0]]),
                           float(tol.ravel()[bad[0]]))


def _rows(pattern, n, n_rows, rng):
    """int64 [n] row ids in [0, n_rows) laid out by `pattern`:
    random; one_row (every entry on the last row); alternating (rows 2 and 5 interleaved); first_at_P (the last
    row first occurs at list position P, again at P + 1 and at some later positions, never before P)."""
    if pattern == "random":
        return rng.integers(0, n_rows, n)
    if pattern == "one_row":
        return np.full(n, n_rows - 1, np.int64)
    if pattern == "alternating":
        return np.where(np.arange(n) % 2 == 0, 2, 5).astype(np.int64)
    p = int(pattern.rsplit("_", 1)[1])
    R = n_rows - 1
    r = rng.integers(0, n_rows - 1, n)
    r[p] = r[p + 1] = R
    rest = np.arange(p + 2, n)
    r[rng.choice(rest, size=max(1, rest.size // 8), replace=False)] = R
    return r


def _scatter_ref(out_init, dst, src_idx, w, src):
    """float64 reference of the scatter: out[r] = sum over entries t with dst[t] == r of w[t] * src[src_idx[t]];
    rows no entry targets keep out_init.  Exact for dyadic weights (any order)."""
    out = np.asarray(out_init, np.float64).copy()
    out[np.unique(dst)] = 0.0
    np.add.at(out, dst, np.asarray(w, np.float64)[:, None] * np.asarray(src, np.float64)[src_idx])
    return out


def _fma_chain_ref(out_init, dst, src_idx, w32, src):
    """The scatter's contract for a non-dyadic fp32 weight: per row, acc = fma(w[t], src[src_idx[t]], acc) in
    ascending list position t, each step exact in float64 (a 24-bit weight times a small integer plus an fp32
    partial sum fits in 53 bits) and rounded once to fp32, exactly like fmaf."""
    out = np.asarray(out_init, np.float32).copy()
    order = np.argsort(dst, kind="stable")
    ds = dst[order]
    head = np.r_[True, ds[1:] != ds[:-1]]
    run = np.cumsum(head) - 1
    start = np.flatnonzero(head)
    rank = np.arange(order.size) - start[run]
    acc = np.zeros((start.size, out.shape[1]), np.float32)
    src64 = np.asarray(src, np.float64)
    for k in range(int(rank.max()) + 1 if rank.size else 0):
        sel = rank == k
        t, r = order[sel], run[sel]
        acc[r] = (w32[t].astype(np.float64)[:, None] * src64[src_idx[t]] + acc[r].astype(np.float64)).astype(np.float32)
    out[ds[start]] = acc
    return out


# ---- 1. gather -> dot -> BCE -------------------------------------------------------------------------------------
def _bce_batch(rng, D, B, nu=50, m=60):
    """Tables (ints in [-8, 8] / 4) whose first rows give the logits +-20, +-90, +-200 and 0 exactly, and a batch
    that starts with those pairs under labels 0, 1 and 0.3, then random pairs with labels 0, 1 or in (0, 1)."""
    U = _dyadic(rng, (nu, D), -2)
    I = _dyadic(rng, (m, D), -2)
    U[:4] = 0.0
    U[0, 0], U[1, 0], U[2, 0] = 20.0, 90.0, 200.0
    I[:2] = 0.0
    I[0, 0], I[1, 0] = 1.0, -1.0
    special = [(u, i, y) for u in range(4) for i in range(2) for y in (0.0, 1.0, 0.3)]
    users = rng.integers(4, nu, B)
    items = rng.integers(2, m, B)
    kind = rng.integers(0, 3, B)
    labels = np.where(kind == 0, 0.0, np.where(kind == 1, 1.0, rng.random(B))).astype(np.float32)
    for b, (u, i, y) in enumerate(special[:B]):
        users[b], items[b], labels[b] = u, i, y
    return U, I, users, items, labels


def _loss_tol(x64, B, extra_terms=6):
    """Bound of an fp32 mean of B per-sample terms of magnitude <= |x| + 1 (see the module docstring)."""
    n_seq = math.ceil(B / 1024) + 10
    return (n_seq + 16 + extra_terms) * U_RND * float(np.sum(np.abs(x64) + 1.0)) / B


def _check_bce(dev, U, I, users, items, labels):
    from torch.nn.functional import binary_cross_entropy_with_logits as bce

    capi = _capi()
    B, D = users.size, U.shape[1]
    Ud, Id = _dev(U, dev), _dev(I, dev)
    ud, idd, yd = _dev(users, dev), _dev(items, dev), _dev(labels, dev)
    gamma = torch.full((B,), SENT, device=dev)
    dgamma = torch.full((B,), SENT, device=dev)
    loss = torch.full((1,), SENT, device=dev)
    capi.call("spex_bce_fwd_f32", _p(Ud), _p(Id), D, _p(ud), _p(idd), _p(yd), B, _p(gamma), _p(loss), _p(dgamma), _st())
    x64 = (U.astype(np.float64) @ I.astype(np.float64).T)[users, items]       # exact: dyadic
    y64 = labels.astype(np.float64)
    assert np.array_equal(gamma.cpu().numpy(), x64.astype(np.float32)), ("gamma", D, B)
    # dgamma = (sigma(x) - y) / B: 4u for sigma, 0.5 ulp for the difference and one ulp for the division by B
    sig = 1.0 / (1.0 + np.exp(-x64))
    ref_dg = (sig - y64) / B
    _assert_within(dgamma.cpu().numpy(), ref_dg, 6 * U_RND / B + _spacing(ref_dg), ("dgamma", D, B))
    ref_loss = float(bce(torch.from_numpy(x64), torch.from_numpy(y64)))
    tol = _loss_tol(x64, B) + float(_spacing(ref_loss))
    _assert_within(loss.cpu().numpy()[0], ref_loss, tol, ("loss", D, B))
    # gather_dot mode (loss, dgamma, labels NULL): the same gamma bits
    gamma2 = torch.full((B,), SENT, device=dev)
    capi.call("spex_bce_fwd_f32", _p(Ud), _p(Id), D, _p(ud), _p(idd), None, B, _p(gamma2), None, None, _st())
    assert torch.equal(gamma2, gamma)
    return loss, Ud, Id, ud, idd, yd


@pytest.mark.parametrize("B", [1, 7, 8, 9, 1023, 1024, 1025])
@pytest.mark.parametrize("D", DS)
def test_bce_forward_against_float64(cuda_device, D, B):
    """gamma exact, dgamma and the loss within their ulp bounds, at logits up to +-200 (no inf / NaN); ops.bce_loss
    gives the entry point's loss bits."""
    from spex_b200 import ops

    rng = np.random.default_rng(1000 * D + B)
    U, I, users, items, labels = _bce_batch(rng, D, B)
    loss, Ud, Id, ud, idd, yd = _check_bce(cuda_device, U, I, users, items, labels)
    out = torch.cat([Ud, Id])
    got = ops.bce_loss(out, U.shape[0], ud, idd, yd)
    assert torch.equal(got.reshape(1), loss)


def test_bce_forward_large_batch_reduce_strides(cuda_device):
    """A few million samples: every thread of the single-CTA reduce sums ~2900 terms before the tree."""
    rng = np.random.default_rng(7)
    B, D = 3_000_001, 64
    U = _dyadic(rng, (1000, D), -2)
    I = _dyadic(rng, (1000, D), -2)
    users = rng.integers(0, 1000, B)
    items = rng.integers(0, 1000, B)
    labels = np.where(rng.random(B) < 0.5, 0.0, rng.random(B)).astype(np.float32)
    _check_bce(cuda_device, U, I, users, items, labels)


@pytest.mark.parametrize("B", [1000, 5000])
@pytest.mark.parametrize("D", DS)
def test_gather_dot_gradient_against_float64_autograd(cuda_device, D, B):
    """ops.gather_dot and its backward (spex_bce_bwd_ws_f32 with grad_loss NULL; B = 5000 takes the sorted form):
    gamma and d/d(out) of sum(gamma * w) for a dyadic w are exact."""
    from spex_b200 import ops

    rng = np.random.default_rng(D + 7 * B)
    nur, m = 70, 90
    out = _dyadic(rng, (nur + m, D), -1)
    users = rng.integers(0, nur, B)
    items = rng.integers(0, m, B)
    w = _dyadic(rng, (B,), -2, -4, 4)
    o64 = torch.from_numpy(out).double().requires_grad_(True)
    ut, it = torch.from_numpy(users), torch.from_numpy(items)
    g64 = (o64[ut] * o64[nur + it]).sum(1)
    (g64 * torch.from_numpy(w).double()).sum().backward()
    od = _dev(out, cuda_device).requires_grad_(True)
    gamma = ops.gather_dot(od, nur, _dev(users, cuda_device), _dev(items, cuda_device))
    (gamma * _dev(w, cuda_device)).sum().backward()
    assert torch.equal(gamma.detach().cpu(), g64.detach().float())
    assert torch.equal(od.grad.cpu(), o64.grad.float())


# ---- 2. the deterministic scatter --------------------------------------------------------------------------------
def _both_forms(run, total, dev):
    """Run `run(work, work_bytes)` without a workspace (scan form) and with one (sorted form above 2048 entries);
    return both results, whose bits must agree."""
    a = run(None, 0)
    ws, nb = _ws(total, dev)
    if total <= 2048:
        assert ws is None
    else:
        assert ws is not None
    return a, run(ws, nb)


BCE_PATTERNS = ["random", "one_row", "first_at_31", "first_at_32", "first_at_33", "alternating"]


@pytest.mark.parametrize("pattern", BCE_PATTERNS)
@pytest.mark.parametrize("B", [64, 2048, 2049])
@pytest.mark.parametrize("D", SCATTER_DS)
def test_bce_backward_scatter_exact_in_both_forms(cuda_device, D, B, pattern):
    """gU[users] = sum gl * dgamma * I[items], gI[items] = sum gl * dgamma * U[users] for a dyadic dgamma: exact,
    scan == sorted bit for bit, untouched rows keep the sentinel.  grad_loss is NULL on every other pattern."""
    capi = _capi()
    dev = cuda_device
    pi = BCE_PATTERNS.index(pattern)
    rng = np.random.default_rng(pi + 10 * D + 1000 * B)
    nu, m = 300, 400
    U, I = _dyadic(rng, (nu, D)), _dyadic(rng, (m, D))
    users, items = _rows(pattern, B, nu, rng), _rows(pattern, B, m, rng)
    dg = _dyadic(rng, (B,), -3, -4, 4)
    gl = None if pi % 2 else 0.5
    Ud, Id, ud, idd, dgd = (_dev(a, dev) for a in (U, I, users, items, dg))
    gld = None if gl is None else torch.tensor([gl], device=dev)

    def run(ws, nb):
        gU = torch.full((nu, D), SENT, device=dev)
        gI = torch.full((m, D), SENT, device=dev)
        capi.call("spex_bce_bwd_ws_f32", _p(Ud), _p(Id), D, _p(ud), _p(idd), _p(dgd), _p(gld), B, _p(gU), _p(gI),
                  _p(ws), nb, _st())
        return gU.cpu().numpy(), gI.cpu().numpy()

    (su, si), (tu, ti) = _both_forms(run, B, dev)
    w = dg.astype(np.float64) * (1.0 if gl is None else gl)
    ref_u = _scatter_ref(np.full((nu, D), SENT), users, items, w, I)
    ref_i = _scatter_ref(np.full((m, D), SENT), items, users, w, U)
    assert np.array_equal(su, ref_u.astype(np.float32)), ("gU scan", D, B, pattern)
    assert np.array_equal(si, ref_i.astype(np.float32)), ("gI scan", D, B, pattern)
    assert np.array_equal(tu, su) and np.array_equal(ti, si), ("sorted != scan", D, B, pattern)


BPR_PATTERNS = BCE_PATTERNS + ["neg_only"]


@pytest.mark.parametrize("pattern", BPR_PATTERNS)
@pytest.mark.parametrize("B", [64, 1024, 1025])
@pytest.mark.parametrize("D", SCATTER_DS)
def test_bpr_backward_scatter_exact_in_both_forms(cuda_device, D, B, pattern):
    """The four BPR scatters over the 2B-entry lists (pos segment, then neg segment): the propagated tables exact for
    a dyadic dscore and grad2, the ego tables (weight grad2[1] * fl(1/B), not dyadic for B = 1025) equal to the fp32
    FMA chain in ascending list order; scan == sorted bit for bit.  neg_only: the neg items are disjoint from the pos
    items, so their rows first occur in the second segment.  grad2 is NULL on every other pattern."""
    capi = _capi()
    dev = cuda_device
    pi = BPR_PATTERNS.index(pattern)
    rng = np.random.default_rng(pi + 10 * D + 1000 * B + 5)
    nu, m = 300, 400
    U, I, U0, I0 = (_dyadic(rng, (n, D)) for n in (nu, m, nu, m))
    users = _rows("random" if pattern == "neg_only" else pattern, B, nu, rng)
    if pattern == "neg_only":
        pos, neg = rng.integers(0, m // 2, B), rng.integers(m // 2, m, B)
    else:
        pos, neg = _rows(pattern, B, m, rng), _rows(pattern, B, m, rng)
    ds = _dyadic(rng, (B,), -3, -4, 4)
    g2 = None if pi % 2 else np.array([0.5, 0.25], np.float32)
    Ud, Id, U0d, I0d = (_dev(a, dev) for a in (U, I, U0, I0))
    ud, pd, nd, dsd = (_dev(a, dev) for a in (users, pos, neg, ds))
    g2d = None if g2 is None else _dev(g2, dev)

    def run(ws, nb):
        outs = [torch.full((n, D), SENT, device=dev) for n in (nu, m, nu, m)]
        capi.call("spex_bpr_bwd_ws_f32", _p(Ud), _p(Id), _p(U0d), _p(I0d), D, _p(ud), _p(pd), _p(nd), _p(dsd),
                  _p(g2d), B, *[_p(o) for o in outs], _p(ws), nb, _st())
        return [o.cpu().numpy() for o in outs]

    scan, srt = _both_forms(run, 2 * B, dev)
    gl, gr = (1.0, 1.0) if g2 is None else (float(g2[0]), float(g2[1]))
    d = ds.astype(np.float64) * gl
    w2 = np.concatenate([-d, d])
    ref_gu = _scatter_ref(np.full((nu, D), SENT), np.concatenate([users, users]), np.concatenate([pos, neg]), w2, I)
    ref_gi = _scatter_ref(np.full((m, D), SENT), np.concatenate([pos, neg]), np.concatenate([users, users]), w2, U)
    w_ego = np.float32(gr) * (np.float32(1.0) / np.float32(B))      # the kernel's fp32 weight of the reg term
    ref_gu0 = _fma_chain_ref(np.full((nu, D), SENT), users, users, np.full(B, w_ego, np.float32), U0)
    pn = np.concatenate([pos, neg])
    ref_gi0 = _fma_chain_ref(np.full((m, D), SENT), pn, pn, np.full(2 * B, w_ego, np.float32), I0)
    for name, got, ref in zip(("gU", "gI", "gU0", "gI0"), scan, (ref_gu, ref_gi, ref_gu0, ref_gi0)):
        assert np.array_equal(got, np.asarray(ref, np.float32)), (name, D, B, pattern)
    for name, a, b in zip(("gU", "gI", "gU0", "gI0"), scan, srt):
        assert np.array_equal(a, b), ("sorted != scan", name, D, B, pattern)


WINDOW_CASES = [
    # (row_lo, row_hi, gscalar, cconst, coef)
    (100, 250, None, -0.75, True),
    (100, 250, 0.5, 1.0, False),
    (0, 0, 0.25, 2.0, True),            # row_hi == 0: every row
]


@pytest.mark.parametrize("case", range(len(WINDOW_CASES)))
@pytest.mark.parametrize("total", [300, 3000])
@pytest.mark.parametrize("D", [4, 100, 132, 512])
def test_scatter_rows_window_exact(cuda_device, D, total, case):
    """spex_scatter_rows_f32: only destinations in [row_lo, row_hi) are written, at row - row_lo; the output pointer
    is a view into a full-height sentinel table, so a write outside the window would land on a sentinel row.  The
    destinations include row_lo - 1, row_lo, row_hi - 1 and row_hi, with duplicates."""
    capi = _capi()
    dev = cuda_device
    lo, hi, gs, cc, use_coef = WINDOW_CASES[case]
    rng = np.random.default_rng(D + total + 100 * case)
    N, S = 500, 300
    src = _dyadic(rng, (S, D))
    dst = rng.integers(0, N, total)
    edges = [x for x in (lo - 1, lo, hi - 1, hi) if 0 <= x < N]
    dst[: 2 * len(edges)] = np.repeat(edges, 2)
    rng.shuffle(dst)
    src_rows = rng.integers(0, S, total)
    coef = _dyadic(rng, (total,), -2, -4, 4) if use_coef else None
    srcd, dstd, srd = _dev(src, dev), _dev(dst, dev), _dev(src_rows, dev)
    coefd = None if coef is None else _dev(coef, dev)
    gsd = None if gs is None else torch.tensor([gs], device=dev)

    def run(ws, nb):
        full = torch.full((N, D), SENT, device=dev)
        capi.call("spex_scatter_rows_f32", _p(dstd), _p(srd), _p(coefd), _p(gsd), float(cc), total, _p(srcd), D,
                  _p(full[lo]), lo, hi, _p(ws), nb, _st())
        return full.cpu().numpy()

    scan, srt = _both_forms(run, total, dev)
    keep = np.ones(total, bool) if hi == 0 else (dst >= lo) & (dst < hi)
    w = (np.ones(total) if coef is None else coef.astype(np.float64)) * (1.0 if gs is None else gs) * cc
    ref = _scatter_ref(np.full((N, D), SENT), dst[keep], src_rows[keep], w[keep], src)
    assert np.array_equal(scan, ref.astype(np.float32)), (D, total, case)
    assert np.array_equal(srt, scan), (D, total, case)


@pytest.mark.parametrize("D", [8, 132])
def test_scatter_at_the_scan_cap(cuda_device, D):
    """2^18 entries: the largest list the scan form takes without a workspace; exact, and equal to the sorted form."""
    capi = _capi()
    dev = cuda_device
    rng = np.random.default_rng(D)
    total, N, S = 1 << 18, 3000, 500
    src = _dyadic(rng, (S, D))
    dst, src_rows = rng.integers(0, N, total), rng.integers(0, S, total)
    coef = _dyadic(rng, (total,), -1, -2, 2)
    srcd, dstd, srd, coefd = (_dev(a, dev) for a in (src, dst, src_rows, coef))

    def run(ws, nb):
        out = torch.full((N + 1, D), SENT, device=dev)
        capi.call("spex_scatter_rows_f32", _p(dstd), _p(srd), _p(coefd), None, 1.0, total, _p(srcd), D, _p(out), 0, 0,
                  _p(ws), nb, _st())
        return out.cpu().numpy()

    scan, srt = _both_forms(run, total, dev)
    ref = _scatter_ref(np.full((N + 1, D), SENT), dst, src_rows, coef, src)
    assert np.array_equal(scan, ref.astype(np.float32))
    assert np.array_equal(srt, scan)


def _refusal_call(entry, dev, total, D, ws_ptr, nb):
    """Call `entry` on a list of `total` entries with a sentinel output; return (rc, outputs unchanged,
    launches made)."""
    capi = _capi()
    Dt = 8
    rows = torch.zeros(total, dtype=torch.int64, device=dev)
    tab = torch.ones(16, Dt, device=dev)
    outs = [torch.full((16, Dt), SENT, device=dev) for _ in range(4)]
    coef = torch.ones(total, device=dev)
    before = capi.launch_count()
    if entry == "scatter_rows":
        rc = capi.lib.spex_scatter_rows_f32(_p(rows), _p(rows), _p(coef), None, 1.0, total, _p(tab), D, _p(outs[0]),
                                            0, 0, ws_ptr, nb, _st())
    elif entry == "bce_bwd":
        rc = capi.lib.spex_bce_bwd_ws_f32(_p(tab), _p(tab), D, _p(rows), _p(rows), _p(coef), None, total,
                                          _p(outs[0]), _p(outs[1]), ws_ptr, nb, _st())
    else:
        B = total // 2
        rc = capi.lib.spex_bpr_bwd_ws_f32(_p(tab), _p(tab), _p(tab), _p(tab), D, _p(rows), _p(rows), _p(rows),
                                          _p(coef), None, B, *[_p(o) for o in outs], ws_ptr, nb, _st())
    launched = capi.launch_count() - before
    torch.cuda.synchronize()
    same = all(bool((o == SENT).all()) for o in outs)
    return rc, same, launched


@pytest.mark.parametrize("entry", ["scatter_rows", "bce_bwd", "bpr_bwd"])
def test_scatter_refusals_launch_nothing(cuda_device, entry):
    """SPEX_E_WORKSPACE for a list above 2^18 entries without a workspace, a workspace one byte short and a
    misaligned one; SPEX_E_BADDIM for D = 0, 6 and 516.  Each before any launch, outputs untouched."""
    dev = cuda_device
    big = (1 << 18) + 2                       # list entries: BPR takes B = 2^17 + 1, i.e. 2B of them
    assert _refusal_call(entry, dev, big, 8, None, 0) == (E_WORKSPACE, True, 0)
    total = 3000
    nbytes = int(_capi().lib.spex_scatter_workspace_bytes(total))
    assert nbytes > 0 and int(_capi().lib.spex_scatter_workspace_bytes(2048)) == 0
    buf = torch.empty(nbytes + 64, dtype=torch.uint8, device=dev)
    base = buf.data_ptr()
    assert base % 16 == 0
    assert _refusal_call(entry, dev, total, 8, C.c_void_p(base), nbytes - 1) == (E_WORKSPACE, True, 0)
    assert _refusal_call(entry, dev, total, 8, C.c_void_p(base + 4), nbytes + 32) == (E_WORKSPACE, True, 0)
    rc, same, launched = _refusal_call(entry, dev, total, 8, C.c_void_p(base), nbytes)
    assert rc == 0 and launched > 0                  # the same call with a proper workspace runs
    for D in (0, 6, 516):
        assert _refusal_call(entry, dev, 64, D, None, 0) == (E_BADDIM, True, 0), D


# ---- 3. BPR forward ----------------------------------------------------------------------------------------------
@pytest.mark.parametrize("B", [1, 9, 1024, 1025])
@pytest.mark.parametrize("D", DS)
def test_bpr_forward_against_float64(cuda_device, D, B):
    """The reg terms 0.5 (|u0|^2 + |p0|^2 + |n0|^2) and their mean exact, softplus(<u,n> - <u,p>) per sample to 4 ulps,
    its mean and dscore = sigma(x)/B within their bounds, at score differences of +-40, +-180 and +-400.  The ego
    tables hold integers in [-2, 2], so that the sum of B <= 1025 reg terms stays below 2^24 halves: exact."""
    capi = _capi()
    dev = cuda_device
    rng = np.random.default_rng(D * 31 + B)
    nu, m = 40, 50
    U, I = _dyadic(rng, (nu, D), -2), _dyadic(rng, (m, D), -2)
    U0, I0 = _dyadic(rng, (nu, D), 0, -2, 2), _dyadic(rng, (m, D), 0, -2, 2)
    U[:3] = 0.0
    U[0, 0], U[1, 0], U[2, 0] = 20.0, 90.0, 200.0
    I[:2] = 0.0
    I[0, 0], I[1, 0] = 1.0, -1.0
    users, pos, neg = rng.integers(0, nu, B), rng.integers(0, m, B), rng.integers(0, m, B)
    special = [(u, p, n) for u in range(3) for (p, n) in ((0, 1), (1, 0))]
    for b, (u, p, n) in enumerate(special[:B]):
        users[b], pos[b], neg[b] = u, p, n
    ts = [_dev(a, dev) for a in (U, I, U0, I0, users, pos, neg)]
    out2 = torch.full((2,), SENT, device=dev)
    dscore = torch.full((B,), SENT, device=dev)
    work = torch.full((2 * B,), SENT, device=dev)
    capi.call("spex_bpr_fwd_f32", *[_p(t) for t in ts[:4]], D, *[_p(t) for t in ts[4:]], B, _p(out2), _p(dscore),
              _p(work), _st())
    S = U.astype(np.float64) @ I.astype(np.float64).T
    x = S[users, neg] - S[users, pos]                                         # exact
    reg = 0.5 * ((U0.astype(np.float64) ** 2).sum(1)[users] + (I0.astype(np.float64) ** 2).sum(1)[pos]
                 + (I0.astype(np.float64) ** 2).sum(1)[neg])                 # exact
    w = work.cpu().numpy()
    assert np.array_equal(w[B:], reg.astype(np.float32))
    reg_sum = np.float32(reg.sum())                                           # exact: integers / 2 below 2^24
    assert float(reg_sum) == reg.sum()
    assert out2.cpu().numpy()[1] == reg_sum / np.float32(B)                   # one IEEE division
    sp = np.logaddexp(0.0, x)
    tiny = sp < 2.0 ** -126
    _assert_within(w[:B], sp, np.where(tiny, 2.0 ** -126, 4 * _spacing(sp)), ("softplus", D, B))
    _assert_within(out2.cpu().numpy()[0], sp.mean(), _loss_tol(x, B) + float(_spacing(sp.mean())), ("loss", D, B))
    ref_ds = 1.0 / (1.0 + np.exp(-x)) / B
    _assert_within(dscore.cpu().numpy(), ref_ds, 4 * U_RND / B + _spacing(ref_ds), ("dscore", D, B))


# ---- the empty batch ---------------------------------------------------------------------------------------------
def test_empty_batch_loss_is_nan_and_gradients_zero(cuda_device):
    """BCEWithLogitsLoss of an empty batch is NaN (0/0); so are ops.bce_loss and both outputs of ops.bpr_loss, and
    their backward leaves zero gradients."""
    from spex_b200 import ops

    assert math.isnan(float(torch.nn.BCEWithLogitsLoss()(torch.zeros(0), torch.zeros(0))))
    dev = cuda_device
    nur, m, D = 6, 5, 64
    rng = np.random.default_rng(3)
    e = torch.zeros(0, dtype=torch.int64, device=dev)
    out = _dev(_dyadic(rng, (nur + m, D)), dev).requires_grad_(True)
    loss = ops.bce_loss(out, nur, e, e, torch.zeros(0, device=dev))
    assert math.isnan(float(loss))
    loss.backward()
    assert torch.equal(out.grad, torch.zeros_like(out))
    out.grad = None
    table = _dev(_dyadic(rng, (nur + m, D)), dev).requires_grad_(True)
    l, r = ops.bpr_loss(out, table, nur, e, e, e)
    assert math.isnan(float(l)) and math.isnan(float(r))
    (l + r).backward()
    assert torch.equal(out.grad, torch.zeros_like(out)) and torch.equal(table.grad, torch.zeros_like(table))


def test_empty_batch_entry_points_write_nan(cuda_device):
    """With B == 0 the loss outputs are written (NaN), not left as they were; per-sample outputs stay untouched."""
    capi = _capi()
    dev = cuda_device
    D = 8
    tab = torch.ones(4, D, device=dev)
    idx = torch.zeros(1, dtype=torch.int64, device=dev)
    lab = torch.zeros(1, device=dev)
    gamma, dgamma, loss = (torch.full((1,), SENT, device=dev) for _ in range(3))
    capi.call("spex_bce_fwd_f32", _p(tab), _p(tab), D, _p(idx), _p(idx), _p(lab), 0, _p(gamma), _p(loss), _p(dgamma),
              _st())
    assert math.isnan(float(loss)) and float(gamma) == SENT and float(dgamma) == SENT
    out2 = torch.full((2,), SENT, device=dev)
    work = torch.full((2,), SENT, device=dev)
    capi.call("spex_bpr_fwd_f32", _p(tab), _p(tab), _p(tab), _p(tab), D, _p(idx), _p(idx), _p(idx), 0, _p(out2),
              _p(dgamma), _p(work), _st())
    assert torch.isnan(out2).all() and float(dgamma) == SENT and bool((work == SENT).all())


# ---- 4. clear_rows / gather_owned_rows ---------------------------------------------------------------------------
@pytest.mark.parametrize("D,n", [(4, 700_000), (128, 20_000), (512, 5_000)])
def test_clear_and_gather_owned_rows_grid_stride(cuda_device, D, n):
    """n * D/4 float4 exceed two passes of the capped grid (303 104 float4 each); duplicate rows, rows on both edges
    of the window, rows outside it, and n = 0 (nothing written)."""
    capi = _capi()
    dev = cuda_device
    assert n * D // 4 > 2 * GRID_FLOAT4
    rng = np.random.default_rng(D)
    N = max(2 * n // 3, 1000)
    lo, hi = N // 4, 3 * N // 4
    table = _dyadic(rng, (N, D))
    rows = rng.integers(0, N, n)
    rows[:8] = [lo - 1, lo, hi - 1, hi, lo, hi - 1, 0, N - 1]
    rows[8:16] = rows[:8]
    rd = _dev(rows, dev)
    # gather: R[i] = table[rows[i]] if lo <= rows[i] < hi else 0, read from the local slice table[lo:hi]
    local = _dev(table[lo:hi], dev)
    R = torch.full((n, D), SENT, device=dev)
    capi.call("spex_gather_owned_rows_f32", _p(local), _p(rd), n, D, lo, hi, _p(R), _st())
    inside = (rows >= lo) & (rows < hi)
    ref = np.where(inside[:, None], table[rows], 0.0).astype(np.float32)
    assert np.array_equal(R.cpu().numpy(), ref)
    R0 = torch.full((2, D), SENT, device=dev)
    capi.call("spex_gather_owned_rows_f32", _p(local), None, 0, D, lo, hi, _p(R0), _st())
    assert bool((R0 == SENT).all())
    # clear: table[rows] = 0, every other row unchanged
    td = _dev(table, dev)
    capi.call("spex_clear_rows_f32", _p(td), _p(rd), n, D, _st())
    ref = table.copy()
    ref[rows] = 0.0
    assert np.array_equal(td.cpu().numpy(), ref)
    td2 = _dev(table, dev)
    capi.call("spex_clear_rows_f32", _p(td2), None, 0, D, _st())
    assert np.array_equal(td2.cpu().numpy(), table)


# ---- 5. Adam -----------------------------------------------------------------------------------------------------
LR, B1, B2, EPS = 1e-3, 0.9, 0.999, 1e-8
ADAM_SPECIAL = np.array([1e4, -1e-20, 0.0, -1e4, 1e-20], np.float32)


def _adam64(p, g, m, v, step, lr, b1, omb1, b2, omb2, eps, bc1_b1, bc2_b2):
    """torch.optim.Adam's formula in float64 (bias corrections from bc1_b1 ** step, bc2_b2 ** step)."""
    p, g, m, v = (np.asarray(a, np.float64) for a in (p, g, m, v))
    m1 = m + (g - m) * omb1
    v1 = v * b2 + omb2 * g * g
    denom = np.sqrt(v1) / math.sqrt(1.0 - bc2_b2 ** step) + eps
    upd = lr / (1.0 - bc1_b1 ** step) * (m1 / denom)
    return p - upd, m1, v1, upd, denom


@pytest.mark.parametrize("step", [1, 2, 1000, 100_000])
@pytest.mark.parametrize("n", [1, 2, 3, 4, 5, 4 * GRID_FLOAT4 + 4 * 7 + 3])
def test_adam_against_float64_and_torch(cuda_device, n, step):
    """spex_adam_f32 against torch's Adam formula in float64 (with the fp32 hyper-parameters the entry point
    receives), and against torch.optim.Adam in fp32.  The large n runs the grid-stride loop four passes and a
    3-element tail; gradients 0, +-1e-20 (eps dominates the denominator) and +-1e4 sit in the tail too."""
    capi = _capi()
    rng = np.random.default_rng(n + step)
    p = rng.standard_normal(n).astype(np.float32)
    if n <= 5:
        g = ADAM_SPECIAL[:n].copy()
    else:
        g = rng.standard_normal(n).astype(np.float32)
        g[:5] = ADAM_SPECIAL
        g[-5:] = ADAM_SPECIAL
    if step == 1:
        m = np.zeros(n, np.float32)
        v = np.zeros(n, np.float32)
    else:
        m = (rng.standard_normal(n) * 1e-2).astype(np.float32)
        v = (np.abs(rng.standard_normal(n)) * 1e-4).astype(np.float32)
        tiny = np.abs(g) == np.float32(1e-20)
        m[tiny], v[tiny] = 0.0, 0.0
    dev = cuda_device
    pd, gd, md, vd = (_dev(a, dev) for a in (p, g, m, v))
    capi.call("spex_adam_f32", _p(pd), _p(gd), _p(md), _p(vd), n, LR, B1, B2, EPS, step, _st())
    pg, mg, vg = (t.cpu().numpy().astype(np.float64) for t in (pd, md, vd))

    f = lambda x: float(np.float32(x))   # noqa: E731  the fp32 value the entry point receives
    b1, b2 = f(B1), f(B2)
    kern = dict(lr=f(LR), b1=b1, omb1=1.0 - b1, b2=b2, omb2=1.0 - b2, eps=f(EPS), bc1_b1=b1, bc2_b2=b2)
    p64, m64, v64, upd, denom = _adam64(p, g, m, v, step, **kern)
    mbig = np.maximum(np.abs(g.astype(np.float64) - m) * kern["omb1"], np.abs(m64))
    tol_m = 2 * 2.0 ** -23 * mbig + 2.0 ** -149
    _assert_within(mg, m64, tol_m, ("m", n, step))
    tol_v = 2 * 2.0 ** -23 * v64 + 2 * 2.0 ** -149
    _assert_within(vg, v64, tol_v, ("v", n, step))
    # the parameter, from the moments the kernel wrote
    denom_k = np.sqrt(vg) / math.sqrt(1.0 - b2 ** step) + kern["eps"]
    p64k = p.astype(np.float64) - kern["lr"] / (1.0 - b1 ** step) * (mg / denom_k)
    upd_k = np.abs(p64k - p)
    _assert_within(pg, p64k, _spacing(p64k) + 4 * 2.0 ** -23 * upd_k, ("p", n, step))

    # torch.optim.Adam in fp32: it rounds the hyper-parameters differently (1 - beta in double, then to fp32; the
    # bias corrections from the double betas), so the bound adds the float64 difference of the two conventions
    pt = torch.from_numpy(p.copy()).requires_grad_(True)
    opt = torch.optim.Adam([pt], lr=LR, betas=(B1, B2), eps=EPS)
    pt.grad = torch.from_numpy(g.copy())
    opt.state[pt] = {"step": torch.tensor(float(step - 1)), "exp_avg": torch.from_numpy(m.copy()),
                     "exp_avg_sq": torch.from_numpy(v.copy())}
    opt.step()
    tch = dict(lr=LR, b1=f(B1), omb1=f(1.0 - B1), b2=f(B2), omb2=f(1.0 - B2), eps=EPS, bc1_b1=B1, bc2_b2=B2)
    p64t, m64t, v64t, _, _ = _adam64(p, g, m, v, step, **tch)
    st = opt.state[pt]
    _assert_within(st["exp_avg"].numpy(), mg, np.abs(m64 - m64t) + 2 * tol_m, ("torch m", n, step))
    _assert_within(st["exp_avg_sq"].numpy(), vg, np.abs(v64 - v64t) + 2 * tol_v, ("torch v", n, step))
    lever = kern["lr"] / (1.0 - b1 ** step) / denom                  # d(update) / d(m)
    tol_p = np.abs(p64 - p64t) + 2 * _spacing(p64) + 8 * 2.0 ** -23 * np.abs(upd) + 2 * lever * tol_m
    _assert_within(pt.detach().numpy(), pg, tol_p, ("torch p", n, step))


# ---- 6. expert gate ----------------------------------------------------------------------------------------------
def _gate64(E0, E1, W, G=None):
    e0, e1, w = (torch.from_numpy(a).double().requires_grad_(G is not None) for a in (E0, E1, W))
    a = torch.softmax(torch.cat([e0, e1], 1) @ w, 1)
    out = e0 * a[:, 0:1] + e1 * a[:, 1:2]
    if G is None:
        return out.detach().numpy(), a.detach().numpy()
    (out * torch.from_numpy(G).double()).sum().backward()
    return e0.grad.numpy(), e1.grad.numpy(), w.grad.numpy(), a.detach().numpy()


@pytest.mark.parametrize("D", DS)
def test_expert_gate_forward_against_float64(cuda_device, D):
    """spex_expert_gate_f32 up to D = 512 (ops.expert_gate stops at 128 on purpose): the mix within 8u of the softmax
    weights times |e0| + |e1| plus three roundings; with tied gate columns the weights are exactly 1/2 and the
    output is exact."""
    capi = _capi()
    dev = cuda_device
    rng = np.random.default_rng(D)
    n = 1001
    E0, E1, W = _dyadic(rng, (n, D), -2), _dyadic(rng, (n, D), -2), _dyadic(rng, (2 * D, 2), -4)
    ref, a = _gate64(E0, E1, W)
    E0d, E1d, Wd = (_dev(x, dev) for x in (E0, E1, W))
    out = torch.full((n, D), SENT, device=dev)
    capi.call("spex_expert_gate_f32", _p(E0d), _p(E1d), _p(Wd), n, D, _p(out), _st())
    mag = np.abs(E0) + np.abs(E1)
    mix = a[:, 0:1] * np.abs(E0) + a[:, 1:2] * np.abs(E1)
    _assert_within(out.cpu().numpy(), ref, U_RND * (8 * mag + 3 * mix), ("gate", D))
    Wt = np.repeat(W[:, :1], 2, axis=1)
    Wtd = _dev(Wt, dev)
    capi.call("spex_expert_gate_f32", _p(E0d), _p(E1d), _p(Wtd), n, D, _p(out), _st())
    assert np.array_equal(out.cpu().numpy(), (0.5 * E0 + 0.5 * E1).astype(np.float32))


GATE_BLOCKS = 1184


@pytest.mark.parametrize("n", [0, 1, 7, 9472, 9473, 30_000])
@pytest.mark.parametrize("D", [20, 128])
def test_expert_gate_backward_against_float64_autograd(cuda_device, D, n):
    """spex_expert_gate_bwd_f32: n = 9473 and 30 000 give the 1184 x 8 warps more than one row each (the strided row
    loop and its dW partials); dE0 / dEout / dW within their bounds of float64 autograd, dW bit-identical on repeat
    and exactly zero for n = 0."""
    capi = _capi()
    dev = cuda_device
    rng = np.random.default_rng(D + n)
    nn = max(n, 1)
    E0, E1, G = _dyadic(rng, (nn, D), -2), _dyadic(rng, (nn, D), -2), _dyadic(rng, (nn, D), -3)
    W = _dyadic(rng, (2 * D, 2), -4)
    E0d, E1d, Gd, Wd = (_dev(x, dev) for x in (E0, E1, G, W))
    work = torch.empty(GATE_BLOCKS * 512, device=dev)

    def run():
        d0 = torch.full((nn, D), SENT, device=dev)
        d1 = torch.full((nn, D), SENT, device=dev)
        dW = torch.full((2 * D, 2), SENT, device=dev)
        capi.call("spex_expert_gate_bwd_f32", _p(E0d), _p(E1d), _p(Wd), _p(Gd), n, D, _p(d0), _p(d1), _p(dW),
                  _p(work), _st())
        return d0.cpu().numpy(), d1.cpu().numpy(), dW.cpu().numpy()

    d0, d1, dW = run()
    assert np.array_equal(run()[2], dW)
    if n == 0:
        assert np.array_equal(dW, np.zeros_like(dW))
        assert (d0 == SENT).all() and (d1 == SENT).all()
        return
    r0, r1, rW, a = _gate64(E0, E1, W, G)
    da = np.stack([(G.astype(np.float64) * E0).sum(1), (G.astype(np.float64) * E1).sum(1)], 1)   # exact
    M = np.abs(da).sum(1, keepdims=True)                                                          # |da0| + |da1|
    Wa = np.abs(W[:D]).sum(1)
    Wb = np.abs(W[D:]).sum(1)
    _assert_within(d0, r0, U_RND * (16 * np.abs(G) + 48 * M * Wa), ("dE0", D, n))
    _assert_within(d1, r1, U_RND * (16 * np.abs(G) + 48 * M * Wb), ("dEout", D, n))
    blocks = min((n + 7) // 8, GATE_BLOCKS)
    L = math.ceil(n / (8 * blocks)) + 8 + blocks
    sdot = (a * da).sum(1, keepdims=True)
    dz = np.abs(a * (da - sdot))                                                                  # [n, 2]
    E = np.concatenate([np.abs(E0), np.abs(E1)], 1).astype(np.float64)                            # [n, 2D]
    tol_w = U_RND * ((L + 2) * (E.T @ dz) + 32 * (E.T @ M))
    _assert_within(dW, rW, tol_w, ("dW", D, n))


# ---- 7. candidate scoring and dense ratings ----------------------------------------------------------------------
@pytest.mark.parametrize("D", DS)
def test_score_candidates_and_rating_exact(cuda_device, D):
    """spex_score_candidates_f32 and ops.rating_dense are exact on dyadic tables; the sigmoid within 3 ulps
    (expf 2 ulp, the add and the division 0.5 each)."""
    from spex_b200 import ops

    dev = cuda_device
    rng = np.random.default_rng(D + 1)
    nu, m = 60, 300
    U, I = _dyadic(rng, (nu, D), -3), _dyadic(rng, (m, D), -3)
    S = U.astype(np.float64) @ I.astype(np.float64).T
    Ud, Id = _dev(U, dev), _dev(I, dev)
    for n_u, n_c in ((37, 101), (1, 1), (9, 7)):
        users = rng.integers(0, nu, n_u)
        cand = rng.integers(0, m, (n_u, n_c)).astype(np.int32)
        got = ops.score_candidates(Ud, Id, _dev(users, dev), _dev(cand, dev))
        assert np.array_equal(got.cpu().numpy(), S[users[:, None], cand].astype(np.float32)), (n_u, n_c)
    users = rng.integers(0, nu, 37)
    raw = ops.rating_dense(Ud, Id, _dev(users, dev), apply_sigmoid=False)
    assert np.array_equal(raw.cpu().numpy(), S[users].astype(np.float32))
    sig = ops.rating_dense(Ud, Id, _dev(users, dev), apply_sigmoid=True).cpu().numpy()
    ref = 1.0 / (1.0 + np.exp(-S[users]))
    _assert_within(sig, ref, np.where(ref < 2.0 ** -126, 2.0 ** -126, 3 * _spacing(ref)), ("sigmoid", D))


@pytest.mark.parametrize("D", [4, 132])
def test_rating_dense_crosses_the_launch_chunk(cuda_device, D):
    """ops.rating_dense launches at most 8 x 65 535 users at a time; one user more crosses the seam, and the entry
    point itself refuses that many with SPEX_E_TOOBIG before writing anything."""
    from spex_b200 import ops

    dev = cuda_device
    rng = np.random.default_rng(D + 2)
    nu, m, B = 1000, 3, 8 * 65535 + 1
    U, I = _dyadic(rng, (nu, D), -3), _dyadic(rng, (m, D), -3)
    users = rng.integers(0, nu, B)
    Ud, Id, ud = _dev(U, dev), _dev(I, dev), _dev(users, dev)
    got = ops.rating_dense(Ud, Id, ud, apply_sigmoid=False)
    S = U.astype(np.float64) @ I.astype(np.float64).T
    assert np.array_equal(got.cpu().numpy(), S[users].astype(np.float32))
    out = torch.full((B, m), SENT, device=dev)
    rc = _capi().lib.spex_rating_f32(_p(Ud), _p(Id), D, _p(ud), B, m, 0, _p(out), _st())
    assert rc == E_TOOBIG
    assert bool((out == SENT).all())
