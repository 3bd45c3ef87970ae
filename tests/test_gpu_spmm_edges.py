"""The SpMM layer of csrc/spmm.cu at the edges of its contract, against float64 references.

Covered entry points: spex_spmm_csr_f32, spex_spmm_layer_f32 (row subsets, x_nonzero masks, the Y / Z epilogue, the
exchange epilogue's peer stores, publish and fused Adam on same-device buffers), spex_propagate_mean_f32 / _bwd_f32,
spex_push_rows_f32_ex and spex_gather_f32, through every kernel path: the 256-bit and 128-bit row loops, the masked
loop, the segment list and segment runs of the long-row pass, its fix-up, and the generic-D kernel.

Exactness by construction.  Edge values are integers in [-8, 8] times 2^-3, tables and addends integers times 2^-4.
Every product and partial sum is then a multiple of 2^-7, and while sum |v| |x| of an output element stays below 2^24
such units every partial sum is exact in fp32, whatever the summation order.  Each case computes that bound in float64
and asserts it before relying on it; under it every path must equal the float64 reference bit for bit.  The
propagation uses values in {+-1, +-1/2} and small integer tables and checks the same bound on every layer; its last
layer multiplies the exact sum by fp32(1/(K+1)), one rounding, which the reference reproduces.  One case runs the real
normalised adjacency with random tables and checks each element against the fp32 summation bound of its row.

The long-row workspace (plan.partial) is filled with NaN before every call: a segment a kernel stops writing would
otherwise still hold the right value from the previous call.  Output rows a call must not write hold a sentinel.

Not covered here: multicast epilogues (NVSwitch memory, two GPUs: test_dist_gpu.py) and edge offsets beyond 2^31
(about 16 GB of col / val).
"""
import ctypes as C

import numpy as np
import pytest
import scipy.sparse as sp
import torch

pytestmark = pytest.mark.gpu

SENT = 12345.0                       # held by output rows a call must not write
UNIT = 2.0 ** -7                     # value unit (2^-3) times table unit (2^-4)
LIMIT = 2.0 ** 24
U_RND = 2.0 ** -24
E_BADARG, E_BADDIM, E_ALIGN = -1, -2, -3
HOT = -(2 ** 31)
HUB_RUN = 8                          # kHubRun in csrc/spmm.cu: hub cells per warp of the segment runs


# ---- helpers -----------------------------------------------------------------------------------------------------
def _capi():
    from spex_b200 import _capi

    return _capi


def _lib():
    return _capi().lib


def _p(t):
    return None if t is None else C.c_void_p(t.data_ptr())


def _st():
    return _capi().stream_ptr()


def _launches():
    return int(_lib().spex_launch_count())


def _table(n, D, dev, align=32, data=None, fill=None):
    """fp32 [n, D] whose first element is 32-byte aligned (align=32) or 16 bytes past a 32-byte boundary (16)."""
    off = 0 if align == 32 else 4
    buf = torch.empty(n * D + 8, dtype=torch.float32, device=dev)
    t = buf[off: off + n * D].view(n, D)
    assert t.data_ptr() % 32 == (0 if align == 32 else 16)
    if data is not None:
        t.copy_(torch.as_tensor(np.asarray(data, np.float32)).view(n, D))
    elif fill is not None:
        t.fill_(fill)
    return t


def _ints(rng, shape, exp=-4, lo=-8, hi=8):
    return (rng.integers(lo, hi + 1, shape) * 2.0 ** exp).astype(np.float32)


def _exact(bound, unit=UNIT):
    """The precondition of every exact comparison: sum |terms| of each element below 2^24 units."""
    m = float(np.max(bound)) if np.size(bound) else 0.0
    assert m < LIMIT * unit, f"exactness bound exceeded: {m / unit:.0f} units"


class Csr:
    """A host CSR (clean columns, fp32 values, optional hot bit 31 on a column subset) and its DeviceGraph."""

    def __init__(self, cols, n_cols, rng, dev, seg_len, hot=False, vals=None):
        self.n_rows, self.n_cols, self.seg_len = len(cols), n_cols, seg_len
        self.rowptr = np.concatenate([[0], np.cumsum([c.size for c in cols])]).astype(np.int64)
        self.col = np.concatenate(cols).astype(np.int32) if cols else np.zeros(0, np.int32)
        nnz = self.col.size
        if vals is None:
            mag = rng.integers(1, 9, nnz)
            vals = (np.where(rng.random(nnz) < 0.5, -mag, mag) * 2.0 ** -3).astype(np.float32)
        self.val = np.asarray(vals, np.float32)
        colh = self.col.copy()
        if hot:
            hot_cols = rng.random(n_cols) < 0.3
            colh = colh | np.where(hot_cols[self.col], HOT, 0).astype(np.int32)
            assert (colh < 0).any() and (colh >= 0).any()
        self.A = sp.csr_matrix((self.val.astype(np.float64), self.col, self.rowptr), shape=(self.n_rows, n_cols))
        from spex_b200 import ops

        self.g = ops.DeviceGraph(torch.from_numpy(self.rowptr).to(dev), torch.from_numpy(colh).to(dev),
                                 torch.from_numpy(self.val).to(dev), n_cols, seg_len=seg_len, col_hot=hot)
        self.deg = np.diff(self.rowptr)

    def ref(self, X):
        """(A X, |A| |X|) in float64."""
        X64 = X.double().cpu().numpy()
        return self.A @ X64, abs(self.A) @ np.abs(X64)

    def plan(self, D):
        """The graph's plan for width D, its partial workspace poisoned."""
        pl = self.g.plan(D)
        if self.g._plan_tensors is not None:
            self.g._plan_tensors.fill_(float("nan"))
        return pl


def _cols(rng, degs, n_cols, ends=True):
    """Sorted unique columns per row; with `ends`, every other row of degree >= 2 gathers columns 0 and n_cols - 1."""
    out = []
    for k, d in enumerate(degs):
        if ends and d >= 2 and k % 2 == 0:
            c = np.concatenate([[0, n_cols - 1], 1 + rng.choice(n_cols - 2, d - 2, replace=False)])
        else:
            c = rng.choice(n_cols, d, replace=False)
        out.append(np.sort(c))
    return out


def _spmm(h, X, Y=None, addend=None, a_s=1.0, Z=None, z_s=1.0, plan=None):
    pl = h.plan(X.shape[1]) if plan is None else plan
    g = h.g
    return _lib().spex_spmm_csr_f32(_p(g.rowptr), _p(g.col), _p(g.val), _p(X), g.n_rows, X.shape[1], _p(Y),
                                    _p(addend), a_s, _p(Z), z_s, pl, _st())


def _ep(Y=None, addend=None, a_s=1.0, Z=None, z_s=1.0, offset=0, y_peers=None, pub_src=None, pub_peers=None,
        adam=None):
    ep = _capi().SpmmEpilogue(Y=_p(Y), addend=_p(addend), addend_scale=a_s, Z=_p(Z), z_scale=z_s,
                              out_row_offset=offset, pub_src=_p(pub_src))
    if y_peers:
        ep.y_peers_host = (C.c_void_p * len(y_peers))(*[t.data_ptr() for t in y_peers])
        ep.n_y_peers = len(y_peers)
    if pub_peers:
        ep.pub_peers_host = (C.c_void_p * len(pub_peers))(*[t.data_ptr() for t in pub_peers])
        ep.n_pub_peers = len(pub_peers)
    if adam is not None:
        ep.adam_p, ep.adam_m, ep.adam_v = _p(adam["p"]), _p(adam["m"]), _p(adam["v"])
        ep.lr, ep.beta1, ep.beta2, ep.eps, ep.step = adam["lr"], adam["b1"], adam["b2"], adam["eps"], adam["step"]
    return ep


def _layer(h, X, ep, subset=None, nz=None, plan=None, n_sel=None):
    """spex_spmm_layer_f32; subset = (rows int32, long_slots, seg_ids) or None (all rows)."""
    rows, slots, segs = subset if subset is not None else (None, None, None)
    if n_sel is None:
        n_sel = -1 if rows is None else rows.numel()
    pl = h.plan(X.shape[1]) if plan is None else plan
    g = h.g
    return _lib().spex_spmm_layer_f32(_p(g.rowptr), _p(g.col), _p(g.val), _p(X), g.n_rows, X.shape[1], _p(rows),
                                      n_sel, _p(slots), 0 if slots is None else slots.numel(), _p(segs),
                                      0 if segs is None else segs.numel(), _p(nz), C.byref(ep), pl, _st())


def _eq(got, ref, what):
    got = got.double().cpu().numpy() if torch.is_tensor(got) else np.asarray(got, np.float64)
    ref = np.asarray(ref, np.float64)
    assert got.shape == ref.shape, (what, got.shape, ref.shape)
    bad = np.argwhere(~(got == ref))
    assert bad.size == 0, (what, bad[0].tolist(), float(got[tuple(bad[0])]), float(ref[tuple(bad[0])]))


def _all_paths(h, X, ref, dev, what, subset_rows=True):
    """Y of every full-layer path for X: the csr entry point, the layer entry point over all rows, every row listed
    in random order (row list + segment list), and an all-one x_nonzero mask."""
    D = X.shape[1]
    n = h.n_rows
    Y = _table(n, D, dev, fill=SENT)
    assert _spmm(h, X, Y=Y) == 0
    _eq(Y, ref, f"{what} csr")
    Y = _table(n, D, dev, fill=SENT)
    assert _layer(h, X, _ep(Y=Y)) == 0
    _eq(Y, ref, f"{what} layer")
    if subset_rows:
        perm = torch.from_numpy(np.random.default_rng(n).permutation(n)).to(dev)
        Y = _table(n, D, dev, fill=SENT)
        assert _layer(h, X, _ep(Y=Y), subset=h.g.row_subset(perm)) == 0
        _eq(Y, ref, f"{what} all rows listed")
    Y = _table(n, D, dev, fill=SENT)
    assert _layer(h, X, _ep(Y=Y), nz=torch.ones(h.n_cols, dtype=torch.uint8, device=dev)) == 0
    _eq(Y, ref, f"{what} all-one mask")
    torch.cuda.synchronize()


def _blocked(monkeypatch, win, min_cb, epb):
    from spex_b200 import ops

    monkeypatch.setattr(ops.DeviceGraph, "L2_WINDOW_BYTES", win)
    monkeypatch.setattr(ops.DeviceGraph, "MIN_CB_COLS", min_cb)
    monkeypatch.setattr(ops.DeviceGraph, "HUB_EDGES_PER_BLOCK", epb)
    monkeypatch.delenv("SPEX_L2_WINDOW_MB", raising=False)
    monkeypatch.delenv("SPEX_HUB_EPB", raising=False)


def _mixed(dev, monkeypatch, hot=False, seed=7):
    """A row block (70 rows over a 960-row table) with a column-blocked plan: columns in 20 blocks of 48 (any D),
    hub rows from 80 edges, seg_len 32; short rows, mid rows of 2 and 3 segments, hub rows with empty blocks and
    single-edge cells, and a degree-0 (padding) row."""
    _blocked(monkeypatch, 4096, 48, 4)
    rng = np.random.default_rng(seed)
    degs = [150, 0, 1, 5, 31, 32, 33, 40, 64, 65, 70, 79, 80, 300, 600, 900, 959] + list(rng.integers(0, 30, 50))
    degs += [90, 33]
    cols = _cols(rng, degs, 960)
    for k, d in enumerate(degs):                 # hub rows: one empty column block and one single-edge block
        if d >= 80 and d < 900:
            c = cols[k]
            b0, b1 = rng.choice(20, 2, replace=False)
            c = c[(c // 48 != b0) & (c // 48 != b1)]
            cols[k] = np.sort(np.concatenate([c, [b1 * 48 + int(rng.integers(48))]]))
    h = Csr(cols, 960, rng, dev, 32, hot=hot)
    assert 0 < h.g.n_hub_seg < h.g.n_seg and h.g.n_hub >= 4
    return h


# ---- 1. row degrees ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("hot", [False, True])
@pytest.mark.parametrize("align", [32, 16])
@pytest.mark.parametrize("D", [32, 64, 128])
@pytest.mark.parametrize("seg_len", [32, 64, 256])
@pytest.mark.parametrize("profile", ["mixed", "all_long"])
def test_row_degrees_every_path(cuda_device, profile, seg_len, D, align, hot):
    """Degrees on the batch (32 edges) and lane-group switches, at seg_len - 1 / seg_len / seg_len + 1, 2 seg_len + 1,
    long rows of more than 32 and more than 64 segments (the fix-up's list spans two and three 32-entry batches), a
    long first row, consecutive long rows and a long last row; columns 0 and n_cols - 1 gathered; X has more rows
    than the output."""
    s = seg_len
    if profile == "mixed":
        degs = [2 * s + 1, 0, 1, 7, 8, 9, 31, 32, 33, 63, 64, 65, 96, 97, s - 1, s, s + 1, 33 * s + 5, 0, 3,
                65 * s + 3, s + 1, 2, 65 * s + 3]
    else:
        degs = [s + 1, s + 2, 2 * s, 2 * s + 1, 3 * s + 7, 33 * s + 5, 65 * s + 3, s + 1]
    n_cols = 65 * s + 41
    rng = np.random.default_rng(seg_len * 1000 + D + align + hot)
    h = Csr(_cols(rng, degs, n_cols), n_cols, rng, cuda_device, seg_len, hot=hot)
    assert h.g.n_long == sum(d > s for d in degs) and h.g.n_hub_seg == 0
    assert max(np.diff(h.g.long_segptr.cpu().numpy())) > 64
    X = _table(n_cols, D, cuda_device, align, _ints(rng, (n_cols, D)))
    ref, bound = h.ref(X)
    _exact(bound)
    _all_paths(h, X, ref, cuda_device, f"{profile} s={s} D={D} a={align}")


# ---- 2. column-blocked plans ---------------------------------------------------------------------------------------
# (seg_len, columns per block, blocks, hub edges per block): hub rows from epb * n_cb edges
BLOCKED = {"s32": (32, 48, 20, 4), "s64": (64, 96, 12, 12)}


def _blocked_graph(dev, monkeypatch, cfg, residue, hot, seed):
    """Hub rows built block by block (cells of 0, 1, up to a whole block of edges: some longer than seg_len), mid rows
    with an odd total of segments, and a last hub row sized so that n_hub_seg % 8 == residue; residue None: no mid
    rows, n_hub_seg == n_seg."""
    s, cb, n_cb, epb = BLOCKED[cfg]
    n_cols = cb * n_cb
    _blocked(monkeypatch, 1024, cb, epb)            # window / (D * 4) < cb for every D: blocks of cb columns
    rng = np.random.default_rng(seed)
    hub_deg = epb * n_cb

    def hub_row(counts):
        return np.concatenate([b * cb + np.sort(rng.choice(cb, int(k), replace=False)) for b, k in enumerate(counts)])

    rows, n_hseg = [], 0
    for _ in range(5):
        counts = rng.integers(0, cb + 1, n_cb)
        counts[rng.integers(n_cb)] = 0
        counts[rng.integers(n_cb)] = 1
        counts[rng.integers(n_cb)] = cb
        if counts.sum() < hub_deg:
            counts[:] = cb
        rows.append(hub_row(counts))
        n_hseg += int(((counts + s - 1) // s).sum())
    # the last hub row: two cells of s + 8 edges (2 segments each) and k single-edge cells
    k = (residue if residue is not None else 0) - (n_hseg + 4)
    k %= 8
    counts = np.zeros(n_cb, np.int64)
    counts[0] = counts[n_cb - 1] = s + 8
    counts[1: 1 + k] = 1
    while counts.sum() < hub_deg:                  # too short for a hub row: add 8 single-edge cells
        free = np.flatnonzero(counts == 0)[:8]
        assert free.size == 8
        counts[free] = 1
    rows.append(hub_row(counts))
    n_hseg += int(((counts + s - 1) // s).sum())
    if residue is not None:
        mids = [s + 1, 2 * s + 1, hub_deg - 1, s + 5]          # 2 + 3 + ... segments: an odd total
        mids = [d for d in mids if s < d < hub_deg]
        n_mid = sum((d + s - 1) // s for d in mids)
        if n_mid % 2 == 0:
            mids.append(2 * s + 3)                             # 3 segments
        rows += [np.sort(rng.choice(n_cols, d, replace=False)) for d in mids]
        rows += _cols(rng, list(rng.integers(0, s + 1, 30)) + [s, 1, 0], n_cols)
    order = rng.permutation(len(rows))
    h = Csr([rows[i] for i in order], n_cols, rng, dev, s, hot=hot)
    g = h.g
    assert g.n_hub == 6 and g.n_hub_seg == n_hseg
    cnt = g.seg_count.cpu().numpy()
    assert (cnt[: g.n_hub_seg] == 1).any() and (cnt[: g.n_hub_seg] == s).any()
    if residue is None:
        assert g.n_hub_seg == g.n_seg
    else:
        assert g.n_hub_seg % HUB_RUN == residue and (g.n_seg - g.n_hub_seg) % 2 == 1
    return h


@pytest.mark.parametrize("hot", [False, True])
@pytest.mark.parametrize("residue", [1, 2, 3, 4, 5, 6, 7, None], ids=lambda r: f"r{r}" if r is not None else "all_hub")
@pytest.mark.parametrize("cfg", list(BLOCKED))
def test_column_blocked_plans(cuda_device, monkeypatch, cfg, residue, hot):
    """Builder plans with hub cells (segment runs of 8 hub cells / 2 mid segments per warp on the 256-bit full layer,
    one segment per warp elsewhere): n_hub_seg in every residue mod 8, all segments hub cells, an odd number of mid
    segments, empty and single-edge cells, cells longer than seg_len; the hot flag on hub, mid and short rows."""
    seed = 100 * list(BLOCKED).index(cfg) + 10 * (residue or 0) + int(hot)
    h = _blocked_graph(cuda_device, monkeypatch, cfg, residue, hot, seed)
    rng = np.random.default_rng(3)
    for D in (32, 64, 128):
        for align in (32, 16):
            X = _table(h.n_cols, D, cuda_device, align, _ints(rng, (h.n_cols, D)))
            ref, bound = h.ref(X)
            _exact(bound)
            _all_paths(h, X, ref, cuda_device, f"{cfg} r={residue} D={D} a={align}")


# ---- 3. hand-made segment lists ------------------------------------------------------------------------------------
def _hand_plan(h, rng, D, dev, hub_frac, hot):
    """A spex_long_plan with random cuts: every long row cut into pieces of 1..seg_len edges, listed in row order,
    n_hub_seg = hub_frac of the list."""
    rp, s = h.rowptr, h.seg_len
    long_rows = np.flatnonzero(h.deg > s)
    starts, counts, segptr = [], [], [0]
    for r in long_rows:
        e = rp[r]
        while e < rp[r + 1]:
            n = int(min(rng.integers(1, s + 1), rp[r + 1] - e))
            starts.append(e)
            counts.append(n)
            e += n
        segptr.append(len(starts))
    n_seg = len(starts)
    t = dict(long_rows=torch.tensor(long_rows, dtype=torch.int32, device=dev),
             long_segptr=torch.tensor(segptr, dtype=torch.int32, device=dev),
             seg_start=torch.tensor(starts, dtype=torch.int64, device=dev),
             seg_count=torch.tensor(counts, dtype=torch.int32, device=dev),
             row_seg=torch.arange(n_seg, dtype=torch.int32, device=dev),
             partial=torch.full((n_seg * D + 8,), float("nan"), device=dev))
    H = int(round(hub_frac * n_seg))
    plan = _capi().LongPlan(s, long_rows.size, n_seg, 1 if hot else 0, t["long_rows"].data_ptr(),
                            t["long_segptr"].data_ptr(), t["partial"].data_ptr(), t["seg_start"].data_ptr(),
                            t["seg_count"].data_ptr(), t["row_seg"].data_ptr(), H)
    return plan, t, np.asarray(segptr), long_rows


@pytest.mark.parametrize("hub_frac", [0.0, 0.37, 1.0])
@pytest.mark.parametrize("D", [32, 64, 128])
def test_hand_made_segment_lists(cuda_device, D, hub_frac):
    """Cuts the builder never makes but the header allows (pieces of 1..seg_len edges at random places), with every
    split of the list into hub cells and mid segments, through the full layer, a row subset and a mask."""
    rng = np.random.default_rng(D + int(hub_frac * 100))
    degs = [300, 5, 33, 64, 0, 1000, 2100, 40, 7, 129, 32, 31, 97]
    n_cols = 2200
    h = Csr(_cols(rng, degs, n_cols), n_cols, rng, cuda_device, 32, hot=bool(hub_frac == 0.37))
    plan, t, segptr, long_rows = _hand_plan(h, rng, D, cuda_device, hub_frac, hot=hub_frac == 0.37)
    pl = C.byref(plan)
    for align in (32, 16):
        X = _table(n_cols, D, cuda_device, align, _ints(rng, (n_cols, D)))
        ref, bound = h.ref(X)
        _exact(bound)
        Y = _table(h.n_rows, D, cuda_device, fill=SENT)
        t["partial"].fill_(float("nan"))
        assert _spmm(h, X, Y=Y, plan=pl) == 0
        _eq(Y, ref, f"hand csr a={align}")
        # a subset in no particular order: long rows 12, 6, 0, 2, 5, short row 1, empty row 4
        sel = np.array([12, 6, 1, 0, 2, 4, 5])
        slots = np.searchsorted(long_rows, sel[np.isin(sel, long_rows)])
        seg_ids = np.concatenate([np.arange(segptr[k], segptr[k + 1]) for k in slots])
        sub = (torch.tensor(sel, dtype=torch.int32, device=cuda_device),
               torch.tensor(slots, dtype=torch.int32, device=cuda_device),
               torch.tensor(seg_ids, dtype=torch.int32, device=cuda_device))
        for nz in (None, torch.ones(n_cols, dtype=torch.uint8, device=cuda_device)):
            Y = _table(h.n_rows, D, cuda_device, fill=SENT)
            t["partial"].fill_(float("nan"))
            assert _layer(h, X, _ep(Y=Y), subset=sub, nz=nz, plan=pl) == 0
            want = np.full_like(ref, SENT)
            want[sel] = ref[sel]
            _eq(Y, want, f"hand subset a={align} mask={nz is not None}")
    torch.cuda.synchronize()


# ---- 4. x_nonzero ----------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("hot", [False, True])
@pytest.mark.parametrize("D", [32, 64, 128])
@pytest.mark.parametrize("case", ["all_zero", "all_one", "superset", "long_row_columns", "ignored_16B", "subset"])
def test_x_nonzero_masks(cuda_device, monkeypatch, case, D, hot):
    h = _mixed(cuda_device, monkeypatch, hot=hot)
    rng = np.random.default_rng(D)
    n, m = h.n_rows, h.n_cols
    Xd = _ints(rng, (m, D))
    live = np.ones(m, bool)
    mask = np.ones(m, np.uint8)
    align, subset = 32, None
    if case == "all_zero":
        live[:] = False
        mask[:] = 0
    elif case == "superset":
        live = rng.random(m) < 0.2
        mask = (live | (rng.random(m) < 0.2)).astype(np.uint8)
        assert (mask.astype(bool) & ~live).any()
    elif case == "long_row_columns":               # the columns of the mid rows (the hub rows gather nearly all)
        lr = np.flatnonzero((h.deg > h.seg_len) & (h.deg < 80))
        live[:] = False
        live[np.unique(np.concatenate([h.col[h.rowptr[r]: h.rowptr[r + 1]] for r in lr]))] = True
        mask = live.astype(np.uint8)
        assert not live.all()
    elif case == "ignored_16B":                     # the 128-bit path does not read the mask: a wrong one is harmless
        align = 16
        mask[:] = 0
    elif case == "subset":
        live = rng.random(m) < 0.3
        mask = live.astype(np.uint8)
        sel = rng.permutation(np.union1d(np.flatnonzero(h.deg > h.seg_len)[::2], rng.choice(n, 15, False)))
        subset = h.g.row_subset(torch.from_numpy(sel).to(cuda_device))
    Xd[~live] = 0.0
    X = _table(m, D, cuda_device, align, Xd)
    nz = torch.from_numpy(mask).to(cuda_device)
    ref, bound = h.ref(X)
    _exact(bound)
    Y = _table(n, D, cuda_device, fill=SENT)
    assert _layer(h, X, _ep(Y=Y), subset=subset, nz=nz) == 0
    want = ref
    if subset is not None:
        want = np.full_like(ref, SENT)
        want[sel] = ref[sel]
    _eq(Y, want, case)
    torch.cuda.synchronize()


# ---- 5. row subsets and the Y / Z epilogue ---------------------------------------------------------------------------
def _subset_rows(h, kind, rng):
    n = h.n_rows
    if kind == "descending":
        return np.arange(n)[::-1].copy()
    if kind == "random":
        return rng.permutation(n)[: n // 2]
    if kind == "long_only":
        return rng.permutation(np.flatnonzero(h.deg > h.seg_len))
    if kind == "padding_row":
        return np.flatnonzero(h.deg == 0)[:1]
    raise ValueError(kind)


@pytest.mark.parametrize("kind", ["descending", "random", "long_only", "padding_row", "none", "all"])
@pytest.mark.parametrize("D", [32, 64, 128])
def test_row_subsets_leave_other_rows(cuda_device, monkeypatch, kind, D):
    """Listed rows get the full layer's value in Y, Z and the Y peer tables; every other row keeps its sentinel.
    n_sel == 0 writes and launches nothing; n_sel < 0 is every row."""
    h = _mixed(cuda_device, monkeypatch)
    rng = np.random.default_rng(D + 1)
    n, m = h.n_rows, h.n_cols
    X = _table(m, D, cuda_device, 32, _ints(rng, (m, D)))
    add = _table(n, D, cuda_device, 32, _ints(rng, (n, D)))
    ref, bound = h.ref(X)
    a64 = add.double().cpu().numpy()
    _exact(bound + np.abs(a64) * 2)
    Y, Z = _table(n, D, cuda_device, fill=SENT), _table(n, D, cuda_device, fill=SENT)
    peers = [_table(n + 40, D, cuda_device, fill=SENT) for _ in range(3)]
    ep = _ep(Y=Y, addend=add, a_s=-2.0, Z=Z, z_s=0.5, offset=37, y_peers=peers)
    if kind == "none":
        sel, subset = np.zeros(0, np.int64), (torch.zeros(1, dtype=torch.int32, device=cuda_device), None, None)
        before = _launches()
        assert _layer(h, X, ep, subset=subset, n_sel=0) == 0
        assert _launches() == before
    elif kind == "all":
        sel = np.arange(n)
        assert _layer(h, X, ep) == 0
    else:
        sel = _subset_rows(h, kind, rng)
        assert sel.size > 0
        if kind == "padding_row":
            assert h.deg[sel[0]] == 0
        assert _layer(h, X, ep, subset=h.g.row_subset(torch.from_numpy(sel).to(cuda_device))) == 0
    wY = np.full_like(ref, SENT)
    wY[sel] = ref[sel]
    wZ = np.full_like(ref, SENT)
    wZ[sel] = (a64[sel] * -2.0 + ref[sel]) * 0.5
    _eq(Y, wY, "Y")
    _eq(Z, wZ, "Z")
    wP = np.full((n + 40, D), SENT)
    wP[37 + sel] = ref[sel]
    for k, P in enumerate(peers):
        _eq(P, wP, f"peer {k}")


@pytest.mark.parametrize("variant", ["Y", "Z_no_addend", "YZ_scale0", "YZ_scale-2", "YZ_scale0.5", "Z_in_place"])
@pytest.mark.parametrize("entry", ["csr", "layer", "layer_subset"])
def test_epilogue_variants(cuda_device, monkeypatch, variant, entry):
    h = _mixed(cuda_device, monkeypatch, hot=True)
    rng = np.random.default_rng(11)
    n, m = h.n_rows, h.n_cols
    for D in (32, 64, 128):
        X = _table(m, D, cuda_device, 32, _ints(rng, (m, D)))
        ref, bound = h.ref(X)
        a0 = _ints(rng, (n, D))
        _exact(bound + 2 * np.abs(a0))
        Y = _table(n, D, cuda_device, fill=SENT) if variant.startswith("Y") else None
        Z = _table(n, D, cuda_device, fill=SENT) if "Z" in variant else None
        add, a_s, z_s = _table(n, D, cuda_device, 32, a0), 1.0, 4.0
        if variant == "Z_no_addend":
            add, z_s = None, 0.25
        elif variant.startswith("YZ_scale"):
            a_s = float(variant[len("YZ_scale"):])
        elif variant == "Z_in_place":
            Z.copy_(add)
            add, a_s, z_s = Z, 0.5, 2.0 ** -3
        sel = np.arange(n)
        if entry == "csr":
            assert _spmm(h, X, Y=Y, addend=add, a_s=a_s, Z=Z, z_s=z_s) == 0
        elif entry == "layer":
            assert _layer(h, X, _ep(Y=Y, addend=add, a_s=a_s, Z=Z, z_s=z_s)) == 0
        else:
            sel = rng.permutation(n)[: n // 3]
            sel = np.union1d(sel, np.flatnonzero(h.deg > h.seg_len)[:3])[::-1].copy()
            sub = h.g.row_subset(torch.from_numpy(sel).to(cuda_device))
            assert _layer(h, X, _ep(Y=Y, addend=add, a_s=a_s, Z=Z, z_s=z_s), subset=sub) == 0
        if Y is not None:
            w = np.full_like(ref, SENT)
            w[sel] = ref[sel]
            _eq(Y, w, f"{variant} Y D={D}")
        if Z is not None:
            a = 0.0 if variant == "Z_no_addend" else a0.astype(np.float64)
            zz = (a * a_s + ref) * z_s
            w = a0.astype(np.float64) if variant == "Z_in_place" else np.full_like(ref, SENT)
            w[sel] = zz[sel]
            _eq(Z, w, f"{variant} Z D={D}")


# ---- 6. exchange epilogue on one GPU -----------------------------------------------------------------------------
@pytest.mark.parametrize("offset", [0, 37])
@pytest.mark.parametrize("n_peers", [1, 3, 8])
def test_y_peers_and_publish(cuda_device, monkeypatch, n_peers, offset):
    """Y to 1, 3 and 8 peer tables (same-device buffers) at out_row_offset 0 and 37, over all rows and a subset,
    and the publish of pub_src rows to the same number of tables."""
    h = _mixed(cuda_device, monkeypatch, hot=n_peers == 3)
    rng = np.random.default_rng(n_peers + offset)
    n, m, D = h.n_rows, h.n_cols, 64
    X = _table(m, D, cuda_device, 32, _ints(rng, (m, D)))
    ref, bound = h.ref(X)
    _exact(bound)
    src = _table(n, D, cuda_device, 32, rng.standard_normal((n, D)))
    src64 = src.double().cpu().numpy()
    tot = n + offset + 5
    for sel in (None, rng.permutation(n)[: n // 2]):
        peers = [_table(tot, D, cuda_device, fill=SENT) for _ in range(n_peers)]
        pubs = [_table(tot, D, cuda_device, fill=SENT) for _ in range(n_peers)]
        Z = _table(n, D, cuda_device, fill=SENT)
        ep = _ep(Z=Z, offset=offset, y_peers=peers, pub_src=src, pub_peers=pubs)
        sub = None if sel is None else h.g.row_subset(torch.from_numpy(sel).to(cuda_device))
        assert _layer(h, X, ep, subset=sub) == 0
        rows = np.arange(n) if sel is None else sel
        wY = np.full((tot, D), SENT)
        wY[offset + rows] = ref[rows]
        wP = np.full((tot, D), SENT)
        wP[offset + rows] = src64[rows]
        wZ = np.full_like(ref, SENT)
        wZ[rows] = ref[rows]
        for k in range(n_peers):
            _eq(peers[k], wY, f"y peer {k} sel={sel is not None}")
            _eq(pubs[k], wP, f"pub peer {k} sel={sel is not None}")
        _eq(Z, wZ, "Z")


@pytest.mark.parametrize("subset", [False, True])
@pytest.mark.parametrize("publish", [False, True])
@pytest.mark.parametrize("with_z", [False, True])
@pytest.mark.parametrize("step", [1, 1000])
def test_fused_adam_equals_spex_adam(cuda_device, monkeypatch, step, with_z, publish, subset):
    """The Adam epilogue on the Z row as gradient equals spex_adam_f32 on the same gradient bit for bit; unlisted rows
    of p / m / v are untouched; the published rows are the updated p rows."""
    h = _mixed(cuda_device, monkeypatch)
    rng = np.random.default_rng(step + 2 * with_z + 4 * publish + 8 * subset)
    n, m, D, off = h.n_rows, h.n_cols, 128, 37
    X = _table(m, D, cuda_device, 32, _ints(rng, (m, D)))
    add = _table(n, D, cuda_device, 32, _ints(rng, (n, D)))
    ref, bound = h.ref(X)
    a64 = add.double().cpu().numpy()
    _exact(bound + np.abs(a64))
    g_ref = ((a64 + ref) * 0.25).astype(np.float32)           # exact: the gradient of every row
    p0 = rng.standard_normal((n, D)).astype(np.float32)
    m0 = (rng.standard_normal((n, D)) * 0.1).astype(np.float32)
    v0 = (rng.random((n, D)) * 0.01).astype(np.float32)
    hyper = dict(lr=1e-3, b1=0.9, b2=0.999, eps=1e-8, step=step)
    p, mm, v = (_table(n, D, cuda_device, 32, a) for a in (p0, m0, v0))
    Z = _table(n, D, cuda_device, fill=SENT) if with_z else None
    pubs = [_table(n + off, D, cuda_device, fill=SENT) for _ in range(2)] if publish else None
    ep = _ep(Z=Z, addend=add, a_s=1.0, z_s=0.25, offset=off, pub_peers=pubs, adam=dict(p=p, m=mm, v=v, **hyper))
    sel = np.sort(rng.permutation(n)[: n // 2])[::-1].copy() if subset else np.arange(n)
    sub = h.g.row_subset(torch.from_numpy(sel).to(cuda_device)) if subset else None
    assert _layer(h, X, ep, subset=sub) == 0
    # spex_adam_f32 over the whole table with the exact gradient
    pe, me, ve = (_table(n, D, cuda_device, 32, a) for a in (p0, m0, v0))
    gd = _table(n, D, cuda_device, 32, g_ref)
    _capi().call("spex_adam_f32", _p(pe), _p(gd), _p(me), _p(ve), n * D, hyper["lr"], hyper["b1"], hyper["b2"],
                 hyper["eps"], step, _st())
    for got, new, old, what in ((p, pe, p0, "p"), (mm, me, m0, "m"), (v, ve, v0, "v")):
        w = old.astype(np.float64).copy()
        w[sel] = new.double().cpu().numpy()[sel]
        _eq(got, w, f"adam {what}")
    assert not np.array_equal(pe.cpu().numpy()[sel], p0[sel])
    if with_z:
        w = np.full_like(ref, SENT)
        w[sel] = g_ref[sel]
        _eq(Z, w, "Z")
    if publish:
        w = np.full((n + off, D), SENT)
        w[off + sel] = pe.double().cpu().numpy()[sel]
        for k, P in enumerate(pubs):
            _eq(P, w, f"published p {k}")


# ---- 7. generic D ----------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("D", [4, 8, 20, 36, 48, 100, 132, 256, 260, 512])
def test_generic_d(cuda_device, D):
    """D outside {32, 64, 128}: one edge per step, long rows serially (the plan is not used), with the Y / Z epilogue
    and, through the layer entry point, Y to three peer tables at a row offset."""
    rng = np.random.default_rng(D)
    degs = [0, 1, 31, 32, 33, 97, 1500, 5, 2 * 1024 + 1, 64, 3]
    n_cols = 2200
    h = Csr(_cols(rng, degs, n_cols), n_cols, rng, cuda_device, 32)
    assert h.g.n_long > 0
    X = _table(n_cols, D, cuda_device, 16, _ints(rng, (n_cols, D)))
    add = _table(h.n_rows, D, cuda_device, 16, _ints(rng, (h.n_rows, D)))
    ref, bound = h.ref(X)
    a64 = add.double().cpu().numpy()
    _exact(bound + 2 * np.abs(a64))
    Y = _table(h.n_rows, D, cuda_device, 16, fill=SENT)
    Z = _table(h.n_rows, D, cuda_device, 16, fill=SENT)
    assert _spmm(h, X, Y=Y, addend=add, a_s=-2.0, Z=Z, z_s=0.5) == 0
    _eq(Y, ref, "Y")
    _eq(Z, (a64 * -2.0 + ref) * 0.5, "Z")
    peers = [_table(h.n_rows + 37, D, cuda_device, fill=SENT) for _ in range(3)]
    assert _layer(h, X, _ep(offset=37, y_peers=peers)) == 0
    w = np.full((h.n_rows + 37, D), SENT)
    w[37:] = ref
    for k, P in enumerate(peers):
        _eq(P, w, f"peer {k}")


# ---- 8. propagation --------------------------------------------------------------------------------------------------
def _prop_graph(dev, N, D_rng):
    """Square graph with values in {+-1, +-1/2}: short rows of degree 0..5 and a few long rows (seg_len 32) that
    gather only short rows, so |A|^K |X| stays small."""
    rng = D_rng
    long = np.arange(0, N, 37)
    short = np.setdiff1d(np.arange(N), long)
    cols = []
    for r in range(N):
        if r in long:
            cols.append(np.sort(rng.choice(short, int(rng.integers(33, 70)), replace=False)))
        else:
            cols.append(np.sort(rng.choice(N, int(rng.integers(0, 6)), replace=False)))
    nnz = sum(c.size for c in cols)
    vals = (rng.choice([-1.0, -0.5, 0.5, 1.0], nnz)).astype(np.float32)
    return Csr(cols, N, rng, dev, 32, vals=vals)


@pytest.mark.parametrize("D", [64, 20])
@pytest.mark.parametrize("K", [0, 1, 2, 3, 4])
def test_propagate_mean_and_backward(cuda_device, K, D):
    rng = np.random.default_rng(K * 10 + D)
    N = 400
    h = _prop_graph(cuda_device, N, rng)
    assert h.g.n_long > 0
    A, Aabs = h.A, abs(h.A)
    E0 = _ints(rng, (N, D), exp=0, lo=-3, hi=3)
    G = _ints(rng, (N, D), exp=0, lo=-3, hi=3)
    inv = np.float64(np.float32(1.0) / np.float32(K + 1))
    lib = _lib()
    for fwd in (True, False):
        x0 = E0 if fwd else G
        # reference: exact layer sums; every partial sum bounded by sum_k |A|^k |x0| in units of 2^-K
        S, cur, babs, bcur = x0.astype(np.float64), x0.astype(np.float64), np.abs(x0).astype(np.float64), np.abs(x0)
        for _ in range(K):
            cur = A @ cur if fwd else x0 + A @ cur
            bcur = Aabs @ bcur if fwd else np.abs(x0) + Aabs @ bcur
            S = S + cur if fwd else cur
            babs = babs + bcur if fwd else bcur
        _exact(babs, unit=2.0 ** -K)
        want = (S * inv).astype(np.float32) if K else x0
        src = _table(N, D, cuda_device, 32, x0)
        out = _table(N, D, cuda_device, fill=SENT)
        tmp = [_table(N, D, cuda_device, fill=float("nan")) for _ in range(2)]
        pl = h.plan(D)
        fn = lib.spex_propagate_mean_f32 if fwd else lib.spex_propagate_mean_bwd_f32
        rc = fn(_p(h.g.rowptr), _p(h.g.col), _p(h.g.val), _p(src), N, D, K, _p(out),
                _p(tmp[0]) if K >= 2 else None, _p(tmp[1]) if K >= 3 else None, pl, _st())
        assert rc == 0
        _eq(out, want, f"fwd={fwd} K={K}")
        # N == 0 writes nothing
        out2 = _table(N, D, cuda_device, fill=SENT)
        assert fn(_p(h.g.rowptr), _p(h.g.col), _p(h.g.val), _p(src), 0, D, K, _p(out2), _p(tmp[0]), _p(tmp[1]),
                  pl, _st()) == 0
        _eq(out2, np.full((N, D), SENT), "N=0")
        # refusals: tmp0 NULL for K >= 2, tmp1 NULL for K >= 3
        before = _launches()
        if K >= 2:
            assert fn(_p(h.g.rowptr), _p(h.g.col), _p(h.g.val), _p(src), N, D, K, _p(out2), None, _p(tmp[1]),
                      pl, _st()) == E_BADARG
        if K >= 3:
            assert fn(_p(h.g.rowptr), _p(h.g.col), _p(h.g.val), _p(src), N, D, K, _p(out2), _p(tmp[0]), None,
                      pl, _st()) == E_BADARG
        assert _launches() == before
        _eq(out2, np.full((N, D), SENT), "refused")


# ---- 9. push rows and gather ---------------------------------------------------------------------------------------
@pytest.mark.parametrize("n_ctas", [0, 1, 3])
@pytest.mark.parametrize("n_peers", [1, 8])
def test_push_rows(cuda_device, n_peers, n_ctas):
    """spex_push_rows_f32_ex: every peer table gets rows [off, off + n) = src, the rest keeps its sentinel; one and
    three CTAs run the grid-stride loop many times and rotate the peer order."""
    rng = np.random.default_rng(n_peers + n_ctas)
    n, D, off = 1000, 64, 37
    src = _table(n, D, cuda_device, 16, rng.standard_normal((n, D)))
    peers = [_table(n + off + 3, D, cuda_device, fill=SENT) for _ in range(n_peers)]
    arr = (C.c_void_p * n_peers)(*[t.data_ptr() for t in peers])
    _capi().call("spex_push_rows_f32_ex", _p(src), n, D, off, arr, n_peers, n_ctas, _st())
    w = np.full((n + off + 3, D), SENT)
    w[off: off + n] = src.double().cpu().numpy()
    for k, P in enumerate(peers):
        _eq(P, w, f"peer {k}")


@pytest.mark.parametrize("divisor", [1.0, 0.6])
@pytest.mark.parametrize("with_scale", [False, True])
@pytest.mark.parametrize("with_idx", [False, True])
def test_gather(cuda_device, with_idx, with_scale, divisor):
    """spex_gather_f32 against numpy fp32 (each operation correctly rounded): out = src[idx] * scale / divisor, over
    more elements than one pass of its capped grid."""
    rng = np.random.default_rng(int(with_idx) + 2 * int(with_scale))
    n = 148 * 16 * 256 + 12345
    src = rng.standard_normal(n).astype(np.float32)
    idx = rng.integers(0, n, n).astype(np.int64) if with_idx else None
    scale = np.where(rng.random(n) < 0.4, 0.0, rng.standard_normal(n)).astype(np.float32) if with_scale else None
    src_d, idx_d, scale_d = (None if a is None else torch.from_numpy(a).to(cuda_device) for a in (src, idx, scale))
    out = torch.full((n,), SENT, device=cuda_device)
    _capi().call("spex_gather_f32", _p(src_d), _p(idx_d), _p(scale_d), divisor, _p(out), n, _st())
    w = src[idx] if with_idx else src.copy()
    if with_scale:
        w = w * scale
    if divisor != 1.0:
        w = w / np.float32(divisor)
    assert np.array_equal(out.cpu().numpy(), w.astype(np.float32))


# ---- 10. refusals --------------------------------------------------------------------------------------------------
def test_refusals_launch_nothing(cuda_device, monkeypatch):
    """Every refusal returns its code before anything is launched and leaves the outputs alone."""
    h = _mixed(cuda_device, monkeypatch)
    rng = np.random.default_rng(0)
    n, m = h.n_rows, h.n_cols
    lib = _lib()
    X = _table(m, 516, cuda_device, 32, _ints(rng, (m, 516)))
    Y = _table(n, 516, cuda_device, fill=SENT)
    Z = _table(n, 516, cuda_device, fill=SENT)
    add = _table(n, 516, cuda_device, 32, _ints(rng, (n, 516)))
    g = h.g

    def csr(D, Xp=None, Yp=None, Ap=None, Zp=None, plan=None):
        return lib.spex_spmm_csr_f32(_p(g.rowptr), _p(g.col), _p(g.val), Xp or _p(X), n, D, Yp or _p(Y),
                                     Ap or _p(add), 1.0, Zp or _p(Z), 1.0, plan or h.plan(64), _st())

    def off(t, b):
        return C.c_void_p(t.data_ptr() + b)

    before = _launches()
    for D in (0, 6, 516, -4):
        assert csr(D) == E_BADDIM, D
    assert csr(64, Yp=off(Y, 4)) == E_ALIGN
    assert csr(64, Zp=off(Z, 8)) == E_ALIGN
    assert csr(64, Ap=off(add, 4)) == E_ALIGN
    assert csr(64, Xp=off(X, 4)) == E_ALIGN
    # the plan: partial misaligned, seg_len < 32, long rows without a segment list, unknown flags
    base = h.g.plan(64)._obj
    fields = [f for f, _ in _capi().LongPlan._fields_]

    def variant(**kw):
        q = _capi().LongPlan(*[getattr(base, f) for f in fields])
        for k, v in kw.items():
            setattr(q, k, v)
        return C.byref(q)

    assert csr(64, plan=variant(partial=base.partial + 4)) == E_ALIGN
    assert csr(64, plan=variant(seg_len=31)) == E_BADARG
    for f in ("seg_start", "seg_count", "row_seg", "long_rows", "long_segptr", "partial"):
        assert csr(64, plan=variant(**{f: None})) == E_BADARG, f
    assert csr(64, plan=variant(flags=2)) == E_BADARG
    assert csr(64, plan=variant(n_hub_seg=base.n_seg + 1)) == E_BADARG
    # generic D: no row subsets, hot flag, publish or Adam
    X20 = X.view(-1)[: m * 20].view(m, 20)
    sub = h.g.row_subset(torch.arange(5, device=cuda_device))
    assert _layer(h, X20, _ep(Y=Y), subset=sub) == E_BADDIM
    assert csr(20, plan=variant(flags=1)) == E_BADDIM
    assert _layer(h, X20, _ep(Y=Y, pub_src=add, pub_peers=[Z])) == E_BADDIM
    assert _layer(h, X20, _ep(Z=Z, adam=dict(p=Y, m=Z, v=add, lr=1e-3, b1=0.9, b2=0.999, eps=1e-8, step=1))) == E_BADDIM
    # the descriptor: misaligned Y / Z / addend / peer table, Adam at step 0
    X64 = X.view(-1)[: m * 64].view(m, 64)
    assert _layer(h, X64, _ep(Y=Y), n_sel=0, subset=(None, None, None)) == 0
    for ep in (_ep(Y=Y[:, 1:]), _ep(Z=Z[:, 2:]), _ep(Z=Z, addend=add[:, 1:]), _ep(y_peers=[Y[:, 3:]]),
               _ep(Z=Z, adam=dict(p=Y, m=Z, v=add, lr=1e-3, b1=0.9, b2=0.999, eps=1e-8, step=0))):
        assert _layer(h, X64, ep) in (E_ALIGN, E_BADARG)
    assert _launches() == before
    torch.cuda.synchronize()
    _eq(Y, np.full((n, 516), SENT), "Y untouched")
    _eq(Z, np.full((n, 516), SENT), "Z untouched")


# ---- 11. the real adjacency: per-element rounding bound ----------------------------------------------------------------
@pytest.mark.parametrize("align", [32, 16])
@pytest.mark.parametrize("blocked", [False, True])
def test_normalised_adjacency_within_row_bound(cuda_device, monkeypatch, blocked, align):
    """build_norm_adj values and random tables at D = 64: each element within (chain + tree depth) u sum |v| |x| of
    the float64 product, chain length at most the row degree, instead of a bound relative to the table's maximum."""
    from oracle import lightgcn_oracle as O
    from spex_b200.graph import build_norm_adj

    if blocked:
        _blocked(monkeypatch, 16 * 1024, 48, 10)
    nu, mi = 1500, 800
    u, i = O.random_bipartite(nu, mi, 20000, 5)
    rng = np.random.default_rng(6)
    hub_deg = (90, 300, 700, 1400)
    hu = np.concatenate([rng.choice(nu, d, replace=False) for d in hub_deg])
    hi = np.repeat(np.arange(len(hub_deg)), hub_deg)
    key = np.unique(np.concatenate([u * mi + i, hu * mi + hi]))
    cg = build_norm_adj(key // mi, key % mi, nu + 1, mi)
    from spex_b200 import ops

    g = ops.DeviceGraph.from_host(cg, cuda_device, seg_len=64)
    assert g.n_long > 0 and (g.n_hub_seg > 0) == blocked
    N, D = cg.n_rows, 64
    A = sp.csr_matrix((cg.val.astype(np.float64), cg.col, cg.rowptr), shape=(N, N))
    X = _table(N, D, cuda_device, align, rng.standard_normal((N, D)))
    X64 = X.double().cpu().numpy()
    ref, s_abs = A @ X64, abs(A) @ np.abs(X64)
    Y = _table(N, D, cuda_device, fill=SENT)
    pl = g.plan(D)
    g._plan_tensors.fill_(float("nan"))
    _capi().call("spex_spmm_csr_f32", _p(g.rowptr), _p(g.col), _p(g.val), _p(X), N, D, _p(Y), None, 1.0, None, 1.0,
                 pl, _st())
    deg = np.diff(cg.rowptr).astype(np.float64)[:, None]
    n = deg + 8                                   # chain of a lane group <= degree; xor tree and fix-up: <= 8 more
    tol = n * U_RND / (1 - n * U_RND) * s_abs
    err = np.abs(Y.double().cpu().numpy() - ref)
    bad = np.argwhere(err > tol)
    assert bad.size == 0, (bad[0].tolist(), float(err[tuple(bad[0])]), float(tol[tuple(bad[0])]))
