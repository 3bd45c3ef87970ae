"""DeviceGraph.long_row_plan (the segment list of spex_long_plan, include/spex_b200.h) over a seeded sweep of degree
profiles, column-block windows, seg_len and D.  The builder is plain torch and runs on CPU tensors, so this module
needs no GPU.

The assertions are the invariants the SpMM kernels rely on, not particular cut positions, so they stay valid when
the cells are cut differently:
  * every edge of every long row lies in exactly one segment, and no other edge does;
  * no segment is empty or longer than seg_len;
  * the hub cells come first, listed block-major, and none crosses a column-block boundary;
  * the mid-row segments follow in ascending row order;
  * row_seg lists each long row's segments in ascending edge order, tiling the row, consistently with long_segptr;
  * n_long, n_hub and n_hub_seg match their definitions;
  * bit 31 (the hot flag) on any columns does not change the plan.
Every profile gives some hub rows a column block holding exactly one edge and some an empty block, so a builder
that drops short or empty cells, or keeps empty ones, fails.
"""
import numpy as np
import pytest
import torch

from spex_b200.ops import DeviceGraph


def _window(n_cols, D, win, min_cb, epb):
    """(blocked, cb_cols, n_cb, hub degree threshold) as the header defines the column-blocked list."""
    blocked = n_cols * D * 4 > 4 * win
    cb = max(win // (D * 4), min_cb)
    n_cb = (n_cols + cb - 1) // cb
    return blocked, cb, n_cb, epb * n_cb


def _profile(rng, n_cols, seg_len, cb):
    """(rowptr int64, col int32) of a CSR whose degrees cover the long-row edges: empty and short rows, seg_len - 1
    .. seg_len + 1, 2 seg_len + 1, rows of many segments, and rows up to the whole table.  Every row with more than
    one block's worth of edges gets one block emptied and one block reduced to a single edge."""
    degs = [0, 1, 7, seg_len - 1, seg_len, seg_len + 1, 2 * seg_len + 1, 3 * seg_len]
    degs += list(rng.integers(0, 3 * seg_len, 12))
    degs += list(rng.integers(seg_len + 1, n_cols + 1, 10))
    degs += [n_cols, n_cols - 1]
    degs = [int(d) for d in rng.permutation(degs)]
    if rng.random() < 0.5:                      # a long first row and a long last row
        degs = [n_cols - 3] + degs + [seg_len + 2]
    n_cb = (n_cols + cb - 1) // cb
    cols = []
    for d in degs:
        c = np.sort(rng.choice(n_cols, d, replace=False))
        if d > 2 * cb and n_cb >= 3:
            b0, b1 = rng.choice(n_cb, 2, replace=False)
            keep = (c // cb != b0) & (c // cb != b1)
            one = rng.integers(b1 * cb, min((b1 + 1) * cb, n_cols))
            c = np.sort(np.concatenate([c[keep], [one]]))
        cols.append(c)
    rowptr = np.concatenate([[0], np.cumsum([c.size for c in cols])]).astype(np.int64)
    return torch.from_numpy(rowptr), torch.from_numpy(np.concatenate(cols).astype(np.int32))


def _check_plan(p, rowptr, col, n_cols, seg_len, D, win, min_cb, epb):
    rp = rowptr.numpy()
    c = (col.numpy().astype(np.int64)) & 0x7FFFFFFF
    deg = np.diff(rp)
    long_rows = np.flatnonzero(deg > seg_len)
    blocked, cb, n_cb, hub_deg = _window(n_cols, D, win, min_cb, epb)
    hubs = long_rows[deg[long_rows] >= hub_deg] if blocked else long_rows[:0]
    assert p["n_long"] == long_rows.size and p["long_rows"].tolist() == long_rows.tolist()
    assert p["n_hub"] == hubs.size

    start = p["seg_start"].numpy().astype(np.int64)
    cnt = p["seg_count"].numpy().astype(np.int64)
    segptr = p["long_segptr"].numpy().astype(np.int64)
    row_seg = p["row_seg"].numpy().astype(np.int64)
    n_seg, H = p["n_seg"], p["n_hub_seg"]
    assert start.size == cnt.size == row_seg.size == n_seg and segptr.size == long_rows.size + 1
    assert segptr[0] == 0 and segptr[-1] == n_seg and (np.diff(segptr) >= 1).all()
    assert ((cnt > 0) & (cnt <= seg_len)).all()
    assert sorted(row_seg.tolist()) == list(range(n_seg))          # a permutation: each segment owned once

    seg_row = np.empty(n_seg, np.int64)
    for k, r in enumerate(long_rows):
        own = row_seg[segptr[k]: segptr[k + 1]]
        seg_row[own] = r
        s, e = start[own], start[own] + cnt[own]
        assert s[0] == rp[r] and e[-1] == rp[r + 1]                   # the row's segments tile it in edge order
        assert (s[1:] == e[:-1]).all()

    # every long-row edge in exactly one segment, nothing else covered
    cover = np.zeros(int(rp[-1]), np.int64)
    for s, n in zip(start, cnt):
        cover[s: s + n] += 1
    want = np.zeros_like(cover)
    for r in long_rows:
        want[rp[r]: rp[r + 1]] = 1
    assert np.array_equal(cover, want)

    # hub cells first, block-major, each inside one column block; then mid rows in ascending row order
    is_hub = np.isin(seg_row, hubs)
    assert is_hub[:H].all() and not is_hub[H:].any()
    if H:
        first_blk = c[start[:H]] // cb
        last_blk = c[start[:H] + cnt[:H] - 1] // cb
        assert np.array_equal(first_blk, last_blk)
        assert (np.diff(first_blk) >= 0).all()
    assert (np.diff(seg_row[H:]) >= 0).all()
    mid_start = start[H:]
    same = seg_row[H:][1:] == seg_row[H:][:-1]
    assert (np.diff(mid_start)[same] > 0).all()

    # n_hub_seg: the segments of the hub rows' non-empty column-block cells, each cut to seg_len
    want_h = 0
    for r in hubs:
        per_block = np.bincount(c[rp[r]: rp[r + 1]] // cb, minlength=n_cb)
        want_h += int(((per_block + seg_len - 1) // seg_len).sum())
    assert H == want_h
    return H


# (window bytes, MIN_CB_COLS, HUB_EDGES_PER_BLOCK): a table that fits in L2, and column-blocked lists with
# narrow and wide blocks
WINDOWS = [(16 << 20, 1024, 16), (16 * 1024, 48, 4), (64 * 1024, 96, 2), (4 * 1024, 32, 1)]


@pytest.mark.parametrize("seed", range(3))
@pytest.mark.parametrize("D", [32, 64, 128])
@pytest.mark.parametrize("seg_len", [32, 64, 256])
@pytest.mark.parametrize("window", WINDOWS, ids=["fits_l2", "narrow", "wide", "tiny"])
def test_long_row_plan_invariants(monkeypatch, window, seg_len, D, seed):
    win, min_cb, epb = window
    monkeypatch.setattr(DeviceGraph, "L2_WINDOW_BYTES", win)
    monkeypatch.setattr(DeviceGraph, "MIN_CB_COLS", min_cb)
    monkeypatch.setattr(DeviceGraph, "HUB_EDGES_PER_BLOCK", epb)
    monkeypatch.delenv("SPEX_L2_WINDOW_MB", raising=False)
    monkeypatch.delenv("SPEX_HUB_EPB", raising=False)
    rng = np.random.default_rng(1000 * seg_len + 10 * D + seed)
    n_cols = int(rng.integers(1200, 3000))
    blocked, cb, _, _ = _window(n_cols, D, win, min_cb, epb)
    rowptr, col = _profile(rng, n_cols, seg_len, cb)
    p = DeviceGraph.long_row_plan(rowptr, col, n_cols, seg_len, D)
    H = _check_plan(p, rowptr, col, n_cols, seg_len, D, win, min_cb, epb)
    assert p["n_seg"] > 0 and (H > 0) == blocked                    # rows of ~n_cols edges are hub rows

    hot = col | torch.from_numpy(np.where(rng.random(col.numel()) < 0.3, -(2 ** 31), 0).astype(np.int32))
    assert bool((hot < 0).any())
    q = DeviceGraph.long_row_plan(rowptr, hot, n_cols, seg_len, D)
    assert q.keys() == p.keys()
    for k, v in p.items():
        assert (torch.equal(q[k], v) if torch.is_tensor(v) else q[k] == v), k


def test_long_row_plan_single_edge_hub_cells(monkeypatch):
    """Hub rows whose cells hold exactly one edge each (every column block but one) and one cell of several
    segments: each single-edge cell is a segment of its own, and the list still covers every edge once."""
    monkeypatch.setattr(DeviceGraph, "L2_WINDOW_BYTES", 4 * 1024)
    monkeypatch.setattr(DeviceGraph, "MIN_CB_COLS", 16)
    monkeypatch.setattr(DeviceGraph, "HUB_EDGES_PER_BLOCK", 1)
    monkeypatch.delenv("SPEX_L2_WINDOW_MB", raising=False)
    monkeypatch.delenv("SPEX_HUB_EPB", raising=False)
    n_cols, cb, seg_len, D = 1600, 16, 32, 64                    # 100 blocks of 16 columns: hub from 100 edges
    cols = [np.arange(0, n_cols, cb) + k for k in (0, 15)]       # one edge in every block
    cols.append(np.concatenate([np.arange(0, n_cols, cb)[:-1], np.arange(n_cols - cb, n_cols)]))
    cols.append(np.arange(40, 75))                               # a mid row (35 edges)
    rowptr = torch.from_numpy(np.concatenate([[0], np.cumsum([c.size for c in cols])]).astype(np.int64))
    col = torch.from_numpy(np.concatenate(cols).astype(np.int32))
    p = DeviceGraph.long_row_plan(rowptr, col, n_cols, seg_len, D)
    H = _check_plan(p, rowptr, col, n_cols, seg_len, D, 4 * 1024, 16, 1)
    assert p["n_hub"] == 3 and H == 100 + 100 + 99 + 1
    assert p["n_seg"] == H + 2
    assert int((p["seg_count"][:H] == 1).sum()) == 299
