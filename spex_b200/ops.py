"""Operators of the LightGCN_SPEX hot path: thin PyTorch host code over the C-ABI (libspex_b200.so).

PyTorch is used for device memory, streams and autograd bookkeeping only; every arithmetic step
below is one of the hand-written sm_100a kernels declared in include/spex_b200.h.  There is no
CPU or ATen fallback: a CPU tensor raises.

Reference call sites replaced (paths relative to /root/reference/LightGCN_SPEX/code):
    propagate_mean      utility1/model.py:66-97   (cat + K x torch.sparse.mm + stack + mean)
    bce_loss/gather_dot utility1/model.py:111-121 (gather, mul, sum, BCEWithLogitsLoss)
    bpr_loss            north_star addition (SURVEY §8 a5)
    score_topk*         north_star addition: getUsersRating (model.py:14-15) + top-k
    score_candidates    utility1/batch_test.py:28-40 (hoisted out of the per-user loop)
    expert_gate         utility1/model_expert_s.py:154-161
    adam_step           main_rec.py:23,37
"""
from __future__ import annotations

import ctypes as C
from typing import Optional

import numpy as np
import torch

from . import _capi
from ._capi import LongPlan, SpmmEpilogue, call, ptr, stream_ptr
from .graph import CSRGraph, DEFAULT_SEG_LEN


class _Workspaces:
    """Persistent device scratch of the training step (SURVEY §2.1 K6/K7: at the 1B-edge size every
    [N, D] fp32 temporary is 3.84 GB; the reference's autograd allocates and zero-fills several per
    step).  Off by default (every call allocates, results never alias); the training loops switch
    it on: the propagation ping-pong tables, the dense gradient table - zero-filled ONCE, afterwards
    only the rows the last scatter touched are cleared - and the sort workspace are then reused."""

    def __init__(self):
        self.enabled = False
        self.buf = {}
        self.dirty = {}      # name -> list of int64 row-index tensors written since the buffer was zero

    def get(self, name, shape, device, zero=False):
        key = (name, tuple(shape), str(device))
        t = self.buf.get(key) if self.enabled else None
        if t is None:
            t = (torch.zeros if zero else torch.empty)(*shape, dtype=torch.float32, device=device)
            if self.enabled:
                self.buf[key] = t
                self.dirty[key] = []
        elif zero:
            D = shape[-1]
            for rows in self.dirty[key]:
                call("spex_clear_rows_f32", ptr(t), ptr(rows), rows.numel(), D, stream_ptr())
            self.dirty[key] = []
        return t, key

    def mark(self, key, *row_lists):
        if self.enabled and key in self.dirty:
            self.dirty[key].extend(r for r in row_lists if r is not None and r.numel())

    def clear(self):
        self.buf.clear()
        self.dirty.clear()


workspaces = _Workspaces()


def enable_persistent_workspaces(on: bool = True):
    """Reuse the [N, D] scratch tables of the training step across steps (see _Workspaces)."""
    workspaces.enabled = bool(on)
    if not on:
        workspaces.clear()


def _scatter_workspace(total, device):
    """Device workspace of the sorted scatter for `total` list entries (None: the scan form is used)."""
    nbytes = int(call("spex_scatter_workspace_bytes", int(total)))
    if nbytes == 0:
        return None, 0
    key = ("scatter_ws", str(device))
    t = workspaces.buf.get(key) if workspaces.enabled else None
    if t is None or t.numel() < nbytes:
        t = torch.empty(nbytes, dtype=torch.uint8, device=device)
        if workspaces.enabled:
            workspaces.buf[key] = t
    return t, nbytes


def _need_cuda(*tensors):
    for t in tensors:
        if t is not None and not t.is_cuda:
            raise RuntimeError(
                "spex_b200 runs on sm_100a only: got a CPU tensor (there is no CPU fallback path)"
            )


def _f32c(t: torch.Tensor) -> torch.Tensor:
    if t.dtype != torch.float32:
        raise TypeError(f"expected float32, got {t.dtype}")
    return t if t.is_contiguous() else t.contiguous()


def _i64c(t: torch.Tensor, device) -> torch.Tensor:
    if not torch.is_tensor(t):
        t = torch.as_tensor(np.asarray(t))
    t = t.to(device=device, dtype=torch.int64, non_blocking=True)
    return t if t.is_contiguous() else t.contiguous()


class DeviceGraph:
    """CSR adjacency resident in HBM + long-row plan + (optional) transpose map.

    Layout in HBM (DESIGN.md §3): rowptr int64 [n_rows+1], col int32 [nnz], val fp32 [nnz];
    for the 1B-edge graph that is 16 GB for (col,val) and 120 MB for rowptr.
    """

    interleave_split = 0   # always 0: bench.py still reports it (config.interleaved_row_classes)

    def __init__(self, rowptr, col, val, n_cols: int, tpos=None, seg_len: int = DEFAULT_SEG_LEN,
                 row_offset: int = 0, symmetric: bool = True, D_hint: int = 64, col_hot: bool = False,
                 values_symmetric: bool = False):
        _need_cuda(rowptr, col, val)
        assert rowptr.dtype == torch.int64 and col.dtype == torch.int32 and val.dtype == torch.float32
        self.rowptr, self.col, self.val = rowptr, col, val
        self.n_rows = rowptr.numel() - 1
        self.n_cols = int(n_cols)
        self.nnz = col.numel()
        self.tpos = tpos
        self.row_offset = int(row_offset)
        self.symmetric = symmetric
        # val of (c, r) == val of (r, c) bit for bit (no tpos needed for the transposed values).  Not implied by
        # `symmetric`: a weighted build computes (d_u*w)*d_i one way and (d_i*w)*d_u the other.
        self.values_symmetric = values_symmetric
        self._tval_pos = None         # a row block's map to its transposed values (from_host)
        self.device = val.device
        self.seg_len = int(seg_len)
        self._plan_struct = None
        self._plan_D = 0
        self._plan_tensors = None
        self.col_hot = False          # bit 31 of col flags hot table rows (SPEX_PLAN_COL_HOTBIT)
        if col_hot:                   # a row block cut from an already marked graph
            self.col_hot = True
        self._build_plan(D_hint)

    # -- construction ---------------------------------------------------------------------------
    @classmethod
    def from_host(cls, g: CSRGraph, device, seg_len: int = DEFAULT_SEG_LEN, D_hint: int = 64):
        dev = torch.device(device)
        rowptr = torch.from_numpy(np.ascontiguousarray(g.rowptr)).to(dev)
        col = torch.from_numpy(np.ascontiguousarray(g.col)).to(dev)
        tpos = None if g.tpos is None else torch.from_numpy(np.ascontiguousarray(g.tpos)).to(dev)
        if g.tval is None:
            val = torch.from_numpy(np.ascontiguousarray(g.val)).to(dev)
            tval_pos = None
        else:
            # a row block's transposed values behind its own values in one buffer, [val | tval], and a block-local
            # map into the second half: spex_edge_dropout_f32 reads the transposed value of edge e at val[tpos[e]],
            # so they reach the kernel through its existing tpos argument (12 B per edge)
            nnz = int(g.val.size)
            val = torch.from_numpy(np.concatenate([g.val, g.tval]).astype(np.float32, copy=False)).to(dev)[:nnz]
            tval_pos = torch.arange(nnz, 2 * nnz, dtype=torch.int64, device=dev)
        out = cls(rowptr, col, val, g.n_cols, tpos, seg_len, g.row_offset, D_hint=D_hint,
                  values_symmetric=g.values_symmetric)
        out._tval_pos = tval_pos
        return out

    @classmethod
    def from_sparse_coo(cls, A: torch.Tensor, device, seg_len: int = DEFAULT_SEG_LEN):
        """From what BasicDataset.getSparseGraph() returns (coalesced COO, int64 indices)."""
        A = A.coalesce()
        idx = A.indices()
        n_rows, n_cols = A.shape
        dev = torch.device(device)
        rows = idx[0].to(dev)
        counts = torch.bincount(rows, minlength=n_rows)
        rowptr = torch.zeros(n_rows + 1, dtype=torch.int64, device=dev)
        torch.cumsum(counts, 0, out=rowptr[1:])
        col = idx[1].to(dev).to(torch.int32)
        val = A.values().to(dev).to(torch.float32)
        return cls(rowptr, col, val, n_cols, None, seg_len)

    # -- long-row plan --------------------------------------------------------------------------
    L2_WINDOW_BYTES = 16 << 20   # table bytes per column block: a window the 126 MB L2 keeps
    MIN_CB_COLS = 1024
    HUB_EDGES_PER_BLOCK = 16     # average edges per (row, column block) that make blocking pay (r02 sweep, ms per layer / GB of DRAM reads of the segment kernel: 64 -> 52.4 / 118, 32 -> 51.3 / 98, 16 -> 51.4 / 84)

    def _build_plan(self, D: int):
        self.__dict__.update(self.long_row_plan(self.rowptr, self.col, self.n_cols, self.seg_len, D))
        self._plan_D = 0

    @classmethod
    def long_row_plan(cls, rowptr: torch.Tensor, col: torch.Tensor, n_cols: int, seg_len: int, D: int) -> dict:
        """The segment list of spex_long_plan (include/spex_b200.h) for a CSR (int64 rowptr, int32 col, which
        may carry the hot flag in bit 31) and embedding width D, built on the tensors' device: the tensors
        long_rows, long_segptr (int32), seg_start (int64), seg_count, row_seg (int32) and the counts n_long,
        n_seg, n_hub (hub rows), n_hub_seg (hub cells, listed first).

        Rows with more than seg_len edges are long.  Hub rows (>= HUB_EDGES_PER_BLOCK edges per column block
        on average) are cut at column-block boundaries and their cells listed BLOCK-MAJOR: concurrently
        running warps gather from one ~32 MB window of the table, which L2 keeps resident.  Measured
        (profiles/microbench/l2_window.py): 12.7 TB/s for 128-edge rows in a 32 MB window vs 6.8 TB/s over
        the whole table - but only 6.7 TB/s for 16-edge rows, so rows too short to fill their blocks are mid
        rows.  A table that fits in L2 has no hub rows.  Mid rows follow, in ascending row order, and every
        cell is cut every seg_len edges from its first edge.
        """
        if seg_len < 32:
            raise ValueError("seg_len must be >= 32")
        dev = rowptr.device
        nnz = col.numel()
        deg = rowptr[1:] - rowptr[:-1]
        long_rows = torch.nonzero(deg > seg_len).flatten()
        n_long = int(long_rows.numel())
        ldeg = deg[long_rows]
        is_hub = torch.zeros_like(ldeg, dtype=torch.bool)
        parts_start, parts_cnt, parts_row = [], [], []
        n_hub_cells = 0                                   # hub cells come first in the list
        if n_cols * D * 4 > 4 * cls.L2_WINDOW_BYTES:
            import os as _os
            win = int(_os.environ.get("SPEX_L2_WINDOW_MB", 0)) << 20 or cls.L2_WINDOW_BYTES
            epb = int(_os.environ.get("SPEX_HUB_EPB", 0)) or cls.HUB_EDGES_PER_BLOCK
            cb_cols = max(win // (D * 4), cls.MIN_CB_COLS)
            n_cb = (n_cols + cb_cols - 1) // cb_cols
            is_hub = ldeg >= epb * n_cb
            hub_slots = torch.nonzero(is_hub).flatten()   # indices into long_rows
            if hub_slots.numel():
                hrows = long_rows[hub_slots]
                nh = hrows.numel()
                lo = rowptr[hrows].unsqueeze(1).expand(nh, n_cb + 1).clone()
                hi = rowptr[hrows + 1].unsqueeze(1).expand(nh, n_cb + 1).clone()
                target = (torch.arange(n_cb + 1, device=dev, dtype=torch.int64) * cb_cols).unsqueeze(0)
                steps = int(ldeg.max().item()).bit_length() + 1
                last = nnz - 1
                for _ in range(steps):  # vectorised lower_bound of every block boundary in every hub row
                    mid = (lo + hi) >> 1
                    go = ((col[mid.clamp(max=last)] & 0x7FFFFFFF).to(torch.int64) < target) & (lo < hi)
                    lo = torch.where(go, mid + 1, lo)
                    hi = torch.where(go, hi, mid)
                pos = lo  # [nh, n_cb+1]: first edge of the row with column >= b * cb_cols
                del lo, hi, mid, go
                cs = pos[:, :-1].t().reshape(-1)               # block-major flattening
                cc = (pos[:, 1:] - pos[:, :-1]).t().reshape(-1)
                cr = hub_slots.repeat(n_cb)
                keep = cc > 0
                parts_start.append(cs[keep]); parts_cnt.append(cc[keep]); parts_row.append(cr[keep])
                n_hub_cells = int(parts_cnt[0].numel())
        mid_slots = torch.nonzero(~is_hub).flatten()
        mrows = long_rows[mid_slots]
        parts_start.append(rowptr[mrows]); parts_cnt.append(deg[mrows]); parts_row.append(mid_slots)
        cell_start = torch.cat(parts_start)
        cell_cnt = torch.cat(parts_cnt)
        cell_row = torch.cat(parts_row)
        pieces = (cell_cnt + seg_len - 1) // seg_len   # cap a segment at seg_len edges
        seg_cell = torch.repeat_interleave(torch.arange(cell_cnt.numel(), device=dev), pieces)
        first = torch.cumsum(pieces, 0) - pieces
        piece_idx = torch.arange(seg_cell.numel(), device=dev) - first[seg_cell]
        seg_start = cell_start[seg_cell] + piece_idx * seg_len
        seg_end = torch.minimum(seg_start + seg_len, (cell_start + cell_cnt)[seg_cell])
        seg_row = cell_row[seg_cell]
        n_seg = int(seg_start.numel())
        if n_seg >= 2 ** 31:
            raise ValueError("too many long-row segments")
        # per row, segments in ascending edge order = fixed summation order
        order = torch.sort(seg_row * (nnz + 1) + seg_start, stable=True).indices
        counts = torch.bincount(seg_row, minlength=n_long)
        segptr = torch.zeros(n_long + 1, dtype=torch.int64, device=dev)
        torch.cumsum(counts, 0, out=segptr[1:])
        return {"n_long": n_long, "n_seg": n_seg, "n_hub": int(is_hub.sum()),
                "n_hub_seg": int(pieces[:n_hub_cells].sum()),
                "long_rows": long_rows.to(torch.int32), "long_segptr": segptr.to(torch.int32),
                "seg_start": seg_start.contiguous(), "seg_count": (seg_end - seg_start).to(torch.int32).contiguous(),
                "row_seg": order.to(torch.int32).contiguous()}

    HOT_L2_BYTES = 48 << 20   # table bytes flagged hot (kept in L2 by the evict_last policy)

    def mark_hot_columns(self, D: int, col_degree: Optional[torch.Tensor] = None,
                         budget_bytes: Optional[int] = None) -> int:
        """Flag the most frequently gathered table rows in bit 31 of `col` (in place).

        The kernels gather flagged rows with the L2 evict_last policy and everything else with
        evict_first, so the hottest HOT_L2_BYTES of the table stay L2-resident.  `col_degree[c]` =
        how many edges gather column c; for the symmetric normalised adjacency that is the row
        degree, which is the default.  Returns the number of hot rows (0: nothing marked).
        """
        if self.col_hot:
            return -1
        import os as _os
        budget = budget_bytes if budget_bytes is not None else (
            int(_os.environ.get("SPEX_HOT_L2_MB", 0)) << 20 or self.HOT_L2_BYTES)   # env: tuning sweeps
        n_hot = min(budget // (D * 4), self.n_cols)
        if self.n_cols * D * 4 <= 2 * budget or n_hot <= 0 or D not in (32, 64, 128):
            return 0  # the table fits in L2 anyway / generic-D path has no hint variant
        if col_degree is None:
            if self.n_rows != self.n_cols:
                raise ValueError("column degrees are needed for a non-square graph")
            col_degree = self.rowptr[1:] - self.rowptr[:-1]
        thr = torch.topk(col_degree, n_hot).values[-1]
        hot = col_degree >= torch.clamp(thr, min=2)     # never flag rows that are gathered once
        if int(hot.sum()) > 2 * n_hot:                  # a flat degree distribution: no hot set
            return 0
        chunk = 1 << 28
        int_min = -(2 ** 31)
        for s0 in range(0, self.nnz, chunk):
            c = self.col[s0: s0 + chunk]
            c.bitwise_or_(hot[c.long()].to(torch.int32) * int_min)
        self.col_hot = True
        self._plan_D = 0
        return int(hot.sum())

    def clean_col(self) -> torch.Tensor:
        """Column indices without the hot flag."""
        return (self.col & 0x7FFFFFFF) if self.col_hot else self.col

    def plan(self, D: int):
        """ctypes pointer to a spex_long_plan for embedding width D (NULL if nothing to say)."""
        if self.n_long == 0 and not self.col_hot:
            return None
        if self._plan_D != D:
            flags = 1 if self.col_hot else 0
            if self.n_long == 0:
                st = LongPlan(self.seg_len, 0, 0, flags)
                self._plan_tensors = None
            else:
                partial = torch.empty(self.n_seg * D, dtype=torch.float32, device=self.device)
                st = LongPlan(self.seg_len, self.n_long, self.n_seg, flags, self.long_rows.data_ptr(),
                              self.long_segptr.data_ptr(), partial.data_ptr(), self.seg_start.data_ptr(),
                              self.seg_count.data_ptr(), self.row_seg.data_ptr(), self.n_hub_seg)
                self._plan_tensors = partial
            self._plan_struct = st
            self._plan_D = D
        return C.byref(self._plan_struct)

    # -- row subsets (receptive field of a mini-batch) ----------------------------------------------
    def _edge_positions(self, rows: torch.Tensor):
        """Positions in col/val of all edges of `rows` (int64 ids), row by row."""
        a = self.rowptr[rows]
        cnt = self.rowptr[rows + 1] - a
        total = int(cnt.sum().item())
        first = torch.cumsum(cnt, 0) - cnt
        pos = torch.repeat_interleave(a - first, cnt, output_size=total) + torch.arange(total, device=self.device)
        return pos, total

    def degree_sum(self, rows: torch.Tensor) -> int:
        return int((self.rowptr[rows + 1] - self.rowptr[rows]).sum().item())

    def neighbors(self, rows: torch.Tensor) -> torch.Tensor:
        """Sorted unique column ids of the listed rows (int64): the rows a layer restricted to `rows` reads."""
        pos, total = self._edge_positions(rows)
        if total == 0:
            return torch.empty(0, dtype=torch.int64, device=self.device)
        c = self.col[pos]
        if self.col_hot:
            c = c & 0x7FFFFFFF
        return torch.unique(c.to(torch.int64))

    def row_subset(self, rows: torch.Tensor):
        """(rows int32, long_slots int32 | None, seg_ids int32 | None) for spex_spmm_layer_f32: the listed
        rows, and - for those on the long-row path - their slots in the plan with all their segments."""
        rows = rows.to(torch.int64)
        r32 = rows.to(torch.int32).contiguous()
        if self.n_long == 0:
            return r32, None, None
        deg = self.rowptr[rows + 1] - self.rowptr[rows]
        lr = rows[deg > self.seg_len]
        if lr.numel() == 0:
            return r32, None, None
        slots = torch.searchsorted(self.long_rows.to(torch.int64), lr)
        segptr = self.long_segptr.to(torch.int64)
        a = segptr[slots]
        cnt = segptr[slots + 1] - a
        total = int(cnt.sum().item())
        first = torch.cumsum(cnt, 0) - cnt
        pos = torch.repeat_interleave(a - first, cnt, output_size=total) + torch.arange(total, device=self.device)
        seg_ids = self.row_seg[pos]
        return r32, slots.to(torch.int32).contiguous(), seg_ids.to(torch.int32).contiguous()

    # -- derived graphs -------------------------------------------------------------------------
    def with_values(self, val: torch.Tensor, symmetric: bool) -> "DeviceGraph":
        g = object.__new__(DeviceGraph)
        g.__dict__.update(self.__dict__)
        g.val = val
        g.symmetric = symmetric
        return g

    def transposed_values(self, val: torch.Tensor) -> torch.Tensor:
        """valT[e] = val[tpos[e]]: values of A^T laid out on the (symmetric) structure of A."""
        if self.tpos is None:
            raise RuntimeError("graph has no transpose map (tpos)")
        out = torch.empty_like(val)
        call("spex_gather_f32", ptr(val), ptr(self.tpos), None, 1.0, ptr(out), self.nnz, stream_ptr())
        return out

    def dropout_values(self, keep_mask: torch.Tensor, keep_prob: float) -> torch.Tensor:
        """val * mask / keep_prob as a per-nnz multiplier (model.py:46-55 in multiplier form)."""
        scale = keep_mask.to(self.device, torch.float32).contiguous()
        out = torch.empty_like(self.val)
        call("spex_gather_f32", ptr(self.val), None, ptr(scale), float(keep_prob), ptr(out), self.nnz,
             stream_ptr())
        return out

    def device_dropout_values(self, seed: int, keep_prob: float):
        """(val, valT) of the edge-dropped graph under the counter-based mask of spex_edge_dropout_f32: edge (r, c)
        is kept by a hash of (seed, global row, column), so no host random numbers and no mask copy.  Fresh
        tensors: autograd holds valT until the backward runs.  A row block (row_offset = its first global row) gives
        its slice of the whole graph's pair when it is bit-symmetric or was cut with CSRGraph.row_block(...,
        transposed_values=True)."""
        tpos = self.tpos if self.tpos is not None else self._tval_pos
        if tpos is None and not self.values_symmetric:
            raise RuntimeError("edge dropout needs the transpose map of the adjacency or bit-symmetric values; "
                               "build the graph through spex_b200.dataloader (getCSR) or synthetic.build_norm_adj_device")
        val = torch.empty_like(self.val)
        valT = torch.empty_like(self.val)
        call("spex_edge_dropout_f32", ptr(self.rowptr), ptr(self.col), ptr(self.val), ptr(tpos), self.n_rows,
             self.row_offset, int(seed), float(keep_prob), ptr(val), ptr(valT), stream_ptr())
        return val, valT

    def to_sparse_coo(self) -> torch.Tensor:
        deg = self.rowptr[1:] - self.rowptr[:-1]
        rows = torch.repeat_interleave(torch.arange(self.n_rows, device=self.device), deg)
        idx = torch.stack([rows + self.row_offset, self.clean_col().to(torch.int64)])
        return torch.sparse_coo_tensor(idx, self.val, (self.n_rows, self.n_cols), is_coalesced=True)


# ------------------------------------------------------------------------------------------------
def spmm(g: DeviceGraph, X: torch.Tensor, Y: Optional[torch.Tensor] = None,
         addend: Optional[torch.Tensor] = None, addend_scale: float = 1.0,
         Z: Optional[torch.Tensor] = None, z_scale: float = 1.0, val: Optional[torch.Tensor] = None):
    """One layer Y = A.X with the fused epilogue Z = (addend*addend_scale + A.X) * z_scale."""
    _need_cuda(X)
    X = _f32c(X)
    D = X.shape[1]
    if X.shape[0] != g.n_cols:
        raise ValueError(f"X has {X.shape[0]} rows, graph has {g.n_cols} columns")
    if Y is None and Z is None:
        Y = torch.empty(g.n_rows, D, dtype=torch.float32, device=X.device)
    v = g.val if val is None else val
    call("spex_spmm_csr_f32", ptr(g.rowptr), ptr(g.col), ptr(v), ptr(X), g.n_rows, D, ptr(Y),
         ptr(addend), float(addend_scale), ptr(Z), float(z_scale), g.plan(D), stream_ptr())
    return Y if Y is not None else Z


def nonzero_mask(n: int, rows: torch.Tensor) -> torch.Tensor:
    """uint8 [n], 1 on `rows`: the x_nonzero argument of spmm_rows (rows of X that may be non-zero)."""
    m = torch.zeros(n, dtype=torch.uint8, device=rows.device)
    m[rows] = 1
    return m


def spmm_rows(g: DeviceGraph, X: torch.Tensor, subset, Y: Optional[torch.Tensor] = None,
              addend: Optional[torch.Tensor] = None, addend_scale: float = 1.0,
              Z: Optional[torch.Tensor] = None, z_scale: float = 1.0, val: Optional[torch.Tensor] = None,
              x_nonzero: Optional[torch.Tensor] = None, out_row_offset: int = 0, y_mcast: Optional[int] = None,
              y_peers=None, pub_src: Optional[torch.Tensor] = None, pub_mcast: Optional[int] = None,
              pub_peers=None, adam: Optional[dict] = None, z_add: Optional[torch.Tensor] = None,
              z_add_rows: Optional[torch.Tensor] = None):
    """spmm() restricted to the rows of `subset` (= g.row_subset(rows); None = all rows): the listed rows of
    Y / Z get exactly the values a full layer gives them, the other rows are left untouched.  `x_nonzero`
    (uint8 [n_cols]): X is exactly zero on the rows it marks 0 - those gathers are skipped, the result is
    bit-identical.  The other arguments are the exchange epilogues of a row partition (spex_spmm_epilogue, whose
    rows out_row_offset + i they write): the Y rows to every rank's table through the multicast address `y_mcast`
    or the ctypes array of peer tables `y_peers`; the rows of `pub_src` (or, with `adam`, the updated rows of
    adam["p"]) likewise through `pub_mcast` / `pub_peers`; `adam` = {p, m, v, lr, beta1, beta2, eps, step}: dense
    Adam on the rows of p with the Z row as gradient; `z_add` (fp32 [n_rows, D]) with `z_add_rows` (uint8 [n_rows]):
    the flagged rows of Z / of Adam's gradient get z_add's row added after the scale (spex_spmm_layer_zadd_f32)."""
    _need_cuda(X)
    X = _f32c(X)
    D = X.shape[1]
    if X.shape[0] != g.n_cols:
        raise ValueError(f"X has {X.shape[0]} rows, graph has {g.n_cols} columns")
    if Y is None and Z is None and adam is None:
        raise ValueError("spmm_rows writes into caller-provided Y, Z or Adam state")
    rows, slots, segs = subset if subset is not None else (None, None, None)
    v = g.val if val is None else val
    if x_nonzero is not None and (x_nonzero.dtype != torch.uint8 or x_nonzero.numel() != g.n_cols):
        raise ValueError("x_nonzero must be uint8 [n_cols]")
    if z_add is not None and (z_add.dtype != torch.float32 or tuple(z_add.shape) != (g.n_rows, D)
                              or not z_add.is_contiguous() or z_add_rows is None or z_add_rows.dtype != torch.uint8
                              or z_add_rows.numel() != g.n_rows):
        raise ValueError("z_add must be contiguous fp32 [n_rows, D] with z_add_rows uint8 [n_rows]")
    ep = SpmmEpilogue(Y=ptr(Y), addend=ptr(addend), addend_scale=addend_scale, Z=ptr(Z), z_scale=z_scale,
                      out_row_offset=out_row_offset, y_mcast=y_mcast, y_peers_host=y_peers,
                      n_y_peers=0 if y_peers is None else len(y_peers), pub_src=ptr(pub_src), pub_mcast=pub_mcast,
                      pub_peers_host=pub_peers, n_pub_peers=0 if pub_peers is None else len(pub_peers))
    if adam is not None:
        ep.adam_p, ep.adam_m, ep.adam_v = ptr(adam["p"]), ptr(adam["m"]), ptr(adam["v"])
        ep.lr, ep.beta1, ep.beta2, ep.eps, ep.step = (adam["lr"], adam["beta1"], adam["beta2"], adam["eps"],
                                                     adam["step"])
    call("spex_spmm_layer_zadd_f32", ptr(g.rowptr), ptr(g.col), ptr(v), ptr(X), g.n_rows, D, ptr(rows),
         -1 if rows is None else rows.numel(), ptr(slots), 0 if slots is None else slots.numel(), ptr(segs),
         0 if segs is None else segs.numel(), ptr(x_nonzero), C.byref(ep), ptr(z_add), ptr(z_add_rows), g.plan(D),
         stream_ptr())


# A layer's input is treated as sparse (x_nonzero mask, gathers of zero rows skipped) while the rows that may be
# non-zero hold fewer than this fraction of nnz(A)
SPARSE_INPUT_MAX_EDGE_FRAC = 0.3
# A layer is restricted to a row list only while the list's edges stay below SUBSET_MAX_EDGE_FRAC of nnz(A)
# (beyond it the skipped rows no longer pay for the indirection), and a list is expanded to its neighbour set
# only while it has fewer than EXPAND_MAX_EDGE_FRAC * nnz(A) edges (the set is built by a gather + sort).
SUBSET_MAX_EDGE_FRAC = 0.5
EXPAND_MAX_EDGE_FRAC = 0.02


class ReceptivePlan:
    """receptive_plan's result.  R[k], k = 1..K: the rows of E^(k) that the rows S = R[K] of the layer mean depend
    on, or None = all rows; edges[k]: the edge count of R[k].  R[0] and edges[0] are None."""

    def __init__(self, K: int, nnz: int):
        self.R, self.edges, self.nnz = [None] * (K + 1), [None] * (K + 1), nnz

    def backward_layer(self, j: int):
        """(rows, x_rows) of backward layer j = 1..K.  H_j = g + A^T H_{j-1} is non-zero only on rows = R[K-j]
        (None = all; always for j = K).  x_rows = R[K-j+1], the rows of H_{j-1} that may be non-zero, is given only
        while they hold at most SPARSE_INPUT_MAX_EDGE_FRAC of nnz(A): the layer then skips the other rows' gathers."""
        k = len(self.R) - j
        sparse = self.edges[k] is not None and self.edges[k] <= SPARSE_INPUT_MAX_EDGE_FRAC * self.nnz
        return self.R[k - 1], (self.R[k] if sparse else None)


def receptive_plan(S: torch.Tensor, K: int, nnz: int, degree_sum, neighbors) -> ReceptivePlan:
    """The rows each layer computes when only the rows S (sorted unique int64 ids) of the layer mean are read:
    R[K] = S, R[k] = S + neighbours(R[k+1]), each set None = all rows from the first one that outgrows the limits
    on.  `degree_sum(rows) -> int` and `neighbors(rows) -> int64 ids` query one graph, or a row partition's blocks
    summed / gathered over the ranks; nnz = nnz(A)."""
    plan = ReceptivePlan(K, nnz)
    R, edges = plan.R, plan.edges
    if K < 1 or (d := degree_sum(S)) > SUBSET_MAX_EDGE_FRAC * nnz:
        return plan
    R[K], edges[K] = S, d
    for k in range(K - 1, 0, -1):
        if edges[k + 1] > EXPAND_MAX_EDGE_FRAC * nnz:
            break
        cand = torch.unique(torch.cat([S, neighbors(R[k + 1])]))
        d = degree_sum(cand)
        if d > SUBSET_MAX_EDGE_FRAC * nnz:
            break
        R[k], edges[k] = cand, d
    return plan


def receptive_rows(graph: DeviceGraph, S: torch.Tensor, K: int):
    """R[k], k = 1..K, of receptive_plan over `graph`."""
    return receptive_plan(S, K, graph.nnz, graph.degree_sum, graph.neighbors).R


class _PropagateMean(torch.autograd.Function):
    """out = mean_k A^k E0 over the fused [N, D] table (model.py:66-97), backward through A^T.

    With a ReceptivePlan whose R[K] is set (a training step whose loss reads only the rows S = R[K] of the
    result), every layer is computed on the rows the batch depends on with the same kernels and epilogues, so
    the rows S of `out`, the loss and dE0 are bit-identical to the full computation; the other rows of `out`
    are NOT valid.  Backward contract: the incoming gradient is then zero outside the rows S."""

    @staticmethod
    def forward(ctx, table, graph: DeviceGraph, K: int, val, valT, plan):
        _need_cuda(table)
        E0 = _f32c(table)
        N, D = E0.shape
        out = torch.empty_like(E0) if not workspaces.enabled else workspaces.get("prop_out", E0.shape, E0.device)[0]
        tmp = [workspaces.get("prop_tmp0", E0.shape, E0.device)[0] if K >= 2 else None,
               workspaces.get("prop_tmp1", E0.shape, E0.device)[0] if K >= 3 else None]
        v = graph.val if val is None else val
        # R[K] None: no layer is restricted and no backward input is masked - the two fused calls
        restricted = plan is not None and plan.R[K] is not None
        subs = [None if r is None else graph.row_subset(r) for r in plan.R] if restricted else None
        if subs is None:
            call("spex_propagate_mean_f32", ptr(graph.rowptr), ptr(graph.col), ptr(v), ptr(E0), N, D, K,
                 ptr(out), ptr(tmp[0]), ptr(tmp[1]), graph.plan(D), stream_ptr())
        else:
            inv = 1.0 / float(K + 1)
            X = E0
            for k in range(1, K + 1):
                last = k == K
                Y = None if last else tmp[(k - 1) & 1]
                kw = dict(Y=Y, addend=E0 if k == 1 else out, addend_scale=1.0, Z=out, z_scale=inv if last else 1.0,
                          val=v)
                if subs[k] is None:
                    spmm(graph, X, **kw)
                else:
                    spmm_rows(graph, X, subs[k], **kw)
                X = Y
        ctx.graph, ctx.K, ctx.valT, ctx.plan, ctx.subs = graph, K, (v if valT is None else valT), plan, subs
        return out

    @staticmethod
    def backward(ctx, g):
        graph, K, plan, subs = ctx.graph, ctx.K, ctx.plan, ctx.subs
        g = _f32c(g)
        N, D = g.shape
        dE0 = torch.empty_like(g) if not workspaces.enabled else workspaces.get("prop_dE0", g.shape, g.device)[0]
        tmp = [workspaces.get("prop_tmp0", g.shape, g.device)[0] if K >= 2 else None,
               workspaces.get("prop_tmp1", g.shape, g.device)[0] if K >= 3 else None]
        if subs is None:
            call("spex_propagate_mean_bwd_f32", ptr(graph.rowptr), ptr(graph.col), ptr(ctx.valT), ptr(g),
                 N, D, K, ptr(dE0), ptr(tmp[0]), ptr(tmp[1]), graph.plan(D), stream_ptr())
            return dE0, None, None, None, None, None
        inv = 1.0 / float(K + 1)
        # H_0 = g; H_j = g + A^T H_{j-1}: a restricted layer writes its rows into a zero table (zero-filled once;
        # afterwards only the rows of the previous step are cleared)
        X = g
        for j in range(1, K + 1):
            last = j == K
            kw = dict(addend=g, addend_scale=1.0, z_scale=inv if last else 1.0, val=ctx.valT)
            rows, x_rows = plan.backward_layer(j)
            mask = None if x_rows is None else nonzero_mask(N, x_rows)
            if rows is None:
                Z = dE0 if last else tmp[(j - 1) & 1]
                if mask is None:
                    spmm(graph, X, Z=Z, **kw)
                else:
                    spmm_rows(graph, X, None, Z=Z, x_nonzero=mask, **kw)
            else:
                Z, zkey = workspaces.get(f"prop_bwd_rows{j}", g.shape, g.device, zero=True)
                spmm_rows(graph, X, subs[K - j], Z=Z, x_nonzero=mask, **kw)
                workspaces.mark(zkey, rows)
            X = Z
        return dE0, None, None, None, None, None


def propagate_mean(table: torch.Tensor, graph: DeviceGraph, K: int,
                   val: Optional[torch.Tensor] = None, valT: Optional[torch.Tensor] = None,
                   rows_needed: Optional[torch.Tensor] = None):
    """K-layer propagation + layer mean.  `val` overrides the graph values (edge dropout); the
    backward then needs `valT` (values of the transposed matrix) unless the override is symmetric.
    `rows_needed` (int64 row ids): the caller reads - and back-propagates into - only these rows of the
    result; the layers are then restricted to the rows they depend on (receptive_plan)."""
    if graph.n_rows != graph.n_cols or table.shape[0] != graph.n_rows:
        raise ValueError("propagate_mean needs the full square adjacency and an [N, D] table")
    plan = None
    if rows_needed is not None and int(K) >= 1 and table.shape[1] in (32, 64, 128):
        plan = receptive_plan(torch.unique(_i64c(rows_needed, table.device)), int(K), graph.nnz, graph.degree_sum,
                              graph.neighbors)
    return _PropagateMean.apply(table, graph, int(K), val, valT, plan)


# ------------------------------------------------------------------------------------------------
class _GatherDot(torch.autograd.Function):
    """gamma[b] = <out[users[b]], out[n_user_rows + items[b]]>   (model.py:115-118)."""

    @staticmethod
    def forward(ctx, out, n_user_rows: int, users, items):
        _need_cuda(out)
        out = _f32c(out)
        D = out.shape[1]
        B = users.numel()
        gamma = torch.empty(B, dtype=torch.float32, device=out.device)
        U, I = out[:n_user_rows], out[n_user_rows:]
        call("spex_bce_fwd_f32", ptr(U), ptr(I), D, ptr(users), ptr(items), None, B, ptr(gamma), None,
             None, stream_ptr())
        ctx.save_for_backward(out, users, items)
        ctx.n_user_rows = n_user_rows
        return gamma

    @staticmethod
    def backward(ctx, dgamma):
        out, users, items = ctx.saved_tensors
        nur = ctx.n_user_rows
        D = out.shape[1]
        g, gkey = workspaces.get("grad_out", out.shape, out.device, zero=True)
        work, wb = _scatter_workspace(users.numel(), out.device)
        call("spex_bce_bwd_ws_f32", ptr(out[:nur]), ptr(out[nur:]), D, ptr(users), ptr(items),
             ptr(_f32c(dgamma)), None, users.numel(), ptr(g[:nur]), ptr(g[nur:]), ptr(work), wb, stream_ptr())
        workspaces.mark(gkey, users, items + nur)
        return g, None, None, None


class _BCELoss(torch.autograd.Function):
    """mean BCEWithLogits(<u,i>, label) with the dloss/dgamma produced in the same pass."""

    @staticmethod
    def forward(ctx, out, n_user_rows: int, users, items, labels):
        _need_cuda(out)
        out = _f32c(out)
        D = out.shape[1]
        B = users.numel()
        dev = out.device
        gamma = torch.empty(B, dtype=torch.float32, device=dev)
        dgamma = torch.empty(B, dtype=torch.float32, device=dev)
        loss = torch.empty(1, dtype=torch.float32, device=dev)
        U, I = out[:n_user_rows], out[n_user_rows:]
        call("spex_bce_fwd_f32", ptr(U), ptr(I), D, ptr(users), ptr(items), ptr(labels), B, ptr(gamma),
             ptr(loss), ptr(dgamma), stream_ptr())
        ctx.save_for_backward(out, users, items, dgamma)
        ctx.n_user_rows = n_user_rows
        ctx.mark_non_differentiable(gamma)
        return loss.reshape(()), gamma

    @staticmethod
    def backward(ctx, gloss, _ggamma):
        out, users, items, dgamma = ctx.saved_tensors
        nur = ctx.n_user_rows
        D = out.shape[1]
        # dense dL/d(out): zero except the rows of this batch (zero-filled once, see _Workspaces)
        g, gkey = workspaces.get("grad_out", out.shape, out.device, zero=True)
        gl = _f32c(gloss.reshape(1))
        work, wb = _scatter_workspace(users.numel(), out.device)
        call("spex_bce_bwd_ws_f32", ptr(out[:nur]), ptr(out[nur:]), D, ptr(users), ptr(items), ptr(dgamma),
             ptr(gl), users.numel(), ptr(g[:nur]), ptr(g[nur:]), ptr(work), wb, stream_ptr())
        workspaces.mark(gkey, users, items + nur)
        return g, None, None, None, None


def gather_dot(out, n_user_rows, users, items):
    dev = out.device
    return _GatherDot.apply(out, int(n_user_rows), _i64c(users, dev), _i64c(items, dev))


def bce_loss(out, n_user_rows, users, items, labels):
    dev = out.device
    if not torch.is_tensor(labels):
        labels = torch.as_tensor(np.asarray(labels))
    labels = labels.to(device=dev, dtype=torch.float32).contiguous()
    loss, _ = _BCELoss.apply(out, int(n_user_rows), _i64c(users, dev), _i64c(items, dev), labels)
    return loss


class _BPRLoss(torch.autograd.Function):
    """(mean softplus(<u,n>-<u,p>), 0.5*(|u0|^2+|p0|^2+|n0|^2)/B)  — north_star bpr_loss."""

    @staticmethod
    def forward(ctx, out, table, n_user_rows: int, users, pos, neg):
        _need_cuda(out, table)
        out, table = _f32c(out), _f32c(table)
        D = out.shape[1]
        B = users.numel()
        dev = out.device
        out2 = torch.empty(2, dtype=torch.float32, device=dev)
        dscore = torch.empty(B, dtype=torch.float32, device=dev)
        work = torch.empty(2 * B, dtype=torch.float32, device=dev)
        nur = n_user_rows
        call("spex_bpr_fwd_f32", ptr(out[:nur]), ptr(out[nur:]), ptr(table[:nur]), ptr(table[nur:]), D,
             ptr(users), ptr(pos), ptr(neg), B, ptr(out2), ptr(dscore), ptr(work), stream_ptr())
        ctx.save_for_backward(out, table, users, pos, neg, dscore)
        ctx.n_user_rows = nur
        return out2[0], out2[1]

    @staticmethod
    def backward(ctx, gloss, greg):
        out, table, users, pos, neg, dscore = ctx.saved_tensors
        nur = ctx.n_user_rows
        D = out.shape[1]
        g, gkey = workspaces.get("grad_out", out.shape, out.device, zero=True)
        g0, g0key = workspaces.get("grad_ego", table.shape, table.device, zero=True)
        grad2 = torch.stack([gloss.reshape(()), greg.reshape(())]).to(torch.float32).contiguous()
        work, wb = _scatter_workspace(2 * users.numel(), out.device)
        call("spex_bpr_bwd_ws_f32", ptr(out[:nur]), ptr(out[nur:]), ptr(table[:nur]), ptr(table[nur:]), D,
             ptr(users), ptr(pos), ptr(neg), ptr(dscore), ptr(grad2), users.numel(), ptr(g[:nur]),
             ptr(g[nur:]), ptr(g0[:nur]), ptr(g0[nur:]), ptr(work), wb, stream_ptr())
        workspaces.mark(gkey, users, pos + nur, neg + nur)
        workspaces.mark(g0key, users, pos + nur, neg + nur)
        return g, g0, None, None, None, None


def bpr_loss(out, table, n_user_rows, users, pos, neg):
    dev = out.device
    return _BPRLoss.apply(out, table, int(n_user_rows), _i64c(users, dev), _i64c(pos, dev),
                          _i64c(neg, dev))


# ------------------------------------------------------------------------------------------------
def score_candidates(U, I, users, cand):
    """score[u,c] = <U[users[u]], I[cand[u,c]]> for a dense [n_u, n_c] int32 candidate matrix."""
    _need_cuda(U, I)
    U, I = _f32c(U), _f32c(I)
    dev = U.device
    users = _i64c(users, dev)
    cand = cand.to(device=dev, dtype=torch.int32).contiguous()
    n_u, n_c = cand.shape
    score = torch.empty(n_u, n_c, dtype=torch.float32, device=dev)
    call("spex_score_candidates_f32", ptr(U), ptr(I), U.shape[1], ptr(users), ptr(cand), n_u, n_c,
         ptr(score), stream_ptr())
    return score


def score_topk_f32(U, I, users, k, mask_rowptr=None, mask_col=None, out_idx=None, out_val=None):
    """Exact fp32 full-ranking top-k (score desc, ties by ascending item id)."""
    _need_cuda(U, I)
    U, I = _f32c(U), _f32c(I)
    dev = U.device
    users = _i64c(users, dev)
    B = users.numel()
    idx = torch.empty(B, k, dtype=torch.int32, device=dev) if out_idx is None else out_idx
    val = torch.empty(B, k, dtype=torch.float32, device=dev) if out_val is None else out_val
    call("spex_score_topk_f32", ptr(U), ptr(I), U.shape[1], ptr(users), B, I.shape[0],
         ptr(mask_rowptr), ptr(mask_col), int(k), ptr(idx), ptr(val), stream_ptr())
    return idx, val


def rating_dense(U, I, users, apply_sigmoid: bool = True):
    """[B, m_items] ratings f(<U[users[b]], I[j]>) — the materialised getUsersRating."""
    _need_cuda(U, I)
    U, I = _f32c(U), _f32c(I)
    dev = U.device
    users = _i64c(users, dev)
    B, m = users.numel(), I.shape[0]
    out = torch.empty(B, m, dtype=torch.float32, device=dev)
    step = 8 * 65535
    for s in range(0, B, step):
        n = min(step, B - s)
        call("spex_rating_f32", ptr(U), ptr(I), U.shape[1], ptr(users[s:]), n, m,
             1 if apply_sigmoid else 0, ptr(out[s:]), stream_ptr())
    return out


def f16_filter_is_selective(U, I, users, n_users: int = 64, n_items: int = 8192, seed: int = 0) -> bool:
    """Probe for spex_score_topk_f16.  Its fp16-accumulated score only FILTERS: everything within 2 eps of a
    row's k-th best (eps = 2^-9 |u| max|v| at D = 64, 2^-8 at D = 128; the probe uses 2^-9) is re-scored
    exactly, one row at a time.  On tables whose scores are nearly equal across items - an untrained NGCF model, whose normalised layer outputs are almost parallel:
    measured 99 ms against 1.7 ms for random tables of the same shape and 7 ms for the exact fp32 scorer - that
    band holds most items and the filter degenerates.  The probe scores a sample (n_users x n_items, exact fp32,
    spex_rating_f32) and compares the band with the spread of each user's scores: selective iff the median of
    2 eps / (max - median score) stays below 0.1 (random / trained tables: ~0.01).  FullRanker(probe=True) falls
    back to the exact fp32 scorer otherwise; the result is the same ranking either way."""
    _need_cuda(U, I)
    dev = U.device
    users = _i64c(users, dev)
    if users.numel() == 0 or I.shape[0] < 64:
        return True
    g = torch.Generator(device=dev)
    g.manual_seed(seed)
    us = users[torch.randint(0, users.numel(), (min(n_users, users.numel()),), device=dev, generator=g)]
    it = torch.randint(0, I.shape[0], (min(n_items, I.shape[0]),), device=dev, generator=g)
    Is = I[it].contiguous()
    s = rating_dense(U, Is, us, apply_sigmoid=False)
    spread = s.max(dim=1).values - s.median(dim=1).values
    eps = (1.0 / 512.0) * U[us].norm(dim=1) * Is.norm(dim=1).max()
    ratio = 2.0 * eps / spread.clamp_min(1e-30)
    return bool(ratio.median() < 0.1)


TC_USER_MULTIPLE = 128   # users per CTA of the tcgen05 scorer (UMMA M)
TC_MAX_K = 64            # larger k: score_topk_f16_wide (or score_topk_f32 up to F32_MAX_K)
F32_MAX_K = 128          # k limit of score_topk_f32
WIDE_MAX_K = 512         # k limit of score_topk_f16_wide
TC_ITEM_MULTIPLE = 128   # items per tile (UMMA N)
# precision -> (the D its full-ranking scorer is built for, None: any; its largest k).  f16 ranks k <= TC_MAX_K with
# score_topk_f16 and larger k with score_topk_f16_wide.
SCORER_LIMITS = {"f16": ((64, 128), WIDE_MAX_K), "bf16": ((64,), TC_MAX_K), "fp32": (None, F32_MAX_K)}


def default_precision(D: int) -> str:
    """The full-ranking precision for D: "f16" where its scorer is built for D, else "fp32" (any D)."""
    return "f16" if D in SCORER_LIMITS["f16"][0] else "fp32"


def pack_bf16(src, rows=None, row_multiple: int = 8, out=None):
    """fp32 [n, D] (optionally gathered by `rows`) -> bf16 UMMA core-matrix layout, zero padded."""
    _need_cuda(src)
    src = _f32c(src)
    dev = src.device
    n = src.shape[0] if rows is None else rows.numel()
    D = src.shape[1]
    n_pad = (n + row_multiple - 1) // row_multiple * row_multiple
    if out is None:
        out = torch.empty(n_pad * D, dtype=torch.bfloat16, device=dev)
    elif out.numel() < n_pad * D:
        raise ValueError("pack_bf16: output buffer too small")
    rows_t = None if rows is None else _i64c(rows, dev)
    call("spex_pack_bf16", ptr(src), ptr(rows_t), n, n_pad, D, ptr(out), stream_ptr())
    return out, n_pad


def score_topk_bf16(Ub, B, B_pad, Ib, m_items, m_pad, k, user_ids=None, mask_rowptr=None,
                    mask_col=None, out_idx=None, out_val=None):
    """tcgen05 bf16 scoring GEMM fused with train-item masking and per-row top-k (D = 64)."""
    _need_cuda(Ub, Ib)
    max_k = SCORER_LIMITS["bf16"][1]
    if not 1 <= k <= max_k:
        raise ValueError(f"score_topk_bf16: k must be in [1, {max_k}] (use score_topk_f32 beyond)")
    dev = Ub.device
    if out_idx is None:
        out_idx = torch.empty(B, k, dtype=torch.int32, device=dev)
    if out_val is None:
        out_val = torch.empty(B, k, dtype=torch.float32, device=dev)
    uid = None if user_ids is None else _i64c(user_ids, dev)
    call("spex_score_topk_bf16", ptr(Ub), ptr(Ib), B, B_pad, m_items, m_pad, ptr(uid),
         ptr(mask_rowptr), ptr(mask_col), int(k), ptr(out_idx), ptr(out_val), stream_ptr())
    return out_idx, out_val


def pack_f16(src, rows=None, row_multiple: int = 8, out=None):
    """fp32 [n, D] (optionally gathered by `rows`) -> scaled fp16 UMMA layout + its meta (scale,
    1/scale, max scaled row norm, max row norm^2): the operands of score_topk_f16."""
    _need_cuda(src)
    src = _f32c(src)
    dev = src.device
    n = src.shape[0] if rows is None else rows.numel()
    D = src.shape[1]
    n_pad = (n + row_multiple - 1) // row_multiple * row_multiple
    if out is None:
        out = torch.empty(n_pad * D, dtype=torch.float16, device=dev)
    elif out.numel() < n_pad * D:
        raise ValueError("pack_f16: output buffer too small")
    meta = torch.empty(4, dtype=torch.float32, device=dev)
    rows_t = None if rows is None else _i64c(rows, dev)
    call("spex_pack_f16", ptr(src), ptr(rows_t), n, n_pad, D, ptr(out), ptr(meta), stream_ptr())
    return out, n_pad, meta


def score_topk_f16(Uh, u_meta, B, B_pad, Ih, i_meta, m_items, m_pad, D, k, user_ids=None,
                   mask_rowptr=None, mask_col=None, out_idx=None, out_val=None):
    """tcgen05 fp16-accumulator filter + exact fp32 re-score, fused mask + per-row top-k
    (D = 64 or 128; NGCF_SPEX/code/utility/batch_test.py:158 semantics + ranking)."""
    return _score_topk_f16(False, Uh, u_meta, B, B_pad, Ih, i_meta, m_items, m_pad, D, k, user_ids, mask_rowptr,
                           mask_col, out_idx, out_val)


def score_topk_f16_wide(Uh, u_meta, B, B_pad, Ih, i_meta, m_items, m_pad, D, k, user_ids=None,
                        mask_rowptr=None, mask_col=None, out_idx=None, out_val=None):
    """score_topk_f16 for 1 <= k <= WIDE_MAX_K: the same operands and output contract, each user row's
    candidate buffer in a device workspace (allocated here, B_pad * (2k + 64) * 8 bytes) instead of shared
    memory."""
    return _score_topk_f16(True, Uh, u_meta, B, B_pad, Ih, i_meta, m_items, m_pad, D, k, user_ids, mask_rowptr,
                           mask_col, out_idx, out_val)


def _score_topk_f16(wide, Uh, u_meta, B, B_pad, Ih, i_meta, m_items, m_pad, D, k, user_ids, mask_rowptr, mask_col,
                    out_idx, out_val):
    name = "score_topk_f16_wide" if wide else "score_topk_f16"
    _need_cuda(Uh, Ih)
    dims, max_k = SCORER_LIMITS["f16"][0], SCORER_LIMITS["f16"][1] if wide else TC_MAX_K
    if not 1 <= k <= max_k:
        raise ValueError(f"{name}: k must be in [1, {max_k}]" + ("" if wide else " (use score_topk_f32 beyond)"))
    if D not in dims:
        raise ValueError(f"{name}: D must be 64 or 128 (use score_topk_f32 otherwise)")
    dev = Uh.device
    if out_idx is None:
        out_idx = torch.empty(B, k, dtype=torch.int32, device=dev)
    if out_val is None:
        out_val = torch.empty(B, k, dtype=torch.float32, device=dev)
    uid = None if user_ids is None else _i64c(user_ids, dev)
    args = (ptr(Uh), ptr(Ih), int(D), B, B_pad, m_items, m_pad, ptr(u_meta), ptr(i_meta), ptr(uid), ptr(mask_rowptr),
            ptr(mask_col), int(k), ptr(out_idx), ptr(out_val))
    if wide:
        nbytes = int(call("spex_score_topk_f16_wide_workspace_bytes", int(B_pad), int(k)))
        work = torch.empty(max(nbytes, 16), dtype=torch.uint8, device=dev)
        call("spex_score_topk_f16_wide", *args, ptr(work), nbytes, stream_ptr())
    else:
        call("spex_score_topk_f16", *args, stream_ptr())
    return out_idx, out_val


def rank_pairs_f16(Uh, a_rows, user_ids, items, Ih, i_meta, m_items, m_pad, D, mask_rowptr=None, mask_col=None,
                   out=None):
    """Rank of each held-out pair (user row a_rows[p] of the packed table Uh, item items[p]) among the items outside
    mask row user_ids[p], under the exact score of the f16 scorer (spex_rank_pairs_f16): int32 [P]."""
    _need_cuda(Uh, Ih)
    if D not in SCORER_LIMITS["f16"][0]:
        raise ValueError("rank_pairs_f16: D must be 64 or 128 (use rank_pairs_f32 otherwise)")
    dev = Uh.device
    items = items.to(device=dev, dtype=torch.int32).contiguous()
    P = items.numel()
    out = torch.empty(P, dtype=torch.int32, device=dev) if out is None else out
    p_pad = (P + TC_USER_MULTIPLE - 1) // TC_USER_MULTIPLE * TC_USER_MULTIPLE
    a_rows = None if a_rows is None else _i64c(a_rows, dev)
    user_ids = None if user_ids is None else _i64c(user_ids, dev)
    call("spex_rank_pairs_f16", ptr(Uh), ptr(Ih), int(D), ptr(a_rows), ptr(user_ids),
         ptr(items), P, p_pad, int(m_items), int(m_pad), ptr(i_meta), ptr(mask_rowptr), ptr(mask_col), ptr(out),
         stream_ptr())
    return out


def rank_pairs_f32(U, I, users, items, mask_rowptr=None, mask_col=None, out=None):
    """Rank of each held-out pair (U[users[p]], item items[p]) among the items outside mask row users[p], under the
    exact fp32 score of score_topk_f32 (spex_rank_pairs_f32): int32 [P]."""
    _need_cuda(U, I)
    U, I = _f32c(U), _f32c(I)
    dev = U.device
    users = _i64c(users, dev)
    items = items.to(device=dev, dtype=torch.int32).contiguous()
    out = torch.empty(items.numel(), dtype=torch.int32, device=dev) if out is None else out
    call("spex_rank_pairs_f32", ptr(U), ptr(I), U.shape[1], ptr(users), ptr(items), items.numel(), I.shape[0],
         ptr(mask_rowptr), ptr(mask_col), ptr(out), stream_ptr())
    return out


def check_k(precision: str, k: int):
    """ValueError unless `precision` serves top-`k` (SCORER_LIMITS); the message names the precision that serves a k
    beyond the limit."""
    limit, wide = SCORER_LIMITS[precision][1], SCORER_LIMITS["f16"][1]
    if not 1 <= k <= limit:
        hint = f"; precision 'f16' serves k <= {wide}" if precision != "f16" and 1 <= k <= wide else ""
        raise ValueError(f"precision '{precision}' serves 1 <= k <= {limit}, got k = {k}{hint}")


class FullRanker:
    """Full-ranking top-k of user rows against one item table, (idx int32 [B, k], score fp32 [B, k]): score
    descending, ties by ascending item id, the items of each user's mask row excluded.

    precision "f16":  tcgen05 fp16-accumulator filter + exact fp32 re-score (D 64 or 128): score_topk_f16 for
                      k <= TC_MAX_K, score_topk_f16_wide up to WIDE_MAX_K;
    precision "bf16": tcgen05 bf16 operands / fp32 accumulators (score_topk_bf16; D = 64; k <= TC_MAX_K);
    precision "fp32": exact CUDA-core scorer (score_topk_f32; any D; k <= F32_MAX_K).
    probe=True lets the near-tie probe send "f16" rankings to "fp32" (scorer_for): the one place where any caller's
    scorer is chosen.  The item table is packed on the first call that needs it packed (the fp32 scorer reads it as
    it is); the users are packed per call."""

    def __init__(self, I_all, precision: str = "f16", probe: bool = False):
        if precision not in SCORER_LIMITS:
            raise ValueError("precision must be 'f16', 'bf16' or 'fp32'")
        dims = SCORER_LIMITS[precision][0]
        if dims is not None and I_all.shape[1] not in dims:
            built = " or ".join(map(str, dims)) if len(dims) > 1 else f"== {dims[0]}"
            raise RuntimeError(f"the {precision} tcgen05 scorer is built for recdim {built}")
        self.precision, self.probe, self.device = precision, probe, I_all.device
        self.m_items, self.D = I_all.shape
        self._I, self._m_pad = I_all, None      # _m_pad: set when the item table is packed

    def scorer_for(self, k, U_all, probe_users) -> str:
        """The precision that ranks top-k: ValueError unless this ranker's precision serves k (check_k).  With
        probe=True, "f16" becomes "fp32" for k <= F32_MAX_K when f16_filter_is_selective(U_all, I_all, probe_users)
        is False: near-equal scores, on which the exact scorer is the faster exact path (above F32_MAX_K only the
        f16 scorer serves k).

        k=None asks for the precision of a rank query (ranks, rank_metrics), which has no k: "f16" (turned into
        "fp32" by the same probe when probe=True) or "fp32"; ValueError for "bf16", which has no rank kernel."""
        if k is None:
            if self.precision == "bf16":
                raise ValueError("precision 'bf16' has no rank kernel; use 'f16' or 'fp32'")
            if (self.precision == "f16" and self.probe
                    and not f16_filter_is_selective(U_all, self._I, probe_users)):
                return "fp32"
            return self.precision
        check_k(self.precision, k)
        if (self.precision == "f16" and self.probe and k <= F32_MAX_K
                and not f16_filter_is_selective(U_all, self._I, probe_users)):
            return "fp32"
        return self.precision

    def topk(self, U_all, users, k, mask_rowptr=None, mask_col=None, user_block=None, probe_users=None):
        """Rank U_all[users] in blocks of `user_block` users (None: one block) with the scorer of
        scorer_for(k, U_all, probe_users) (None: `users`).

        f16: the result does not depend on `user_block`.  The users of the call are packed once, so one user
        scale 2^s, chosen over all of them, rounds every user's operands (a per-block scale would round a user's
        fp16 subnormal components differently depending on its block-mates); each block is a slice of that
        buffer, `user_block` rounded up to a multiple of 128 rows."""
        users = _i64c(users, self.device)
        scorer = self.scorer_for(k, U_all, users if probe_users is None else probe_users)
        B = users.numel()
        idx = torch.empty(B, k, dtype=torch.int32, device=self.device)
        val = torch.empty(B, k, dtype=torch.float32, device=self.device)
        for _ in self._ranked_blocks(scorer, U_all, users, k, mask_rowptr, mask_col, user_block or max(B, 1),
                                     lambda s, n: (idx[s: s + n], val[s: s + n])):
            pass
        return idx, val

    def _pack_items(self, scorer):
        """Pack the item table for `scorer` ("f16" or "bf16", this ranker's precision) on the first call that needs
        it: self._Ih / self._imeta or self._Ib, and self._m_pad."""
        if self._m_pad is not None:
            return
        if scorer == "f16":
            self._Ih, self._m_pad, self._imeta = pack_f16(self._I, None, TC_ITEM_MULTIPLE)
        else:
            self._Ib, self._m_pad = pack_bf16(self._I, None, TC_ITEM_MULTIPLE)

    def _ranked_blocks(self, scorer, U_all, users, k, mask_rowptr, mask_col, step, dest):
        """Rank users[s: s + step] for s = 0, step, 2 step, ... with `scorer` into the (idx, val) [n, k] views
        dest(s, n) and yield (s, idx view) after each block's launches."""
        m, D = self.m_items, self.D
        B = users.numel()
        if scorer != "fp32":
            self._pack_items(scorer)
        if scorer == "f16":
            step = (step + TC_USER_MULTIPLE - 1) // TC_USER_MULTIPLE * TC_USER_MULTIPLE
            if B:
                Uh_all, _, umeta = pack_f16(U_all, users, TC_USER_MULTIPLE)
        for s in range(0, B, step):
            ub = users[s: s + step]
            o_i, o_v = dest(s, ub.numel())
            if scorer == "f16":
                # the canonical layout keeps every 8-row group contiguous: rows [s, s + b_pad) are one slice
                b_pad = (ub.numel() + TC_USER_MULTIPLE - 1) // TC_USER_MULTIPLE * TC_USER_MULTIPLE
                Uh = Uh_all[s * D: (s + b_pad) * D]
                f16 = score_topk_f16 if k <= TC_MAX_K else score_topk_f16_wide
                f16(Uh, umeta, ub.numel(), b_pad, self._Ih, self._imeta, m, self._m_pad, D, k, ub, mask_rowptr,
                    mask_col, o_i, o_v)
            elif scorer == "bf16":
                Ub, b_pad = pack_bf16(U_all, ub, TC_USER_MULTIPLE)
                score_topk_bf16(Ub, ub.numel(), b_pad, self._Ib, m, self._m_pad, k, ub, mask_rowptr, mask_col,
                                o_i, o_v)
            else:
                score_topk_f32(U_all, self._I, ub, k, mask_rowptr, mask_col, o_i, o_v)
            yield s, o_i

    def metric_sums(self, U_all, users, cutoffs, truth_rowptr, truth_col, mask_rowptr=None, mask_col=None,
                    user_block=None, per_user=False, probe_users=None):
        """(sums fp64 [n_cut, 4], per-user fp64 [B, n_cut, 4] or None) of evaluate(), on the device; the last
        axis is METRIC_NAMES.  The sums are over users, each chunk of METRICS_CHUNK users summed on its own and
        the chunks in ascending order, so they do not depend on `user_block`."""
        cutoffs = check_cutoffs(cutoffs)
        k = cutoffs[-1]
        dev = self.device
        users = _i64c(users, dev)
        B = users.numel()
        trp, tcol = self._truth_csr(truth_rowptr, truth_col, B)
        scorer = self.scorer_for(k, U_all, users if probe_users is None else probe_users)
        if tcol.numel() == 0:
            tcol = torch.zeros(1, dtype=torch.int32, device=dev)   # all rows empty: never read, but not NULL
        n_cut = len(cutoffs)
        cut_host = (C.c_int32 * n_cut)(*cutoffs)
        disc, idcg = rank_discounts(k)
        disc = torch.from_numpy(disc).to(dev)
        idcg = torch.from_numpy(idcg).to(dev)
        step = user_block or EVAL_USER_BLOCK
        step = (step + METRICS_CHUNK - 1) // METRICS_CHUNK * METRICS_CHUNK     # also a multiple of TC_USER_MULTIPLE
        n_chunks = (B + METRICS_CHUNK - 1) // METRICS_CHUNK
        chunk_sums = torch.empty(n_chunks, n_cut, 4, dtype=torch.float64, device=dev)
        pu = torch.empty(B, n_cut, 4, dtype=torch.float64, device=dev) if per_user else None
        nb = min(step, B)
        bi = torch.empty(nb, k, dtype=torch.int32, device=dev)      # one [block, k] buffer for every block
        bv = torch.empty(nb, k, dtype=torch.float32, device=dev)
        for s, o_i in self._ranked_blocks(scorer, U_all, users, k, mask_rowptr, mask_col, step,
                                          lambda s, n: (bi[:n], bv[:n])):
            n = o_i.shape[0]
            call("spex_fullrank_metrics", ptr(o_i), n, k, ptr(trp[s:]), ptr(tcol), cut_host, n_cut, ptr(disc),
                 ptr(idcg), ptr(None if pu is None else pu[s:]), ptr(chunk_sums[s // METRICS_CHUNK:]), stream_ptr())
        return _reduce_chunks(chunk_sums, n_cut), pu

    def evaluate(self, U_all, users, cutoffs, truth_rowptr, truth_col, mask_rowptr=None, mask_col=None,
                 user_block=None, per_user=False, probe_users=None):
        """Recall, precision, NDCG and hit rate of the full ranking of U_all[users] at each of `cutoffs` (1 to 8
        strictly ascending k): {"recall", "precision", "ndcg", "hit": float64 [n_cut], "users": B}, means over all
        B users (an empty truth row counts as zeros), and with per_user=True "per_user": fp64 [B, n_cut, 4] on the
        device (last axis METRIC_NAMES).  Definitions of metrics.fullrank_recall_ndcg, precision = hits / K.

        truth_rowptr int64 [B + 1] / truth_col: the held-out items as a CSR over the POSITIONS in `users`, every
        row ascending (ValueError otherwise; graph.truth_csr builds one).  The users are ranked at
        k = max(cutoffs) by the scorer topk() would use (probe_users as there), in blocks of `user_block` users
        rounded up to a multiple of METRICS_CHUNK (None: EVAL_USER_BLOCK); each block's ids stay on the device in
        one reused [block, k] buffer and go straight into spex_fullrank_metrics.  The result does not depend on
        `user_block`."""
        users = _i64c(users, self.device)
        sums, pu = self.metric_sums(U_all, users, cutoffs, truth_rowptr, truth_col, mask_rowptr, mask_col,
                                    user_block, per_user, probe_users)
        return metric_means(sums.cpu().numpy(), users.numel(), pu)

    def _truth_csr(self, truth_rowptr, truth_col, B):
        """(rowptr int64, col int32) of a truth CSR over B users on the device; ValueError unless check_truth_csr
        accepts it."""
        trp = _i64c(truth_rowptr, self.device)
        tcol = torch.as_tensor(np.asarray(truth_col) if not torch.is_tensor(truth_col) else truth_col)
        tcol = tcol.to(device=self.device, dtype=torch.int32).contiguous()
        check_truth_csr(trp, tcol, B)
        return trp, tcol

    def _check_items(self, items):
        items = torch.as_tensor(items).to(device=self.device, dtype=torch.int64)
        if items.numel() and bool((items.min() < 0) | (items.max() >= self.m_items)):
            raise ValueError(f"item ids must lie in [0, {self.m_items})")
        return items.to(torch.int32).contiguous()

    def _rank(self, scorer, U_all, urows, a_rows, pair_users, items, mask_rowptr, mask_col):
        """Ranks of the pairs (U_all[pair_users[p]], items[p]) with `scorer`, in launches of RANK_PAIR_BLOCK pairs.
        f16: the users `urows` are packed once (one scale 2^s over all of them, as topk() packs its users) and
        pair p reads packed row a_rows[p]."""
        P = items.numel()
        out = torch.empty(P, dtype=torch.int32, device=self.device)
        if P == 0:
            return out
        if scorer == "f16":
            self._pack_items(scorer)
            Uh, _, _ = pack_f16(U_all, urows)
        for s in range(0, P, RANK_PAIR_BLOCK):
            e = min(s + RANK_PAIR_BLOCK, P)
            if scorer == "f16":
                rank_pairs_f16(Uh, a_rows[s:e], pair_users[s:e], items[s:e], self._Ih, self._imeta, self.m_items,
                               self._m_pad, self.D, mask_rowptr, mask_col, out[s:e])
            else:
                rank_pairs_f32(U_all, self._I, pair_users[s:e], items[s:e], mask_rowptr, mask_col, out[s:e])
        return out

    def ranks(self, U_all, users, items, mask_rowptr=None, mask_col=None, probe_users=None):
        """Rank of item items[p] for user users[p], int32 [P] on the device: the number of items outside the user's
        mask row, other than items[p], that come before it in the order of topk() (score descending, ties by
        ascending id) under the exact score of scorer_for(None, U_all, probe_users) (None: `users`).  It is the
        item's position in topk(...) when the item is listed there, >= k otherwise; a masked item still has one.
        ValueError for an item outside [0, m_items).  The result does not depend on RANK_PAIR_BLOCK."""
        users = _i64c(users, self.device)
        items = self._check_items(items)
        if users.numel() != items.numel():
            raise ValueError(f"{users.numel()} users but {items.numel()} items")
        scorer = self.scorer_for(None, U_all, users if probe_users is None else probe_users)
        if scorer == "f16" and users.numel():
            urows, a_rows = torch.unique(users, return_inverse=True)
        else:
            urows, a_rows = users, None
        return self._rank(scorer, U_all, urows, a_rows, users, items, mask_rowptr, mask_col)

    def rank_metrics(self, U_all, users, cutoffs, truth_rowptr, truth_col, mask_rowptr=None, mask_col=None,
                     probe_users=None):
        """Recall, precision, NDCG and hit rate at `cutoffs` (1 to 8 strictly ascending K, 1 <= K <= m_items), MRR
        and AUC of the full ranking of U_all[users], from the rank of every held-out item (ranks()):
        {"recall", "precision", "ndcg", "hit": float64 [n_cut], "mrr", "auc": float, "users": B}.

        The truth CSR is evaluate()'s; so are the definitions, with "rank < K" for "in the top K": a held-out item
        in the user's mask is never a hit.  MRR = 1 / (1 + the best rank among the user's hits), AUC = the mean over
        the held-out items of the fraction of the user's negatives (items outside the mask and the truth row) that
        score below the item (1 when the user has no negative; 0 for a masked item); spex_rank_metrics has the
        exact rules.  Means over all users, an empty truth row counting as zeros.  The users are packed as
        evaluate() packs them, so the ranks are the positions evaluate() ranks by; sums run per chunk of
        METRICS_CHUNK users in a fixed order on the device."""
        cutoffs = check_cutoffs(cutoffs)
        if cutoffs[-1] > self.m_items:
            raise ValueError(f"cutoffs must be <= m_items = {self.m_items}, got {cutoffs[-1]}")
        dev = self.device
        users = _i64c(users, dev)
        B = users.numel()
        trp, tcol = self._truth_csr(truth_rowptr, truth_col, B)
        scorer = self.scorer_for(None, U_all, users if probe_users is None else probe_users)
        a = int(trp[0]) if B else 0
        tcol = self._check_items(tcol[a: int(trp[-1])] if B else tcol[:0])
        trp = (trp - a).contiguous()
        pos = torch.repeat_interleave(torch.arange(B, device=dev), trp[1:] - trp[:-1])
        ranks = self._rank(scorer, U_all, users, pos, users[pos], tcol, mask_rowptr, mask_col)
        n_cut = len(cutoffs)
        disc, idcg = rank_discounts(cutoffs[-1])
        disc = torch.from_numpy(disc).to(dev)
        idcg = torch.from_numpy(idcg).to(dev)
        n_chunks = (B + METRICS_CHUNK - 1) // METRICS_CHUNK
        chunk_sums = torch.empty(n_chunks, n_cut, 4, dtype=torch.float64, device=dev)
        chunk_extra = torch.empty(n_chunks, 4, dtype=torch.float64, device=dev)
        if tcol.numel() == 0:
            tcol = torch.zeros(1, dtype=torch.int32, device=dev)       # all rows empty: never read, but not NULL
            ranks = torch.zeros(1, dtype=torch.int32, device=dev)
        call("spex_rank_metrics", ptr(ranks), B, ptr(trp), ptr(tcol), ptr(users), ptr(mask_rowptr), ptr(mask_col),
             self.m_items, (C.c_int32 * n_cut)(*cutoffs), n_cut, ptr(disc), ptr(idcg), ptr(chunk_sums),
             ptr(chunk_extra), stream_ptr())
        sums, extra = _reduce_chunks(chunk_sums, n_cut), _reduce_chunks(chunk_extra, 1)
        out = metric_means(sums.cpu().numpy(), B)
        ex = extra.cpu().numpy()[0] / max(float(B), 1.0)
        out["mrr"], out["auc"] = float(ex[0]), float(ex[1])
        return out


METRICS_CHUNK = 1024           # SPEX_METRICS_CHUNK in include/spex_b200.h: users per partial sum
METRICS_MAX_CUTOFFS = 8        # SPEX_METRICS_MAX_CUTOFFS
METRIC_NAMES = ("recall", "precision", "ndcg", "hit")
EVAL_USER_BLOCK = 148 * METRICS_CHUNK   # users ranked per block by FullRanker.evaluate (None)
RANK_PAIR_BLOCK = 1 << 22      # pairs per rank launch of FullRanker.ranks / rank_metrics


def _reduce_chunks(chunk_sums, n_cut):
    """fp64 [n_cut, 4]: the [n_chunks, n_cut, 4] chunk sums summed over the chunks in ascending order, on the
    device."""
    sums = torch.empty(n_cut, 4, dtype=torch.float64, device=chunk_sums.device)
    call("spex_fullrank_metrics_reduce", ptr(chunk_sums), chunk_sums.shape[0], n_cut, ptr(sums), stream_ptr())
    return sums


def check_cutoffs(cutoffs):
    """The cutoffs as a list of ints; ValueError unless 1 to METRICS_MAX_CUTOFFS of them, strictly ascending, >= 1."""
    cutoffs = [int(c) for c in cutoffs]
    if not 1 <= len(cutoffs) <= METRICS_MAX_CUTOFFS:
        raise ValueError(f"1 to {METRICS_MAX_CUTOFFS} cutoffs, got {len(cutoffs)}")
    if cutoffs[0] < 1 or any(b <= a for a, b in zip(cutoffs, cutoffs[1:])):
        raise ValueError(f"cutoffs must be >= 1 and strictly ascending, got {cutoffs}")
    return cutoffs


def rank_discounts(k: int):
    """(disc fp64 [k], idcg fp64 [k + 1]) of spex_fullrank_metrics, computed as metrics.fullrank_recall_ndcg
    computes its disc and cum: the ideal DCGs are bit-equal to the host's by construction."""
    disc = 1.0 / np.log2(np.arange(2, k + 2))
    return disc, np.concatenate([[0.0], np.cumsum(disc)])


def check_truth_csr(truth_rowptr: torch.Tensor, truth_col: torch.Tensor, B: int):
    """ValueError unless truth_rowptr (int64 [B + 1]) is non-decreasing inside [0, len(truth_col)] and every row
    of truth_col is ascending: the kernel's binary search relies on it.  Checked on the device."""
    if truth_rowptr.numel() != B + 1:
        raise ValueError(f"truth_rowptr must have {B + 1} entries (users + 1), got {truth_rowptr.numel()}")
    if B == 0:
        return
    rp = truth_rowptr
    if bool((rp[1:] < rp[:-1]).any() | (rp[0] < 0) | (rp[-1] > truth_col.numel())):
        raise ValueError("truth_rowptr must be non-decreasing and inside truth_col")
    a, b = int(rp[0]), int(rp[-1])
    if b - a < 2:
        return
    c = truth_col[a:b]
    starts = rp[:-1]
    first = torch.zeros(b - a, dtype=torch.bool, device=c.device)
    first[starts[starts < b] - a] = True
    if bool(((c[1:] < c[:-1]) & ~first[1:]).any()):
        raise ValueError("every truth row must be sorted ascending (graph.build_interaction_csr sorts)")


def metric_means(sums: np.ndarray, n_users: int, per_user=None) -> dict:
    """The result dict of FullRanker.evaluate from metric sums [n_cut, 4] over n_users users."""
    mean = np.asarray(sums, dtype=np.float64).reshape(-1, 4) / max(float(n_users), 1.0)
    out = {name: mean[:, j].copy() for j, name in enumerate(METRIC_NAMES)}
    out["users"] = int(n_users)
    if per_user is not None:
        out["per_user"] = per_user
    return out


GATE_BWD_BLOCKS = 1184  # SPEX_GATE_BWD_BLOCKS in include/spex_b200.h


class _ExpertGate(torch.autograd.Function):
    """out = a0*E0 + a1*Eout, a = softmax([E0|Eout].W) per row (model_expert_s.py:154-161)."""

    @staticmethod
    def forward(ctx, E0, Eout, W):
        _need_cuda(E0, Eout, W)
        E0, Eout, W = _f32c(E0), _f32c(Eout), _f32c(W)
        out = torch.empty_like(E0)
        call("spex_expert_gate_f32", ptr(E0), ptr(Eout), ptr(W), E0.shape[0], E0.shape[1], ptr(out),
             stream_ptr())
        ctx.save_for_backward(E0, Eout, W)
        return out

    @staticmethod
    def backward(ctx, g):
        E0, Eout, W = ctx.saved_tensors
        g = _f32c(g)
        dE0, dE1 = torch.empty_like(E0), torch.empty_like(Eout)
        dW = torch.empty_like(W)
        work = torch.empty(GATE_BWD_BLOCKS * 512, dtype=torch.float32, device=E0.device)
        call("spex_expert_gate_bwd_f32", ptr(E0), ptr(Eout), ptr(W), ptr(g), E0.shape[0], E0.shape[1],
             ptr(dE0), ptr(dE1), ptr(dW), ptr(work), stream_ptr())
        return dE0, dE1, dW


def expert_gate(E0, Eout, W):
    """softmax([E0|Eout].W) convex mix per row (model_expert_s.py:154-161), differentiable.

    The reference multiplies cat([E0, Eout], 1) [n, 2D] by att_exp [2*hiddenSize, 2]
    (model_expert_s.py:158-161) and raises a shape error when hiddenSize != recdim; so do we.
    """
    D = E0.shape[1]
    if E0.shape != Eout.shape:
        raise ValueError(f"expert_gate: E0 {tuple(E0.shape)} and Eout {tuple(Eout.shape)} differ")
    if tuple(W.shape) != (2 * D, 2):
        raise ValueError(f"expert_gate: gate weights must be [{2 * D}, 2] (2*recdim x 2), got {tuple(W.shape)}")
    if D > 128 or D % 4:
        raise ValueError("expert_gate: recdim must be a multiple of 4 and <= 128")
    return _ExpertGate.apply(E0, Eout, W)


def adam_step(p, g, m, v, lr, beta1, beta2, eps, step):
    """In-place dense Adam over one flat fp32 table (torch.optim.Adam arithmetic)."""
    _need_cuda(p, g, m, v)
    call("spex_adam_f32", ptr(p), ptr(_f32c(g)), ptr(m), ptr(v), p.numel(), float(lr), float(beta1),
         float(beta2), float(eps), int(step), stream_ptr())


def ngcf_epilogue(ego, side, W1, b1, W2, b2, negative_slope, out=None, norm=None, norm_stride=64):
    _need_cuda(ego, side)
    n, D = ego.shape
    if out is None:
        out = torch.empty_like(ego)
    call("spex_ngcf_epilogue_f32", ptr(_f32c(ego)), ptr(_f32c(side)), ptr(_f32c(W1)), ptr(b1),
         ptr(_f32c(W2)), ptr(b2), n, D, float(negative_slope), ptr(out), ptr(norm), int(norm_stride),
         stream_ptr())
    return out


NGCF_BWD_BLOCKS = 296            # SPEX_NGCF_BWD_BLOCKS in include/spex_b200.h
NGCF_BWD_WORK_PER_BLOCK = 8320   # SPEX_NGCF_BWD_WORK_PER_BLOCK


class _NGCFLayer(torch.autograd.Function):
    """One NGCF layer after the SpMM (NGCF_SPEX/code/main_rec.py:77-82) on the library's kernels:
    (hd, norm) = f(ego, side; W1, b1, W2, b2, mask) with its hand-written backward (deterministic weight
    gradients).  `mask` is nn.Dropout's 0 / 1/(1-p) pattern (None: no dropout)."""

    @staticmethod
    def forward(ctx, ego, side, W1, b1, W2, b2, mask, slope):
        _need_cuda(ego, side, W1, W2)
        ego, side, W1, W2 = _f32c(ego), _f32c(side), _f32c(W1), _f32c(W2)
        n, D = ego.shape
        hd = torch.empty_like(ego)
        norm = torch.empty_like(ego)
        call("spex_ngcf_layer_fwd_f32", ptr(ego), ptr(side), ptr(W1), ptr(b1), ptr(W2), ptr(b2), ptr(mask), n, D,
             float(slope), ptr(hd), ptr(norm), D, stream_ptr())
        ctx.save_for_backward(ego, side, W1, b1, W2, b2, mask)
        ctx.slope = float(slope)
        return hd, norm

    @staticmethod
    def backward(ctx, g_hd, g_norm):
        ego, side, W1, b1, W2, b2, mask = ctx.saved_tensors
        n, D = ego.shape
        dev = ego.device
        d_ego, d_side = torch.empty_like(ego), torch.empty_like(side)
        dW1, dW2 = torch.empty_like(W1), torch.empty_like(W2)
        db1 = torch.empty(D, dtype=torch.float32, device=dev)
        db2 = torch.empty(D, dtype=torch.float32, device=dev)
        work = torch.empty(NGCF_BWD_BLOCKS * NGCF_BWD_WORK_PER_BLOCK, dtype=torch.float32, device=dev)
        g_hd = None if g_hd is None else _f32c(g_hd)
        g_norm = None if g_norm is None else _f32c(g_norm)
        if g_hd is None and g_norm is None:
            g_norm = torch.zeros_like(ego)
        call("spex_ngcf_layer_bwd_f32", ptr(ego), ptr(side), ptr(W1), ptr(b1), ptr(W2), ptr(b2), ptr(mask),
             ptr(g_hd), ptr(g_norm), D, n, D, ctx.slope, ptr(d_ego), ptr(d_side), ptr(dW1), ptr(db1), ptr(dW2),
             ptr(db2), ptr(work), stream_ptr())
        return d_ego, d_side, dW1, (db1 if b1 is not None else None), dW2, (db2 if b2 is not None else None), None, None


def ngcf_layer(ego, side, W1, b1, W2, b2, mask=None, negative_slope: float = 0.01):
    """(hd, norm) of one NGCF layer given side = A . ego; differentiable (see _NGCFLayer)."""
    return _NGCFLayer.apply(ego, side, W1, b1, W2, b2, mask, negative_slope)


def launch_count() -> int:
    return _capi.launch_count()
