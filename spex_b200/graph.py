"""Normalised bipartite adjacency in the layout the sm_100a kernels read (host side, numpy).

What the reference builds in ``Loader.getSparseGraph``
(/root/reference/LightGCN_SPEX/code/utility1/dataloader.py:187-225) with a dok/lil Python loop,
this module builds with vectorised numpy and hands to the GPU as CSR:

    rowptr int64 [N+1]   col int32 [nnz] (ascending per row)   val fp32 [nnz]

N = n_user_rows + m_items where n_user_rows = n_users + 1 (the reference keeps one padding user
row of degree 0, dataloader.py:93,110-111,196).  Rows [0, n_user_rows) are users (columns are
n_user_rows + item id), rows [n_user_rows, N) are items (columns are user ids).

Arithmetic order of the values follows the reference so they are bit-equal to its npz cache:
    rowsum (fp32) -> d = rowsum ** -0.5 (fp32, inf -> 0)            dataloader.py:205-207
    val[i,j] = fl32( fl32(d[i] * a[i,j]) * d[j] )                    dataloader.py:208-212
Duplicate (user,item) pairs add up (a[i,j] = multiplicity) exactly like the csr_matrix
constructor at dataloader.py:110-111.
"""
from __future__ import annotations

from dataclasses import dataclass, field
from typing import List, Optional, Tuple

import numpy as np

DEFAULT_SEG_LEN = 1024  # edges per warp-segment for long rows (see csrc/spmm.cu)


@dataclass
class CSRGraph:
    """Host copy of a CSR matrix (+ optional transpose map) with reference-compatible values."""

    n_rows: int
    n_cols: int
    rowptr: np.ndarray  # int64 [n_rows+1]
    col: np.ndarray  # int32 [nnz]
    val: np.ndarray  # fp32  [nnz]
    # tpos[e] = CSR position of the transposed entry (col[e], row(e)); only for square,
    # structurally symmetric matrices.  Used to form A_drop^T for the dropout backward.
    tpos: Optional[np.ndarray] = None
    row_offset: int = 0  # first global row when this is a row block of a larger matrix
    meta: dict = field(default_factory=dict)

    @property
    def nnz(self) -> int:
        return int(self.rowptr[-1])

    def degrees(self) -> np.ndarray:
        return np.diff(self.rowptr)

    def row_block(self, r0: int, r1: int) -> "CSRGraph":
        """Rows [r0, r1) as a standalone CSR whose columns still index the full table."""
        lo, hi = int(self.rowptr[r0]), int(self.rowptr[r1])
        return CSRGraph(
            n_rows=r1 - r0,
            n_cols=self.n_cols,
            rowptr=(self.rowptr[r0 : r1 + 1] - lo).astype(np.int64),
            col=self.col[lo:hi],
            val=self.val[lo:hi],
            tpos=None,
            row_offset=self.row_offset + r0,
        )

    def rows_of_entries(self) -> np.ndarray:
        return np.repeat(np.arange(self.n_rows, dtype=np.int64), self.degrees())


def _inv_sqrt_degree(rowsum_f32: np.ndarray) -> np.ndarray:
    with np.errstate(divide="ignore"):
        d = np.power(rowsum_f32, -0.5)
    d[np.isinf(d)] = 0.0
    return d.astype(np.float32, copy=False)


def build_norm_adj(
    users: np.ndarray, items: np.ndarray, n_user_rows: int, m_items: int, with_tpos: bool = True
) -> CSRGraph:
    """D^-1/2 [[0,R],[R^T,0]] D^-1/2 as CSR, values bit-equal to the reference builder."""
    users = np.asarray(users, dtype=np.int64).ravel()
    items = np.asarray(items, dtype=np.int64).ravel()
    if users.shape != items.shape:
        raise ValueError("users and items must have the same length")
    if users.size and (users.min() < 0 or users.max() >= n_user_rows):
        raise ValueError("user id out of range")
    if items.size and (items.min() < 0 or items.max() >= m_items):
        raise ValueError("item id out of range")
    N = n_user_rows + m_items
    if N >= 2**31:
        raise ValueError("node count must fit int32 column ids")

    # user half: unique (u,i) in (u,i) order, multiplicity as weight
    key = users * m_items + items
    ukey, mult = np.unique(key, return_counts=True)
    u = ukey // m_items
    i = ukey - u * m_items
    w = mult.astype(np.float32)
    nR = ukey.size

    # item half: same entries in (i,u) order
    perm = np.argsort(i * n_user_rows + u, kind="stable")  # item-half position -> user-half position
    ui, uu, wi = i[perm], u[perm], w[perm]

    deg_u = np.bincount(u, minlength=n_user_rows)
    deg_i = np.bincount(i, minlength=m_items)
    rowptr = np.zeros(N + 1, dtype=np.int64)
    np.cumsum(np.concatenate([deg_u, deg_i]), out=rowptr[1:])

    # fp32 row sums of the (possibly weighted) adjacency
    rs_u = np.bincount(u, weights=w, minlength=n_user_rows).astype(np.float32)
    rs_i = np.bincount(i, weights=w, minlength=m_items).astype(np.float32)
    d = _inv_sqrt_degree(np.concatenate([rs_u, rs_i]))

    col = np.empty(2 * nR, dtype=np.int32)
    col[:nR] = (i + n_user_rows).astype(np.int32)
    col[nR:] = uu.astype(np.int32)
    val = np.empty(2 * nR, dtype=np.float32)
    val[:nR] = (d[u] * w) * d[n_user_rows + i]
    val[nR:] = (d[n_user_rows + ui] * wi) * d[uu]

    tpos = None
    if with_tpos:
        tpos = np.empty(2 * nR, dtype=np.int64)
        tpos[perm] = nR + np.arange(nR, dtype=np.int64)  # user-half entry perm[p] <-> item-half p
        tpos[nR:] = perm
    return CSRGraph(N, N, rowptr, col, val, tpos, 0, {"n_user_rows": n_user_rows, "m_items": m_items})


def build_interaction_csr(users: np.ndarray, items: np.ndarray, n_rows: int, m_items: int):
    """CSR of R (training items per user, ascending, de-duplicated): the top-k mask."""
    users = np.asarray(users, dtype=np.int64).ravel()
    items = np.asarray(items, dtype=np.int64).ravel()
    ukey = np.unique(users * m_items + items)
    u = ukey // m_items
    i = (ukey - u * m_items).astype(np.int32)
    rowptr = np.zeros(n_rows + 1, dtype=np.int64)
    np.cumsum(np.bincount(u, minlength=n_rows), out=rowptr[1:])
    return rowptr, i


def csr_from_coo(rows: np.ndarray, cols: np.ndarray, vals: np.ndarray, n_rows: int, n_cols: int,
                 assume_sorted: bool = False, with_tpos: bool = False) -> CSRGraph:
    """CSR from COO triplets.  A coalesced torch sparse tensor is already (row, col)-sorted."""
    rows = np.asarray(rows, dtype=np.int64)
    cols = np.asarray(cols, dtype=np.int64)
    vals = np.asarray(vals, dtype=np.float32)
    if not assume_sorted:
        order = np.lexsort((cols, rows))
        rows, cols, vals = rows[order], cols[order], vals[order]
    rowptr = np.zeros(n_rows + 1, dtype=np.int64)
    np.cumsum(np.bincount(rows, minlength=n_rows), out=rowptr[1:])
    g = CSRGraph(n_rows, n_cols, rowptr, cols.astype(np.int32), vals)
    if with_tpos:
        g.tpos = transpose_positions(g)
    return g


def transpose_positions(g: CSRGraph) -> np.ndarray:
    """tpos for a structurally symmetric square CSR (raises if it is not symmetric)."""
    if g.n_rows != g.n_cols:
        raise ValueError("transpose map needs a square matrix")
    rows = g.rows_of_entries()
    cols = g.col.astype(np.int64)
    fwd = rows * g.n_cols + cols  # ascending by construction
    bwd = cols * g.n_cols + rows
    order = np.argsort(bwd, kind="stable")
    if not np.array_equal(bwd[order], fwd):
        raise ValueError("matrix is not structurally symmetric")
    tpos = np.empty(g.nnz, dtype=np.int64)
    tpos[order] = np.arange(g.nnz, dtype=np.int64)
    return tpos


def partition_rows_by_nnz(rowptr: np.ndarray, parts: int, row_cost: float = 2.0) -> List[int]:
    """Contiguous row ranges with balanced work = nnz + row_cost * rows (SURVEY §8e).

    Returns parts+1 boundaries b with b[0] = 0, b[-1] = n_rows.  Balancing by nnz rather than
    rows matters because users-then-items ordering makes row blocks heterogeneous.
    """
    rowptr = np.asarray(rowptr, dtype=np.int64)
    n = rowptr.size - 1
    work = rowptr + (row_cost * np.arange(n + 1)).astype(np.int64)
    total = work[-1]
    bounds = [0]
    for p in range(1, parts):
        target = total * p // parts
        b = int(np.searchsorted(work, target, side="left"))
        b = min(max(b, bounds[-1]), n)
        bounds.append(b)
    bounds.append(n)
    return bounds


def rebalance_bounds(rowptr: np.ndarray, bounds: List[int], times, row_cost: float = 2.0) -> List[int]:
    """Re-split the rows so that every part takes the same MEASURED time.

    `times[p]` is the time part p needed for its current block.  The cost of a row is modelled as
    (its nnz + row_cost) times the cost density of the block it currently lives in (user rows that
    gather popular items hit L2, item rows that gather random users do not, so the density differs
    between blocks).  Returns new boundaries with equal modelled cost per part.
    """
    rowptr = np.asarray(rowptr, dtype=np.int64)
    n = rowptr.size - 1
    parts = len(bounds) - 1
    work = (rowptr + (row_cost * np.arange(n + 1)).astype(np.int64)).astype(np.float64)
    cost = np.zeros(n + 1, dtype=np.float64)  # cumulative modelled cost at each row boundary
    acc = 0.0
    for p in range(parts):
        a, b = int(bounds[p]), int(bounds[p + 1])
        w = work[b] - work[a]
        dens = (float(times[p]) / w) if w > 0 else 0.0
        cost[a: b + 1] = acc + (work[a: b + 1] - work[a]) * dens
        acc = cost[b]
    new = [0]
    for p in range(1, parts):
        target = acc * p / parts
        r = int(np.searchsorted(cost, target, side="left"))
        new.append(min(max(r, new[-1]), n))
    new.append(n)
    return new


def fold_rows(n: int, folds: int) -> List[Tuple[int, int]]:
    """The reference's serial row folds (dataloader.py:167-177): equal row counts, last takes the rest."""
    fold_len = n // folds
    out = []
    for f in range(folds):
        start = f * fold_len
        end = n if f == folds - 1 else (f + 1) * fold_len
        out.append((start, end))
    return out
