"""Seeded synthetic bipartite graphs at benchmark scale, generated ON the GPU.

The reference builds its adjacency with an O(nnz) Python loop over a scipy dok matrix
(/root/reference/LightGCN_SPEX/code/utility1/dataloader.py:99-100,197-202), which cannot produce
BASELINE.json's 10 M x 5 M, 10^9-interaction configuration.  This module produces that graph
directly in the HBM layout the kernels read (rowptr int64 / col int32 / val fp32).  It is input
preparation (torch sort/unique as plumbing), never part of a timed region.

Shape of the data (SURVEY §8d): every user has at least one interaction, user activity uniform,
item popularity Zipf-Mandelbrot p(r) ~ (r + q)^-alpha over a random permutation of item ids (so
ids carry no locality), duplicate pairs removed.
"""
from __future__ import annotations

from typing import Tuple

import torch

from .ops import DeviceGraph


def _zipf_mandelbrot(n: int, m_items: int, alpha: float, shift: float, gen, device) -> torch.Tensor:
    """n item ranks in [0, m_items) by inverse-CDF sampling of p(x) ~ (x + shift)^-alpha."""
    U = torch.rand(n, dtype=torch.float64, device=device, generator=gen)
    e = 1.0 - alpha
    lo, hi = shift ** e, (m_items + shift) ** e
    x = (lo - U * (lo - hi)).pow_(1.0 / e).sub_(shift)
    return x.floor_().clamp_(0, m_items - 1).to(torch.int64)


def generate_interactions(n_users: int, m_items: int, n_inter: int, seed: int = 2020,
                          device="cuda", zipf_alpha: float = 1.3, zipf_shift: float = None,
                          chunk: int = 1 << 27) -> torch.Tensor:
    """Sorted unique int64 keys u * m_items + i of the interactions (about n_inter of them)."""
    dev = torch.device(device)
    gen = torch.Generator(device=dev)
    gen.manual_seed(seed)
    if zipf_shift is None:
        zipf_shift = max(m_items / 1000.0, 1.0)
    item_perm = torch.randperm(m_items, device=dev, generator=gen)
    parts = []
    # one guaranteed interaction per user, then uniform users for the rest
    todo = n_inter
    first = True
    while todo > 0:
        n = min(chunk, todo)
        if first:
            nu = min(n_users, n)
            u = torch.cat([torch.arange(nu, device=dev),
                           torch.randint(0, n_users, (n - nu,), device=dev, generator=gen)])
            first = False
        else:
            u = torch.randint(0, n_users, (n,), device=dev, generator=gen)
        it = item_perm[_zipf_mandelbrot(n, m_items, zipf_alpha, zipf_shift, gen, dev)]
        parts.append(torch.unique(u * m_items + it))
        todo -= n
    keys = parts[0] if len(parts) == 1 else torch.unique(torch.cat(parts))
    return keys


def build_norm_adj_device(keys: torch.Tensor, n_users: int, m_items: int,
                          seg_len: int = 1024) -> Tuple[DeviceGraph, torch.Tensor, torch.Tensor]:
    """Normalised adjacency (dataloader.py:196-212 semantics, unit weights) from sorted unique keys.

    Returns (graph, mask_rowptr int64 [n_user_rows+1], mask_col int32 [|R|]): the interaction CSR
    doubles as the training-item mask of the full-ranking evaluation.
    """
    dev = keys.device
    nur = n_users + 1
    N = nur + m_items
    nR = keys.numel()
    u = torch.div(keys, m_items, rounding_mode="floor")
    it = keys - u * m_items
    deg_u = torch.bincount(u, minlength=nur)
    deg_i = torch.bincount(it, minlength=m_items)
    deg = torch.cat([deg_u, deg_i])
    rowptr = torch.zeros(N + 1, dtype=torch.int64, device=dev)
    torch.cumsum(deg, 0, out=rowptr[1:])
    d = deg.to(torch.float32).pow(-0.5)
    d[torch.isinf(d)] = 0.0
    del deg
    col = torch.empty(2 * nR, dtype=torch.int32, device=dev)
    val = torch.empty(2 * nR, dtype=torch.float32, device=dev)
    col[:nR] = (it + nur).to(torch.int32)
    val[:nR] = d[u] * d[nur + it]
    mask_col = it.to(torch.int32)
    mask_rowptr = rowptr[: nur + 1].clone()
    # item half: the same pairs in (item, user) order
    k2 = it * nur + u
    del u, it
    k2 = torch.sort(k2).values
    i2 = torch.div(k2, nur, rounding_mode="floor")
    u2 = k2 - i2 * nur
    del k2
    col[nR:] = u2.to(torch.int32)
    val[nR:] = d[nur + i2] * d[u2]
    del i2, u2
    # values d[u]*d[i] both ways and no duplicate pairs: symmetric bit for bit, so dropout needs no tpos
    g = DeviceGraph(rowptr, col, val, N, None, seg_len, values_symmetric=True)
    return g, mask_rowptr, mask_col


def xavier_table(n_user_rows: int, m_items: int, D: int, seed: int, device) -> torch.Tensor:
    """Fused [N, D] table initialised like model.py:34-35 (xavier-uniform, gain 1, per table)."""
    gen = torch.Generator(device=device)
    gen.manual_seed(seed)
    t = torch.empty(n_user_rows + m_items, D, dtype=torch.float32, device=device)
    for lo, n in ((0, n_user_rows), (n_user_rows, m_items)):
        a = (6.0 / (n + D)) ** 0.5
        t[lo: lo + n].uniform_(-a, a, generator=gen)
    return t
