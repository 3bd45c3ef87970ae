"""LightGCN with the reference's API surface, computed by the sm_100a kernels of libspex_b200.

Drop-in for /root/reference/LightGCN_SPEX/code/utility1/model.py (class LightGCN, lines 19-121):
same constructor ``LightGCN(args_r, dataset)``, same attributes (``embedding_user``,
``embedding_item``, ``Graph``, ``num_users``, ``num_items``, ``n_layers``, ``keep_prob``,
``A_split``, ``f``, ``bcel``), same methods ``computer()`` and ``forward(users, items, labels,
flag)``, same RNG consumption at construction (so a shared seed gives identical initial weights).
It adds what BASELINE.json's north_star asks for and the reference leaves abstract or undefined:
``getUsersRating`` (model.py:14-15 raises NotImplementedError), ``bpr_loss`` and the fused
full-ranking ``rank_topk``.

Differences in HOW (not in WHAT):
  * the two embedding tables live in one [n_users+1+m_items, D] buffer, the nn.Embedding weights
    are views of it: no torch.cat per call (model.py:72);
  * K layers = K launches of the CSR SpMM, the layer mean rides in the epilogue: no stack/mean
    temporaries (model.py:94-95);
  * edge dropout (model.py:46-55) keeps the CSR structure and scales values by mask/keep_prob;
    with ``dropout=1`` the mask is drawn by the same CPU ``torch.rand(nnz)`` call so a shared seed
    drops the same edges; ``dropout=2`` generates it on the GPU from a hash of (seed, row, column)
    (ops.DeviceGraph.device_dropout_values): other edges than the reference drops, with the same
    distribution, and no host random numbers or copies at any graph size;
  * the backward is explicit (A^T SpMMs + deterministic segmented scatter), no atomics.
"""
from __future__ import annotations

import contextlib
from typing import Optional

import numpy as np
import torch
from torch import nn

from . import ops
from .graph import build_interaction_csr


class BasicModel(nn.Module):
    def getUsersRating(self, users):
        raise NotImplementedError


class _FusedTable(torch.autograd.Function):
    """Autograd glue: (user_weight, item_weight) -> the fused [N, D] table they are views of."""

    @staticmethod
    def forward(ctx, user_w, item_w, table):
        nur = user_w.shape[0]
        row_bytes = table.shape[1] * table.element_size()
        fused = (user_w.data_ptr() == table.data_ptr()
                 and item_w.data_ptr() == table.data_ptr() + nur * row_bytes)
        if not fused:  # somebody re-pointed a weight: refresh the table (rare path)
            table[:nur].copy_(user_w)
            table[nur:].copy_(item_w)
        ctx.nur = nur
        return table.detach()

    @staticmethod
    def backward(ctx, g):
        return g[: ctx.nur], g[ctx.nur:], None


class LightGCN(BasicModel):
    def __init__(self, args_r, dataset):
        super().__init__()
        self.args_r = args_r
        self.dataset = dataset
        self.bcel = nn.BCEWithLogitsLoss()  # kept for API parity; the fused kernel computes it

        self.num_users = dataset.n_users
        self.num_items = dataset.m_items
        self.latent_dim = args_r.recdim
        self.n_layers = args_r.layer
        self.keep_prob = args_r.keepprob
        self.A_split = args_r.A_split

        # same construction order as model.py:32-35 => same RNG stream => same initial weights
        self.embedding_user = nn.Embedding(self.num_users + 1, self.latent_dim)
        self.embedding_item = nn.Embedding(self.num_items, self.latent_dim)
        nn.init.xavier_uniform_(self.embedding_user.weight, gain=1)
        nn.init.xavier_uniform_(self.embedding_item.weight, gain=1)

        self.f = nn.Sigmoid()
        self.Graph = dataset.getSparseGraph()

        self._table: Optional[torch.Tensor] = None
        self._dev_graph: Optional[ops.DeviceGraph] = None
        self._mask_csr = None
        self._frozen_out: Optional[torch.Tensor] = None
        self._freeze = False
        self._ranker: Optional[ops.FullRanker] = None
        self._fuse()

    # ---- fused table ---------------------------------------------------------------------------
    @property
    def n_user_rows(self) -> int:
        return self.num_users + 1

    def _fuse(self):
        uw, iw = self.embedding_user.weight, self.embedding_item.weight
        nur = uw.shape[0]
        table = torch.empty(nur + iw.shape[0], uw.shape[1], dtype=uw.dtype, device=uw.device)
        with torch.no_grad():
            table[:nur].copy_(uw)
            table[nur:].copy_(iw)
        uw.data = table[:nur]
        iw.data = table[nur:]
        self._table = table

    def _apply(self, fn, *args, **kwargs):
        super()._apply(fn, *args, **kwargs)
        self._fuse()  # .to()/.cuda() moved the two weights separately: re-fuse on the new device
        self._dev_graph = None
        self._mask_csr = None
        self._frozen_out = None
        self._ranker = None
        return self

    def train(self, mode: bool = True):
        self._frozen_out = None
        self._ranker = None
        return super().train(mode)

    # ---- graph ---------------------------------------------------------------------------------
    def device_graph(self) -> ops.DeviceGraph:
        dev = self.embedding_user.weight.device
        if self._dev_graph is None or self._dev_graph.device != dev:
            if dev.type != "cuda":
                raise RuntimeError("spex_b200.LightGCN computes on sm_100a only: move the model to "
                                   "a CUDA device (there is no CPU fallback)")
            host = getattr(self.dataset, "getCSR", None)
            if host is not None:
                self._dev_graph = ops.DeviceGraph.from_host(host(), dev, D_hint=self.latent_dim)
            else:
                A = self.Graph
                if isinstance(A, (list, tuple)):  # A_split row folds (dataloader.py:167-177)
                    A = _stack_row_folds(A)
                self._dev_graph = ops.DeviceGraph.from_sparse_coo(A, dev)
            if self._dev_graph.n_rows == self._dev_graph.n_cols:
                self._dev_graph.mark_hot_columns(self.latent_dim)  # no-op unless the table dwarfs L2
        return self._dev_graph

    def _dropout_values(self, g: ops.DeviceGraph):
        if self.args_r.dropout == 2:
            return g.device_dropout_values(dropout_seed(), self.keep_prob)
        # model.py:50-53: keep edge e iff int(rand[e] + keep_prob) != 0; kept values / keep_prob.
        # Same CPU generator call as the reference, in coalesced (= CSR) edge order.
        keep = (torch.rand(g.nnz) + self.keep_prob).int().bool()
        val = g.dropout_values(keep, self.keep_prob)
        valT = g.transposed_values(val) if g.tpos is not None else None
        if valT is None:
            raise RuntimeError("edge dropout needs the transpose map of the adjacency; build the "
                               "graph through spex_b200.dataloader (getCSR)")
        return val, valT

    # ---- propagation ---------------------------------------------------------------------------
    def _propagate(self, rows_needed=None) -> torch.Tensor:
        """[N, D] layer-mean embeddings; rows [0, n_users] users, the rest items.  With `rows_needed`
        (training step) only those rows of the result are valid: every layer is restricted to the rows the
        batch depends on (ops.propagate_mean), loss and gradients unchanged bit for bit."""
        g = self.device_graph()
        table = _FusedTable.apply(self.embedding_user.weight, self.embedding_item.weight, self._table)
        val = valT = None
        if self.args_r.dropout and self.training:
            val, valT = self._dropout_values(g)
        return ops.propagate_mean(table, g, self.n_layers, val, valT, rows_needed=rows_needed)

    # main_rec.py:34 runs computer() over all N rows for a batch of 256: the training loss reads ~1.8 k of them.
    # True: forward(flag=0) / bpr_loss in training mode compute only the batch's receptive field.
    receptive_field = True

    def _batch_rows(self, users, *item_lists):
        """Row ids of the fused table a batch touches, or None when the full table is wanted."""
        if not (self.receptive_field and self.training and torch.is_grad_enabled()
                and type(self)._compute_final is LightGCN._compute_final and not self._freeze):
            return None
        dev = self.embedding_user.weight.device
        parts = [torch.as_tensor(users, device=dev).long().reshape(-1)]
        parts += [torch.as_tensor(i, device=dev).long().reshape(-1) + self.n_user_rows for i in item_lists]
        return torch.cat(parts)

    def _compute_final(self) -> torch.Tensor:
        """The [N, D] table forward() scores against (subclasses add the expert gate)."""
        return self._propagate()

    def _final(self) -> torch.Tensor:
        if self._freeze and self._frozen_out is not None:
            return self._frozen_out
        out = self._compute_final()
        if self._freeze:
            self._frozen_out = out.detach()
        return out

    def computer(self):
        """propagate methods for lightGCN: returns (users [n_users+1, D], items [m_items, D])."""
        out = self._final() if type(self)._compute_final is LightGCN._compute_final else self._propagate()
        return out[: self.n_user_rows], out[self.n_user_rows:]

    def final_embeddings(self):
        """(users, items) of the table forward() scores against: computer() for this model, the
        expert-gated tables for the multi-task model.  The hoisted Test() ranks with these."""
        out = self._final()
        return out[: self.n_user_rows], out[self.n_user_rows:]

    @contextlib.contextmanager
    def frozen_eval(self):
        """Reuse one propagation across many forward(flag=1) calls (the reference's Test() calls
        the model once per user, utility1/batch_test.py:33; weights do not change in between)."""
        if self.training:
            raise RuntimeError("frozen_eval() is for eval mode")
        self._freeze, self._frozen_out = True, None
        try:
            yield self
        finally:
            self._freeze, self._frozen_out = False, None

    # ---- reference forward ---------------------------------------------------------------------
    def forward(self, users, items, labels, flag=0):
        if flag not in (0, 1):
            raise UnboundLocalError("loss")  # the reference falls through to `return loss` unbound
        rows = self._batch_rows(users, items)
        out = self._final() if rows is None else self._propagate(rows_needed=rows)
        if flag == 1:
            return ops.gather_dot(out, self.n_user_rows, users, items)
        return ops.bce_loss(out, self.n_user_rows, users, items, labels)

    # ---- north_star additions ------------------------------------------------------------------
    def bpr_loss(self, users, pos, neg):
        """(loss, reg_loss): mean softplus(<u,n> - <u,p>) and 0.5*(|u0|^2+|p0|^2+|n0|^2)/B with
        u,p,n from computer() and u0,p0,n0 the raw embedding rows."""
        rows = self._batch_rows(users, pos, neg)
        out = self._final() if rows is None else self._propagate(rows_needed=rows)
        table = _FusedTable.apply(self.embedding_user.weight, self.embedding_item.weight, self._table)
        return ops.bpr_loss(out, table, self.n_user_rows, users, pos, neg)

    def getUsersRating(self, users):
        """sigmoid(out_users[users] . out_items^T) -> [B, m_items] (dense; for ranking use
        rank_topk, which never materialises this matrix)."""
        all_users, all_items = self.computer()
        users = torch.as_tensor(users, device=all_users.device).long()
        return ops.rating_dense(all_users, all_items, users)

    def train_mask_csr(self):
        """CSR of the training interactions on the device (rows = user ids): the top-k mask."""
        if self._mask_csr is None:
            dev = self.embedding_user.weight.device
            ds = self.dataset
            if hasattr(ds, "getInteractionCSR"):
                rp, col = ds.getInteractionCSR()
            else:
                rp, col = build_interaction_csr(ds.trainUser, ds.trainItem, self.n_user_rows,
                                                self.num_items)
            self._mask_csr = (torch.as_tensor(rp, dtype=torch.int64).to(dev),
                              torch.as_tensor(col, dtype=torch.int32).to(dev))
        return self._mask_csr

    @torch.no_grad()
    def rank_topk(self, users, k: int = 20, exclude_train: bool = True, precision: str = "f16",
                  user_block: int = 1 << 16, probe: bool = True):
        """Full-ranking top-k items per user: (idx int32 [B,k], score fp32 [B,k]).

        precision "f16":  tcgen05 fp16-accumulator filter + exact fp32 re-score of the survivors
                          (operands fp16(x 2^s); recdim 64 or 128) - the default; a probe
                          (ops.f16_filter_is_selective) routes tables with near-equal scores to "fp32";
        precision "bf16": round 1's tcgen05 GEMM, bf16 operands / fp32 accumulators (recdim 64);
        precision "fp32": exact CUDA-core scorer (bit-exact ordering, any recdim).
        Ordering: score descending, ties by ascending item id; masked = the user's train items.
        """
        all_users, all_items = self.computer()
        dev = all_users.device
        users = torch.as_tensor(users, device=dev).long().contiguous()
        mrp = mcol = None
        if exclude_train:
            mrp, mcol = self.train_mask_csr()
        # the packed item table is reused across eval-mode calls; fp32 reads the current table as it is
        r = self._ranker
        if r is None or self.training or r.precision != precision or precision == "fp32":
            r = self._ranker = ops.FullRanker(all_items, precision)
        if precision == "f16" and probe and not ops.f16_filter_is_selective(all_users, all_items, users):
            # degenerate score distribution (near-ties everywhere): the exact scorer is the faster exact path
            return ops.score_topk_f32(all_users, all_items, users, k, mrp, mcol)
        return r.topk(all_users, users, k, mrp, mcol, user_block)


def dropout_seed() -> int:
    """Seed of one training forward's device dropout mask (dropout=2), drawn from torch's default CPU generator so
    that torch.manual_seed reproduces a run."""
    return int(torch.randint(1 << 62, (1,)))


def _stack_row_folds(folds):
    idx, vals, r0 = [], [], 0
    n_cols = folds[0].shape[1]
    for f in folds:
        f = f.coalesce()
        i = f.indices().clone()
        i[0] += r0
        idx.append(i)
        vals.append(f.values())
        r0 += f.shape[0]
    return torch.sparse_coo_tensor(torch.cat(idx, 1), torch.cat(vals), (r0, n_cols)).coalesce()
