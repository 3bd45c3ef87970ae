"""NGCF_SPEX propagation (BASELINE.json configs[2], SURVEY §8 rows a10/a11) on the sm_100a kernels.

Mirrors /root/reference/NGCF_SPEX/code/main_rec.py::Model_Wrapper (constructor arguments, attribute
names, forward(user, item, labels_list, flag)) and utility/load_data.py::Data.create_adj_mat:

    norm_adj = D^-1 (A + I)                       load_data.py:122-166 (row-normalised, NOT symmetric)
    per layer (main_rec.py:76-85):  side = norm_adj . ego
        ego' = dropout( lrelu(W1 side + b1) + lrelu(W2 (ego * side) + b2) )
        all += normalize_2(ego');  output = concat over layers on the feature dimension
    flag 1 -> (user rows, item rows) [*, 64 (L+1)];  flag 0 -> BCEWithLogitsLoss of the row dots.

Inference (no gradient needed) runs the CSR SpMM + the fused `spex_ngcf_epilogue_f32` kernel that
writes the normalised rows straight into the concat buffer.  When gradients are needed the same SpMM
is used through an autograd function (backward = SpMM with the transposed values) and the dense part of
the layer - both 64x64 products, leaky-relu, message dropout, L2 normalisation - is ONE kernel forward
(`spex_ngcf_layer_fwd_f32`) and one backward (`spex_ngcf_layer_bwd_f32`, weight gradients reduced in a
fixed order, no atomics): no cuBLAS / ATen elementwise op on the training path.
Scoring: `rate_all_items` (the dense [B, n_items] matrix of utility/batch_test.py:158) and `rank_topk`
(the same contraction on the tcgen05 scorer at D = 128, fused with mask + top-k).
The user table keeps the reference's extra padding row, dropped in forward (main_rec.py:73).
There is no CPU fallback: every op raises on a CPU tensor.
"""
from __future__ import annotations

import ast

import numpy as np
import torch
import torch.nn as nn
import torch.nn.functional as F

from . import ops
from .graph import CSRGraph


def build_ngcf_norm_adj(users, items, n_users: int, n_items: int) -> CSRGraph:
    """D^-1 (A + I) over n_users + n_items nodes as CSR with the transpose map.

    Arithmetic as the reference: A is float32, `A + sp.eye` and everything after it float64
    (load_data.py:137-146,162), the model casts the result to float32 (main_rec.py:104).  Every
    entry of row r is fl32(1 / (deg_r + 1)); duplicate interactions add up like dok assignment
    does NOT (R[u, i] = 1.0 overwrites, load_data.py:56-69), so duplicates are dropped.
    """
    users = np.asarray(users, dtype=np.int64).ravel()
    items = np.asarray(items, dtype=np.int64).ravel()
    if users.size and (users.min() < 0 or users.max() >= n_users or items.min() < 0 or items.max() >= n_items):
        raise ValueError("interaction id out of range")
    N = n_users + n_items
    key = np.unique(users * n_items + items)
    u = key // n_items
    i = key - u * n_items
    rows = np.concatenate([u, n_users + i, np.arange(N, dtype=np.int64)])
    cols = np.concatenate([n_users + i, u, np.arange(N, dtype=np.int64)])
    order = np.lexsort((cols, rows))
    rows, cols = rows[order], cols[order]
    deg = np.bincount(rows, minlength=N)                      # includes the self loop
    rowptr = np.zeros(N + 1, dtype=np.int64)
    np.cumsum(deg, out=rowptr[1:])
    dinv = (1.0 / deg.astype(np.float64)).astype(np.float32)  # deg >= 1 everywhere
    val = dinv[rows]
    # position of the transposed entry (c, r): the pattern is symmetric, entries are sorted by
    # (row, col), so sorting by (col, row) enumerates the transposes in CSR order
    tpos = np.empty(rows.size, dtype=np.int64)
    tpos[np.lexsort((rows, cols))] = np.arange(rows.size, dtype=np.int64)
    return CSRGraph(n_rows=N, n_cols=N, rowptr=rowptr, col=cols.astype(np.int32), val=val, tpos=tpos)


def csr_from_scipy(norm_adj) -> CSRGraph:
    """The reference hands Model_Wrapper a scipy matrix (data_config['norm_adj']): take it as is."""
    m = norm_adj.tocsr().astype(np.float32)
    m.sort_indices()
    coo = m.tocoo()
    rows, cols = coo.row.astype(np.int64), coo.col.astype(np.int64)
    tpos = None
    if m.shape[0] == m.shape[1]:
        t = np.empty(rows.size, dtype=np.int64)
        t[np.lexsort((rows, cols))] = np.arange(rows.size, dtype=np.int64)
        if np.array_equal(rows[t], cols) and np.array_equal(cols[t], rows):   # symmetric pattern
            tpos = t
    return CSRGraph(n_rows=m.shape[0], n_cols=m.shape[1], rowptr=m.indptr.astype(np.int64),
                    col=m.indices.astype(np.int32), val=m.data.astype(np.float32), tpos=tpos)


class _SpMM(torch.autograd.Function):
    """Y = A . X with dX = A^T . dY (A^T shares A's pattern; its values are val[tpos])."""

    @staticmethod
    def forward(ctx, X, graph: ops.DeviceGraph, graph_t: ops.DeviceGraph):
        ctx.graph_t = graph_t
        return ops.spmm(graph, X.contiguous())

    @staticmethod
    def backward(ctx, g):
        return ops.spmm(ctx.graph_t, g.contiguous()), None, None


class Model_Wrapper(nn.Module):
    """Drop-in for NGCF_SPEX/code/main_rec.py::Model_Wrapper (flags 0 and 1)."""

    def __init__(self, data_config, device, args=None):
        super().__init__()
        self.device = torch.device(device)
        self.n_users = int(data_config["n_users"])
        self.n_items = int(data_config["n_items"])
        g = lambda name, default: getattr(args, name, default) if args is not None else default  # noqa: E731
        self.embedding_dim = int(g("embed_size", 64))
        layer_size = g("layer_size", "[64]")
        self.weight_size = list(ast.literal_eval(layer_size)) if isinstance(layer_size, str) else list(layer_size)
        self.n_layers = len(self.weight_size)
        mess = g("mess_dropout", "[0.1]")
        self.mess_dropout = list(ast.literal_eval(mess)) if isinstance(mess, str) else list(mess)
        regs = g("regs", "[1e-5]")
        self.regs = list(ast.literal_eval(regs)) if isinstance(regs, str) else list(regs)
        self.decay = self.regs[0]
        self.negative_slope = 0.01                      # F.leaky_relu default (main_rec.py:77,79)
        if any(w != self.embedding_dim for w in self.weight_size) or self.embedding_dim != 64:
            raise ValueError("the fused NGCF epilogue is built for embed_size == layer_size == 64")
        self.dropout_list = nn.ModuleList()
        self.GC_Linear_list = nn.ModuleList()
        self.Bi_Linear_list = nn.ModuleList()
        ws = [self.embedding_dim] + self.weight_size
        for i in range(self.n_layers):
            self.GC_Linear_list.append(nn.Linear(ws[i], ws[i + 1]))
            self.Bi_Linear_list.append(nn.Linear(ws[i], ws[i + 1]))
            self.dropout_list.append(nn.Dropout(self.mess_dropout[i]))
        self.user_embedding = nn.Embedding(self.n_users + 1, self.embedding_dim)
        nn.init.xavier_uniform_(self.user_embedding.weight)
        self.item_embedding = nn.Embedding(self.n_items, self.embedding_dim)
        nn.init.xavier_uniform_(self.item_embedding.weight)
        self.rec_loss_function = nn.BCEWithLogitsLoss()
        adj = data_config["norm_adj"]
        self._host_graph = adj if isinstance(adj, CSRGraph) else csr_from_scipy(adj)
        if self._host_graph.n_rows != self.n_users + self.n_items:
            raise ValueError("norm_adj must be (n_users + n_items) square")
        self._graph = self._graph_t = None

    # -- graph on the device (uploaded once; the reference re-uploads it every call, main_rec.py:76)
    def _graphs(self):
        if self._graph is None:
            dev = self.user_embedding.weight.device
            if dev.type != "cuda":
                raise RuntimeError("spex_b200.ngcf runs on a B200 only (no CPU fallback)")
            hg = self._host_graph
            self._graph = ops.DeviceGraph.from_host(hg, dev)
            if hg.tpos is not None:
                valT = self._graph.val[torch.from_numpy(hg.tpos).to(dev)]
                self._graph_t = self._graph.with_values(valT, symmetric=False)
        return self._graph, self._graph_t

    def propagate(self):
        """(user rows [n_users, 64 (L+1)], item rows [n_items, 64 (L+1)]) - main_rec.py:72-86."""
        graph, graph_t = self._graphs()
        D, L = self.embedding_dim, self.n_layers
        ego = torch.cat((self.user_embedding.weight[:-1], self.item_embedding.weight), dim=0)
        need_grad = torch.is_grad_enabled() and any(p.requires_grad for p in self.parameters())
        if not need_grad and not (self.training and any(p > 0 for p in self.mess_dropout)):
            N = ego.shape[0]
            out = torch.empty(N, D * (L + 1), dtype=torch.float32, device=ego.device)
            out[:, :D] = ego
            ego = ego.contiguous()
            for i in range(L):
                side = ops.spmm(graph, ego)
                ego = ops.ngcf_epilogue(ego, side, self.GC_Linear_list[i].weight, self.GC_Linear_list[i].bias,
                                        self.Bi_Linear_list[i].weight, self.Bi_Linear_list[i].bias,
                                        self.negative_slope, norm=out[:, D * (i + 1):], norm_stride=D * (L + 1))
            all_embeddings = out
        else:
            if graph_t is None:
                raise RuntimeError("training needs a structurally symmetric norm_adj (transpose map)")
            embs = [ego]
            for i in range(L):
                side = _SpMM.apply(ego, graph, graph_t)
                # message dropout (main_rec.py:81): the mask comes from the reference's own RNG call - the
                # nn.Dropout module applied to a tensor of the layer's shape - and is applied inside the kernel
                mask = None
                if self.training and self.mess_dropout[i] > 0:
                    mask = self.dropout_list[i](torch.ones_like(side))
                ego, norm = ops.ngcf_layer(ego, side, self.GC_Linear_list[i].weight, self.GC_Linear_list[i].bias,
                                           self.Bi_Linear_list[i].weight, self.Bi_Linear_list[i].bias, mask,
                                           self.negative_slope)
                embs.append(norm)
            all_embeddings = torch.cat(embs, dim=1)
        return torch.split(all_embeddings, [self.n_users, self.n_items], dim=0)

    def forward(self, user, item, labels_list, flag):
        if flag not in (0, 1):
            raise ValueError("flag must be 0 (loss) or 1 (embeddings)")
        ua, ia = self.propagate()
        if flag == 1:
            return ua, ia
        dev = ua.device
        u = ua[torch.as_tensor(user, device=dev).long()]
        v = ia[torch.as_tensor(item, device=dev).long()]
        return self.compute_rec_loss(u, v, labels_list)

    def compute_rec_loss(self, u_g_embeddings, i_g_embeddings, labels_list):
        predict = torch.sum(torch.mul(u_g_embeddings, i_g_embeddings), dim=1)
        real = torch.as_tensor(labels_list, device=predict.device).float()
        return self.rec_loss_function(predict, real)

    @torch.no_grad()
    def rank_topk(self, users, k: int = 20, mask_rowptr=None, mask_col=None, precision: str = "f16",
                  probe: bool = True):
        """Top-k items per user over the concatenated layer outputs (utility/batch_test.py:158 followed by
        the ranking) through ops.FullRanker: tcgen05 fp16-accumulator filter + exact fp32 re-score at
        D = 64 (L + 1) in {64, 128}, k <= 512, or the exact fp32 CUDA-core scorer (precision "fp32", or "f16" at
        any other D; k <= 128).  probe: near-equal scores (an untrained NGCF's normalised outputs are almost
        parallel) go to the fp32 scorer when k <= 128 (ops.FullRanker.scorer_for).  Returns (idx int32 [B, k],
        score fp32 [B, k])."""
        ua, ia = self.propagate()
        ua, ia = ua.contiguous(), ia.contiguous()
        if precision == "f16":
            precision = ops.default_precision(ua.shape[1])
        return ops.FullRanker(ia, precision, probe=probe).topk(ua, users, k, mask_rowptr, mask_col)

    @torch.no_grad()
    def rate_all_items(self, users):
        """utility/batch_test.py:158: [B, n_items] scores of a user block over the 128-d outputs."""
        ua, ia = self.propagate()
        users = torch.as_tensor(users, device=ua.device).long()
        return ops.rating_dense(ua.contiguous(), ia.contiguous(), users, apply_sigmoid=False)
