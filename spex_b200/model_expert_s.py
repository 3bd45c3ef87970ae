"""Multi-task LightGCN (recommendation + trust-path prediction) with the API of the reference's
/root/reference/LightGCN_SPEX/code/utility1/model_expert_s.py (class LightGCN, lines 18-193), the
model behind main_11.py.

Recommendation branch (the hot path): computer() = the CSR SpMM propagation of spex_b200.model,
then the expert gate of model_expert_s.py:154-161 as one fused kernel per table
(spex_expert_gate_f32 / _bwd_f32), then the fused gather-dot-BCE.

Trust-path branch (model_expert_s.py:170-193, utility2/layers.py:15-72): paths of <= 5 user ids,
batches of a few hundred paths — host-loop bound in the reference (a Python double loop over paths
x positions) and far too small to be a kernel target (SURVEY §2, out of scope).  It is written here
as vectorised PyTorch with exactly the reference's arithmetic so that main_11 runs end to end on
the GPU; its parameters are created in the reference's order so a shared seed gives the same
initial weights.
"""
from __future__ import annotations

import math

import numpy as np
import torch
import torch.nn.functional as F
from torch import nn

from . import ops
from .model import BasicModel, LightGCN as _RecLightGCN, _FusedTable


class GraphAttentionLayer(nn.Module):
    """utility2/layers.py:5-72, vectorised over (path, position)."""

    def __init__(self, hidden_size, concat=True):
        super().__init__()
        self.concat = concat
        self.hidden_size = hidden_size
        self.a = nn.Parameter(torch.zeros(size=(2 * hidden_size, 1)))
        nn.init.xavier_uniform_(self.a.data, gain=1.414)

    def forward(self, emb, seq, seq_l):
        """concat=True: seq is [P, L] user ids, position embeddings (L_p - i) are added;
        concat=False: seq is [P, L, H] hidden vectors.  For i < L_p - 1 the output is the
        attention mix of (x_i, x_{i+1}) with logits [x_i|x_i].a and [x_i|x_{i+1}].a; elsewhere x_i."""
        if self.concat:
            x = emb[seq.long()]                                   # [P, L, H]
            P, L, _ = x.shape
            pos = (seq_l.view(P, 1) - torch.arange(L, device=x.device).view(1, L)).to(x.dtype)
            xi = x + pos.unsqueeze(2)                             # emb + (L_p - i)
        else:
            x = seq
            P, L, _ = x.shape
            xi = x
        if L < 2:
            return x
        cur, nxt = xi[:, :-1], xi[:, 1:]                          # nxt carries (L_p - i - 1) already
        a = self.a
        s0 = torch.cat([cur, cur], dim=2) @ a                     # [P, L-1, 1]
        s1 = torch.cat([cur, nxt], dim=2) @ a
        att = F.softmax(torch.cat([s0, s1], dim=2), dim=2)        # over the two rows of h
        mixed = att[..., 0:1] * cur + att[..., 1:2] * nxt
        active = (torch.arange(L - 1, device=x.device).view(1, L - 1) < (seq_l.view(P, 1) - 1)).unsqueeze(2)
        head = torch.where(active, mixed, x[:, :-1])
        return torch.cat([head, x[:, -1:]], dim=1)


class LightGCN(_RecLightGCN):
    def __init__(self, args_r, dataset):
        # parameter creation order of model_expert_s.py:19-66 (RNG parity under a shared seed)
        BasicModel.__init__(self)
        self.args_r = args_r
        self.dataset = dataset
        self.hidden_size = args_r.hiddenSize
        self.batch_size = args_r.batchSize
        self.nonhybrid = args_r.nonhybrid
        self.linear_one = nn.Linear(self.hidden_size, self.hidden_size, bias=True)
        self.linear_two = nn.Linear(self.hidden_size, self.hidden_size, bias=True)
        self.linear_three = nn.Linear(self.hidden_size, 1, bias=False)
        self.linear_transform = nn.Linear(self.hidden_size * 2, self.hidden_size, bias=True)
        stdv = 1.0 / math.sqrt(self.hidden_size)
        for weight in self.parameters():
            weight.data.uniform_(-stdv, stdv)
        self.in_att = [GraphAttentionLayer(self.hidden_size, concat=True) for _ in range(args_r.nb_heads)]
        for i, attention in enumerate(self.in_att):
            self.add_module("attention_{}".format(i), attention)
        self.out_att = GraphAttentionLayer(self.hidden_size, concat=False)
        self.w = nn.Parameter(torch.zeros(size=(args_r.nb_heads * self.hidden_size, self.hidden_size)))
        nn.init.xavier_uniform_(self.w.data, gain=1.414)

        self.num_users = dataset.n_users
        self.num_items = dataset.m_items
        self.latent_dim = args_r.recdim
        self.n_layers = args_r.layer
        self.keep_prob = args_r.keepprob
        self.A_split = args_r.A_split
        self.embedding_user = nn.Embedding(self.num_users + 1, self.latent_dim)
        self.embedding_item = nn.Embedding(self.num_items, self.latent_dim)
        nn.init.xavier_uniform_(self.embedding_user.weight, gain=1)
        nn.init.xavier_uniform_(self.embedding_item.weight, gain=1)
        self.f = nn.Sigmoid()
        self.Graph = dataset.getSparseGraph()

        self.task_weights = nn.Parameter(torch.FloatTensor([0.0, 0.0]))
        self.rec_loss = nn.BCEWithLogitsLoss()
        self.bcel = self.rec_loss
        self.loss_function = nn.CrossEntropyLoss()
        self.att_exp1 = nn.Parameter(torch.zeros(size=(2 * self.hidden_size, 2)))
        self.att_exp2 = nn.Parameter(torch.zeros(size=(2 * self.hidden_size, 2)))
        nn.init.xavier_uniform_(self.att_exp1.data, gain=1)
        nn.init.xavier_uniform_(self.att_exp2.data, gain=1)
        self.att_t = nn.Parameter(torch.zeros(size=(2 * self.hidden_size, 2)))
        nn.init.xavier_normal_(self.att_t.data, gain=1)

        self._table = None
        self._dev_graph = None
        self._mask_csr = None
        self._frozen_out = None
        self._freeze = False
        self._ranker = None
        self._fuse()

    # ---- recommendation branch -----------------------------------------------------------------
    def _compute_final(self) -> torch.Tensor:
        """[N, D] gated embeddings: softmax([E0 | E_prop] . att_exp) mix per row, users with
        att_exp1 and items with att_exp2 (model_expert_s.py:154-161)."""
        nur = self.n_user_rows
        prop = self._propagate()
        table = _FusedTable.apply(self.embedding_user.weight, self.embedding_item.weight, self._table)
        users = ops.expert_gate(table[:nur], prop[:nur], self.att_exp1)
        items = ops.expert_gate(table[nur:], prop[nur:], self.att_exp2)
        return torch.cat([users, items])

    # ---- trust branch --------------------------------------------------------------------------
    def compute_scores(self, hidden, inputs, mask):
        """model_expert_s.py:128-148."""
        P = mask.shape[0]
        ht = hidden[torch.arange(P, device=hidden.device), torch.sum(mask, 1) - 1]
        q1 = self.linear_one(ht).view(P, 1, ht.shape[1])
        q2 = self.linear_two(hidden)
        alpha = self.linear_three(torch.sigmoid(q1 + q2))
        a = torch.sum(alpha * hidden * mask.view(P, -1, 1).float(), 1)
        p_a = a if self.nonhybrid else self.linear_transform(torch.cat([a, ht], 1))
        b = self.embedding_user.weight[:-1]
        p_i = self.embedding_user.weight[inputs] * mask.unsqueeze(2)
        p_maxpool = torch.max(p_i, dim=1)[0]
        att = torch.softmax(torch.matmul(torch.cat([p_a, p_maxpool], 1), self.att_t), 1)
        a = p_a * att[:, 0].unsqueeze(1) + p_maxpool * att[:, 1].unsqueeze(1)
        return torch.matmul(a, b.transpose(1, 0))

    def _trust_scores(self, inputs, mask):
        seq_l = torch.sum(mask, 1)
        emb = self.embedding_user.weight
        mul_seq = torch.cat([att(emb, inputs, seq_l) for att in self.in_att], dim=2)
        P, L, _ = mul_seq.shape
        mul_one = F.elu(torch.mm(mul_seq.reshape(P * L, -1), self.w))
        hidden = self.out_att(emb, mul_one.view(P, L, self.hidden_size), seq_l)
        return self.compute_scores(hidden, inputs, mask)

    # ---- reference forward ---------------------------------------------------------------------
    def forward(self, users, items, labels, slice_indices=None, trust_data=None, flag=0):
        dev = self.embedding_user.weight.device
        loss1 = None
        if flag in (0, 1):
            out = self._final()
            if flag == 1:
                return ops.gather_dot(out, self.n_user_rows, users, items)
            loss1 = ops.bce_loss(out, self.n_user_rows, users, items, labels)
        if flag in (0, 2):
            sl = trust_data.get_slice(slice_indices)
            inputs = torch.as_tensor(np.asarray(sl[0]), device=dev).long()
            mask = torch.as_tensor(np.asarray(sl[1]), device=dev).long()
            targets = torch.as_tensor(np.asarray(sl[2]), device=dev).long()
            scores = self._trust_scores(inputs, mask)
            if flag == 2:
                return scores, torch.as_tensor(np.asarray(sl[3]), device=dev).long()
            loss2 = self.loss_function(scores, targets)
            return loss1, loss2
        raise UnboundLocalError("loss1")  # the reference falls through with loss1/loss2 unbound
