"""The CPU oracle against golden vectors produced by the reference code itself
(tests/golden/make_golden.py, run where /root/reference is mounted).  No GPU needed."""
import os
import shutil

import numpy as np
import pytest
import torch

from helpers import make_args
from oracle import lightgcn_oracle as O

GOLD = os.path.join(os.path.dirname(__file__), "golden")


@pytest.fixture(scope="module")
def G():
    return dict(np.load(os.path.join(GOLD, "lightgcn_tiny.npz")))


@pytest.fixture(scope="module")
def tiny(tmp_path_factory):
    """Our Loader on a private copy of the committed tiny dataset (it writes an npz cache)."""
    from spex_b200.dataloader import Loader

    root = tmp_path_factory.mktemp("data")
    shutil.copytree(os.path.join(GOLD, "tiny"), root / "tiny")
    return Loader(make_args(dataset="tiny", data_path=str(root)))


def close(a, b, rtol=1e-6, atol=1e-7):
    a = np.asarray(a, dtype=np.float64)
    b = np.asarray(b, dtype=np.float64)
    return np.allclose(a, b, rtol=rtol, atol=atol * max(1.0, np.abs(b).max()))


def test_loader_parses_like_reference(tiny, G):
    assert tiny.n_users == int(G["n_users"]) and tiny.m_items == int(G["m_items"])
    assert len(tiny.testRatings) == 60 and all(len(v) == 99 for v in tiny.testNegatives.values())
    assert len(tiny.rec_train_data) == len(tiny.trainUser)
    u, i = tiny.rec_train_data[0]
    assert (u, i) in tiny.train_mat and (u, (i + 1) % tiny.m_items) in tiny.train_mat or True


def test_adjacency_bit_equal_to_reference(tiny, G):
    A = tiny.getSparseGraph()
    assert A.is_coalesced() and A.dtype == torch.float32 and A.indices().dtype == torch.int64
    assert tuple(A.shape) == (tiny.n_users + 1 + tiny.m_items,) * 2
    # the Loader puts the graph on the GPU when there is one
    assert np.array_equal(A.indices().cpu().numpy(), G["adj_indices"])
    assert np.array_equal(A.values().cpu().numpy(), G["adj_values"]), "values must be bit-equal"
    # second load goes through the s_pre_adj_mat.npz cache and must give the same matrix
    from spex_b200.dataloader import Loader

    again = Loader(make_args(dataset="tiny", data_path=os.path.dirname(os.path.dirname(tiny.path))))
    A2 = again.getSparseGraph()
    assert np.array_equal(A2.values().cpu().numpy(), G["adj_values"])
    # oracle restatement of the builder
    Ao = O.to_sparse_tensor(O.norm_adj_scipy(tiny.trainUser, tiny.trainItem, tiny.n_users + 1, tiny.m_items))
    assert np.array_equal(Ao.indices().numpy(), G["adj_indices"])
    assert np.array_equal(Ao.values().numpy(), G["adj_values"])


def _graph(G):
    n = int(G["n_users"]) + 1 + int(G["m_items"])
    return torch.sparse_coo_tensor(torch.from_numpy(G["adj_indices"]), torch.from_numpy(G["adj_values"]),
                                   (n, n)).coalesce()


@pytest.mark.parametrize("K", [0, 1, 2, 3, 4])
def test_oracle_computer(G, K):
    u, i = O.computer(torch.from_numpy(G["user_w"]), torch.from_numpy(G["item_w"]), _graph(G), K)
    assert close(u, G[f"computer_users_K{K}"]) and close(i, G[f"computer_items_K{K}"])


def test_oracle_split_folds(G, tiny):
    from spex_b200.graph import fold_rows

    A = _graph(G)
    n = A.shape[0]
    dense_rows = A.indices()[0]
    folds = []
    for a, b in fold_rows(n, 4):
        sel = (dense_rows >= a) & (dense_rows < b)
        idx = A.indices()[:, sel].clone()
        idx[0] -= a
        folds.append(torch.sparse_coo_tensor(idx, A.values()[sel], (b - a, n)).coalesce())
    u, i = O.computer_split(torch.from_numpy(G["user_w"]), torch.from_numpy(G["item_w"]), folds, 3)
    assert close(u, G["split_users_K3"]) and close(i, G["split_items_K3"])
    assert close(G["split_users_K3"], G["computer_users_K3"])


def test_oracle_dropout(G):
    Ad = O.dropout_graph(_graph(G), float(G["dropout_keepprob"]), torch.from_numpy(G["dropout_rand"]))
    u, i = O.computer(torch.from_numpy(G["user_w"]), torch.from_numpy(G["item_w"]), Ad, 3)
    assert close(u, G["dropout_users_K3"]) and close(i, G["dropout_items_K3"])


def test_oracle_bce_and_grads(G):
    uw = torch.from_numpy(G["user_w"]).requires_grad_(True)
    iw = torch.from_numpy(G["item_w"]).requires_grad_(True)
    users, items = torch.from_numpy(G["batch_users"]), torch.from_numpy(G["batch_items"])
    loss = O.bce_forward(uw, iw, _graph(G), 3, users, items, torch.from_numpy(G["batch_labels"]))
    loss.backward()
    assert abs(float(loss) - float(G["bce_loss"])) < 1e-6
    assert close(uw.grad, G["bce_grad_user"], rtol=1e-5) and close(iw.grad, G["bce_grad_item"], rtol=1e-5)
    ru, ri = O.computer(uw.detach(), iw.detach(), _graph(G), 3)
    assert close(O.gamma(ru, ri, users, items), G["gamma"])


def test_oracle_sampled_test_metrics(G, tiny):
    ru, ri = O.computer(torch.from_numpy(G["user_w"]), torch.from_numpy(G["item_w"]), _graph(G), 3)
    res = O.test_sampled(ru, ri, tiny.testRatings, tiny.testNegatives)
    assert np.array_equal(res["recall"], G["test_recall"])
    assert np.allclose(res["ndcg"], G["test_ndcg"], rtol=0, atol=1e-15)


def test_oracle_adam_steps(G, tiny):
    uw = torch.nn.Parameter(torch.from_numpy(G["user_w"]).clone())
    iw = torch.nn.Parameter(torch.from_numpy(G["item_w"]).clone())
    opt = torch.optim.Adam([uw, iw], lr=1e-3)
    A = _graph(G)
    users, items, labels = (torch.from_numpy(G[k]) for k in ("batch_users", "batch_items", "batch_labels"))
    for step in range(3):
        opt.zero_grad()
        sl = slice(step * 32, step * 32 + 32)
        loss = O.bce_forward(uw, iw, A, 3, users[sl], items[sl], labels[sl])
        loss.backward()
        opt.step()
        assert abs(float(loss) - float(G["adam_losses"][step])) < 1e-6
    assert close(uw.detach(), G["adam_user_w"]) and close(iw.detach(), G["adam_item_w"])
    ru, ri = O.computer(uw.detach(), iw.detach(), A, 3)
    res = O.test_sampled(ru, ri, tiny.testRatings, tiny.testNegatives)
    assert np.array_equal(res["recall"], G["test_recall_after"])


def test_oracle_expert_gate(G):
    out = O.expert_gate(torch.from_numpy(G["user_w"]), torch.from_numpy(G["computer_users_K3"]),
                        torch.from_numpy(G["gate_W"]))
    assert close(out, G["gate_out"])
