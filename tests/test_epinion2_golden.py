"""BASELINE.json configs[0] - LightGCN_SPEX main_rec.py on epinion2 (3 layers, dim 64) - against
golden vectors produced by the unmodified reference on its own shipped data
(tests/golden/make_epinion2.py: /root/reference/Data_process/rec/data_process_rec.py on
Data_process/rec/epinion2/*.mat, then LightGCN_SPEX/code/utility1/{dataloader,model,batch_test}.py).
3 185 users x 12 407 items, 209 304 train interactions, N = 15 593, nnz(A) = 418 608.
CPU tests pin the Loader / graph builder / oracle; the `gpu` tests pin the CUDA path."""
import os

import numpy as np
import pytest
import torch

from helpers import make_args, rel_err
from oracle import lightgcn_oracle as O

GOLD = os.path.join(os.path.dirname(__file__), "golden")


def seeded_weights(n_user_rows, m_items, D=64, seed=7):
    """Same numpy stream as tests/golden/make_epinion2.py::seeded_weights."""
    rng = np.random.default_rng(seed)
    au, ai = np.sqrt(6.0 / (n_user_rows + D)), np.sqrt(6.0 / (m_items + D))
    U = rng.uniform(-au, au, (n_user_rows, D)).astype(np.float32)
    I = rng.uniform(-ai, ai, (m_items, D)).astype(np.float32)
    return U, I


@pytest.fixture(scope="module")
def G():
    return dict(np.load(os.path.join(GOLD, "epinion2_golden.npz")))


@pytest.fixture(scope="module")
def ep2_root(tmp_path_factory):
    """The processed dataset written back in the reference's on-disk format
    (`user item 1` lines; `.test.rating`: the last line of a user is the held-out positive,
    dataloader.py:139-148; `.test.negative`: `user n1 .. n99`, dataloader.py:150-165)."""
    d = np.load(os.path.join(GOLD, "epinion2_data.npz"))
    root = tmp_path_factory.mktemp("ep2")
    rec = root / "epinion2" / "rec"
    rec.mkdir(parents=True)
    with open(rec / "epinion2.train.rating", "w") as f:
        f.write("".join(f"{u} {i} 1\n" for u, i in zip(d["train_user"].tolist(), d["train_item"].tolist())))
    with open(rec / "epinion2.test.rating", "w") as f:
        for u, p, neg in zip(d["test_user"].tolist(), d["test_pos"].tolist(), d["test_neg"].tolist()):
            f.write(f"{u} {neg[0]} 0\n")          # an earlier line of the user must lose
            f.write(f"{u} {p} 1\n")
    with open(rec / "epinion2.test.negative", "w") as f:
        for u, neg in zip(d["test_user"].tolist(), d["test_neg"].tolist()):
            f.write(" ".join([str(u)] + [str(x) for x in neg]) + "\n")
    return str(root)


@pytest.fixture(scope="module")
def ep2(ep2_root):
    from spex_b200.dataloader import Loader

    return Loader(make_args(dataset="epinion2", data_path=ep2_root))


def test_loader_and_adjacency_match_reference(ep2, G):
    assert (ep2.n_users, ep2.m_items) == (int(G["n_users"]), int(G["m_items"])) == (3185, 12407)
    assert len(ep2.trainUser) == 209304 and len(ep2.testRatings) == 3185
    A = ep2.getSparseGraph()
    assert A.is_coalesced() and A._nnz() == int(G["adj_nnz"]) == 418608
    idx, val = A.indices().cpu().numpy(), A.values().cpu().numpy()   # on the GPU when there is one
    pick = G["adj_pick"]
    assert np.array_equal(idx[:, pick], G["adj_pick_rc"])
    assert np.array_equal(val[pick], G["adj_pick_val"]), "adjacency values must be bit-equal"
    assert float(val.astype(np.float64).sum()) == float(G["adj_value_sum"])
    rowsum = np.bincount(idx[0], weights=val.astype(np.float64), minlength=A.shape[0])[::13]
    assert np.array_equal(rowsum, G["adj_rowsum"])


def test_oracle_computer_and_loss_on_epinion2(ep2, G):
    U, I = seeded_weights(ep2.n_users + 1, ep2.m_items)
    A = O.to_sparse_tensor(O.norm_adj_scipy(ep2.trainUser, ep2.trainItem, ep2.n_users + 1, ep2.m_items))
    uw = torch.from_numpy(U).requires_grad_(True)
    iw = torch.from_numpy(I).requires_grad_(True)
    cu, ci = O.computer(uw, iw, A, 3)
    rows = torch.cat([cu, ci]).detach().numpy()
    assert np.allclose(rows[::13], G["computer_rows_13"], rtol=1e-6, atol=1e-9)
    assert np.allclose(rows.astype(np.float64).sum(0), G["computer_colsum"], rtol=1e-6, atol=1e-7)
    bu, bi, bl = (torch.from_numpy(G[k]) for k in ("batch_users", "batch_items", "batch_labels"))
    loss = O.bce_forward(uw, iw, A, 3, bu, bi, bl)
    loss.backward()
    assert abs(float(loss) - float(G["bce_loss"])) < 1e-6
    assert np.allclose(uw.grad.numpy()[::13], G["grad_user_rows_13"], rtol=1e-5, atol=1e-10)
    assert np.allclose(iw.grad.numpy()[::13], G["grad_item_rows_13"], rtol=1e-5, atol=1e-10)


def _gpu_model(ep2_root, dev):
    from spex_b200.dataloader import Loader
    from spex_b200.model import LightGCN

    args = make_args(dataset="epinion2", data_path=ep2_root)
    ds = Loader(args)
    model = LightGCN(args, ds)
    U, I = seeded_weights(ds.n_users + 1, ds.m_items)
    with torch.no_grad():
        model.embedding_user.weight.copy_(torch.from_numpy(U))
        model.embedding_item.weight.copy_(torch.from_numpy(I))
    return ds, model.to(dev)


@pytest.mark.gpu
def test_gpu_computer_loss_and_gradients_on_epinion2(ep2_root, G, cuda_device):
    ds, model = _gpu_model(ep2_root, cuda_device)
    model.eval()
    with torch.no_grad():
        cu, ci = model.computer()
    rows = torch.cat([cu, ci]).cpu()
    assert rel_err(rows[::13], torch.from_numpy(G["computer_rows_13"])) < 1e-5     # north_star fp32 bar
    assert np.allclose(rows.double().sum(0).numpy(), G["computer_colsum"], rtol=1e-5, atol=1e-6)
    bu, bi, bl = (torch.from_numpy(G[k]).to(cuda_device) for k in ("batch_users", "batch_items", "batch_labels"))
    model.train()
    model.zero_grad()
    loss = model(bu, bi, bl, flag=0)
    loss.backward()
    assert abs(float(loss) - float(G["bce_loss"])) < 1e-5 * abs(float(G["bce_loss"]))
    gu, gi = model.embedding_user.weight.grad.cpu(), model.embedding_item.weight.grad.cpu()
    assert rel_err(gu[::13], torch.from_numpy(G["grad_user_rows_13"])) < 1e-5
    assert rel_err(gi[::13], torch.from_numpy(G["grad_item_rows_13"])) < 1e-5
    assert abs(float(gu.abs().double().sum()) - float(G["grad_user_abs_sum"])) < 1e-4 * float(G["grad_user_abs_sum"])


@pytest.mark.gpu
def test_gpu_sampled_test_metrics_identical_on_epinion2(ep2_root, G, cuda_device):
    from spex_b200 import batch_test

    ds, model = _gpu_model(ep2_root, cuda_device)
    model.eval()
    sub = [int(u) for u in G["test_users"]]
    ret = batch_test.test(model, {u: ds.testRatings[u] for u in sub}, {u: ds.testNegatives[u] for u in sub})
    assert np.array_equal(ret["recall"], G["test_recall"])
    assert np.allclose(ret["ndcg"], G["test_ndcg"], rtol=0, atol=1e-12)


@pytest.fixture(scope="module")
def F():
    return dict(np.load(os.path.join(GOLD, "epinion2_full.npz")))


@pytest.mark.gpu
def test_gpu_every_row_and_every_test_user_on_epinion2(ep2_root, G, F, cuda_device):
    """epinion2_full.npz (tests/golden/make_epinion2.py with SPEX_EP2_FULL=1): two float64 numbers per row
    (sum, sum of squares) of the reference's computer() output and of both gradient tables - so EVERY row is
    checked, not every 13th - and the reference's Test() over ALL 3 185 test users (one propagation per
    user there, one in total here): Recall identical, NDCG to 1e-12."""
    from spex_b200 import batch_test

    ds, model = _gpu_model(ep2_root, cuda_device)
    model.eval()
    with torch.no_grad():
        cu, ci = model.computer()
    rows = torch.cat([cu, ci]).double().cpu().numpy()
    scale = np.sqrt(F["computer_row_sq"]).max()
    assert np.abs(rows.sum(1) - F["computer_row_sum"]).max() < 1e-5 * scale * 8          # 64 terms per row
    assert np.abs(np.sqrt((rows ** 2).sum(1)) - np.sqrt(F["computer_row_sq"])).max() < 1e-5 * scale
    bu, bi, bl = (torch.from_numpy(G[k]).to(cuda_device) for k in ("batch_users", "batch_items", "batch_labels"))
    model.train()
    model.zero_grad()
    model(bu, bi, bl, flag=0).backward()
    for name, grad in (("user", model.embedding_user.weight.grad), ("item", model.embedding_item.weight.grad)):
        g = grad.double().cpu().numpy()
        gs = np.sqrt(F[f"grad_{name}_row_sq"]).max()
        assert np.abs(g.sum(1) - F[f"grad_{name}_row_sum"]).max() < 1e-5 * gs * 8, name
        assert np.abs(np.sqrt((g ** 2).sum(1)) - np.sqrt(F[f"grad_{name}_row_sq"])).max() < 1e-5 * gs, name
    model.eval()
    assert len(ds.testRatings) == int(F["n_test_users"]) == 3185
    ret = batch_test.test(model, ds.testRatings, ds.testNegatives)
    assert np.array_equal(ret["recall"], F["test_recall_all"])
    assert np.allclose(ret["ndcg"], F["test_ndcg_all"], rtol=0, atol=1e-12)
