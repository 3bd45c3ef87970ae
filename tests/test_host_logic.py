"""Host-side logic that needs no GPU: graph builder, partitioning, metrics, ranking semantics,
negative sampler stream, C-ABI surface."""
import ctypes
import heapq
import os
import re

import numpy as np
import pytest
import torch

from helpers import random_graph
from oracle import lightgcn_oracle as O

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_norm_adj_matches_scipy_builder_with_duplicates_and_empty_rows():
    from spex_b200.graph import build_norm_adj, transpose_positions

    u, i = random_graph(300, 200, 3000, 1)
    u = np.concatenate([u, u[:7]])
    i = np.concatenate([i, i[:7]])  # duplicate pairs add up (csr_matrix constructor semantics)
    u = u[u != 5]  # make user 5 ... still might exist; force an empty row explicitly below
    i = i[: u.size]
    A = O.norm_adj_scipy(u, i, 301, 200)
    g = build_norm_adj(u, i, 301, 200)
    assert np.array_equal(A.indptr, g.rowptr) and np.array_equal(A.indices, g.col)
    assert np.array_equal(A.data, g.val)
    assert g.rowptr[301] - g.rowptr[300] == 0  # padding user row is empty
    assert np.array_equal(transpose_positions(g), g.tpos)
    rows = g.rows_of_entries()
    assert np.array_equal(g.col[g.tpos], rows) and np.array_equal(rows[g.tpos], g.col)


def test_empty_graph_and_single_edge():
    from spex_b200.graph import build_norm_adj

    g = build_norm_adj(np.zeros(0, np.int64), np.zeros(0, np.int64), 4, 3)
    assert g.nnz == 0 and g.rowptr.tolist() == [0] * 8
    g = build_norm_adj(np.array([2]), np.array([1]), 4, 3)
    assert g.nnz == 2 and g.val.tolist() == [1.0, 1.0] and g.col.tolist() == [5, 2]


def _plan_segments(p):
    """(segment -> long-row slot) and the (start, count) pairs of a DeviceGraph.long_row_plan result."""
    segptr, row_seg = p["long_segptr"].tolist(), p["row_seg"].tolist()
    seg_slot = [0] * p["n_seg"]
    for k in range(p["n_long"]):
        for j in row_seg[segptr[k]: segptr[k + 1]]:
            seg_slot[j] = k
    return seg_slot, list(zip(p["seg_start"].tolist(), p["seg_count"].tolist()))


def test_long_row_plan_segment_list_fits_in_l2():
    """DeviceGraph.long_row_plan on CPU tensors.  A table that fits in L2 has no hub rows: every long row is cut
    every seg_len edges, in ascending row order, and row_seg is the identity."""
    from spex_b200.ops import DeviceGraph

    rowptr = torch.tensor([0, 10, 10, 110, 174, 1200])
    col = torch.cat([torch.arange(int(d), dtype=torch.int32) for d in rowptr.diff()])
    p = DeviceGraph.long_row_plan(rowptr, col, 2000, 64, 64)
    assert p["long_rows"].tolist() == [2, 4] and p["n_long"] == 2
    assert p["long_segptr"].tolist() == [0, 2, 2 + 17] and p["n_seg"] == 19
    assert p["n_hub"] == 0 and p["n_hub_seg"] == 0
    cuts = [(s, min(64, int(rowptr[r + 1]) - s)) for r in (2, 4) for s in range(int(rowptr[r]), int(rowptr[r + 1]), 64)]
    assert _plan_segments(p)[1] == cuts
    assert p["row_seg"].tolist() == list(range(19))
    p = DeviceGraph.long_row_plan(rowptr, col, 2000, 2048, 64)
    assert p["n_long"] == 0 and p["n_seg"] == 0 and p["long_segptr"].tolist() == [0]
    with pytest.raises(ValueError):
        DeviceGraph.long_row_plan(rowptr, col, 2000, 16, 64)


def test_long_row_plan_segment_list_column_blocked(monkeypatch):
    """A window far smaller than the table: hub rows are cut at column-block boundaries and their cells listed
    first, block-major; every long-row edge is in exactly one segment; each row's segments ascend; the hot flag
    in bit 31 of col does not change the plan."""
    from spex_b200.ops import DeviceGraph

    monkeypatch.setattr(DeviceGraph, "L2_WINDOW_BYTES", 16 * 1024)    # 64 columns per block at D = 64
    monkeypatch.setattr(DeviceGraph, "MIN_CB_COLS", 48)
    monkeypatch.setattr(DeviceGraph, "HUB_EDGES_PER_BLOCK", 10)       # 4000 columns = 63 blocks: hub from 630 edges
    monkeypatch.delenv("SPEX_L2_WINDOW_MB", raising=False)
    monkeypatch.delenv("SPEX_HUB_EPB", raising=False)
    n_cols, cb, seg_len = 4000, 64, 64
    rng = np.random.default_rng(0)
    degs = [10, 3000, 200, 5, 1500, 700, 100, 64, 65, 500, 2500, 0]
    col = torch.from_numpy(np.concatenate([np.sort(rng.choice(n_cols, d, replace=False)) for d in degs]).astype(np.int32))
    rowptr = torch.from_numpy(np.concatenate([[0], np.cumsum(degs)]).astype(np.int64))
    p = DeviceGraph.long_row_plan(rowptr, col, n_cols, seg_len, 64)
    long_rows = [r for r, d in enumerate(degs) if d > seg_len]
    hubs = [r for r, d in enumerate(degs) if d >= 630]
    assert p["long_rows"].tolist() == long_rows and p["n_hub"] == len(hubs)
    H = p["n_hub_seg"]
    seg_slot, segs = _plan_segments(p)
    assert 0 < H < p["n_seg"]
    assert all(0 < c <= seg_len for _, c in segs)
    seg_row = [long_rows[k] for k in seg_slot]
    assert all(r in hubs for r in seg_row[:H]) and not any(r in hubs for r in seg_row[H:])
    c = col.numpy()
    blocks = [int(c[s]) // cb for s, _ in segs[:H]]
    assert blocks == sorted(blocks)                                     # hub cells block-major
    assert all(int(c[s]) // cb == int(c[s + n - 1]) // cb for s, n in segs[:H])   # a cell stays in its block
    mid = [(s, min(seg_len, int(rowptr[r + 1]) - s)) for r in long_rows if r not in hubs
           for s in range(int(rowptr[r]), int(rowptr[r + 1]), seg_len)]
    assert segs[H:] == mid                                              # mid rows: seg_len cuts, row order
    edges = sorted(e for s, n in segs for e in range(s, s + n))
    assert edges == [e for r in long_rows for e in range(int(rowptr[r]), int(rowptr[r + 1]))]
    segptr, row_seg = p["long_segptr"].tolist(), p["row_seg"].tolist()
    for k, r in enumerate(long_rows):                                   # each row's segments tile it in order
        own = [segs[j] for j in row_seg[segptr[k]: segptr[k + 1]]]
        assert own[0][0] == int(rowptr[r]) and own[-1][0] + own[-1][1] == int(rowptr[r + 1])
        assert all(a[0] + a[1] == b[0] for a, b in zip(own, own[1:]))
    hot = col | torch.where(torch.from_numpy(rng.random(col.numel()) < 0.3), -(2 ** 31), 0).to(torch.int32)
    q = DeviceGraph.long_row_plan(rowptr, hot, n_cols, seg_len, 64)
    assert all(torch.equal(q[k], v) if torch.is_tensor(v) else q[k] == v for k, v in p.items())


def test_partition_balances_nnz():
    from spex_b200.graph import build_norm_adj, partition_rows_by_nnz

    u, i = random_graph(2000, 300, 40000, 3)
    g = build_norm_adj(u, i, 2001, 300)
    for parts in (1, 2, 4, 8):
        b = partition_rows_by_nnz(g.rowptr, parts)
        assert b[0] == 0 and b[-1] == g.n_rows and len(b) == parts + 1
        assert all(b[k] <= b[k + 1] for k in range(parts))
        work = [g.rowptr[b[k + 1]] - g.rowptr[b[k]] for k in range(parts)]
        assert max(work) <= 1.25 * g.nnz / parts + g.degrees().max()
    blk = g.row_block(b[1], b[2])
    assert blk.rowptr[0] == 0 and blk.nnz == g.rowptr[b[2]] - g.rowptr[b[1]] and blk.row_offset == b[1]


def test_metrics_match_reference_formulas():
    from spex_b200 import metrics

    rng = np.random.default_rng(0)
    R = (rng.random((200, 50)) < 0.05).astype(float)
    R[0] = 0
    n_pos = np.maximum(R.sum(1), 1)
    rec, ndcg = metrics.batch_recall_ndcg(R, n_pos, [10, 20, 50])
    for r in range(200):
        for j, k in enumerate([10, 20, 50]):
            assert rec[r, j] == O.recall_at_k(list(R[r]), k, n_pos[r])
            assert abs(ndcg[r, j] - O.ndcg_at_k(list(R[r]), k)) < 1e-15
            assert abs(metrics.ndcg_at_k(list(R[r]), k) - O.ndcg_at_k(list(R[r]), k)) < 1e-15
    assert metrics.recall_at_k([1, 0], 2, 0) == 0.0


def test_rank_hits_has_heapq_dict_semantics():
    """batch_test.py:80-90: dict keyed by item, heapq.nlargest is a stable descending sort in
    insertion order; the positive is inserted last so it loses exact ties; a repeated item id
    keeps its first slot."""
    from spex_b200.batch_test import rank_hits

    rng = np.random.default_rng(1)
    for trial in range(50):
        n_c = 100
        cand = rng.choice(500, size=n_c, replace=False).astype(np.int32)
        scores = np.round(rng.normal(size=n_c), 1).astype(np.float32)  # many exact ties
        if trial % 3 == 0:
            cand[-1] = cand[3]  # positive equals one of the negatives
            scores[-1] = scores[3]
        if trial % 5 == 0:
            cand[10] = cand[11]
            scores[10] = scores[11]
        pos = [int(cand[-1])]
        rating = {}
        for c, s in zip(cand.tolist(), scores.tolist()):
            rating[c] = s
        top = heapq.nlargest(50, rating, key=rating.get)
        want = [1 if t in pos else 0 for t in top]
        got = rank_hits(scores[None], cand[None], [pos], 50)[0]
        assert got[: len(want)].tolist() == want and not got[len(want):].any()


def test_negative_sampler_consumes_the_reference_stream():
    from spex_b200.dataloader import LightTrainData, _PairSet

    rng = np.random.default_rng(0)
    nu, m = 200, 30  # dense: ~40% of draws collide
    u, i = random_graph(nu, m, 2400, 2)
    feats = np.stack([u, i], 1).tolist()
    ps = _PairSet(u, i, m, (nu + 1, m))
    np.random.seed(11)
    ref = []
    for x in feats:  # dataloader.py:253-260
        for _ in range(5):
            j = np.random.randint(m)
            while (x[0], j) in ps:
                j = np.random.randint(m)
            ref.append([x[0], j])
    tail_ref = np.random.randint(1 << 30)
    np.random.seed(11)
    d = LightTrainData(feats, m, ps)
    d.ng_sample()
    assert d.features_ng == ref
    assert np.random.randint(1 << 30) == tail_ref, "generator must end in the reference's state"
    assert len(d) == 6 * len(feats)
    assert d[0] == (feats[0][0], feats[0][1], 1) and d[len(feats)][2] == 0
    users, items, labels = d.arrays()
    assert not ps.contains(users[len(feats):], items[len(feats):]).any()


def test_capi_exports_every_declared_symbol_at_abi_3():
    hdr = open(os.path.join(ROOT, "include", "spex_b200.h")).read()
    hdr = re.sub(r"/\*.*?\*/", "", hdr, flags=re.S)
    declared = set(re.findall(r"\b(spex_[a-z0-9_]+)\s*\(", hdr))
    assert len(declared) >= 25
    lib = ctypes.CDLL(os.path.join(ROOT, "spex_b200", "libspex_b200.so"))
    for name in declared:
        assert hasattr(lib, name), f"{name} declared in include/spex_b200.h but not exported"
    from spex_b200 import _capi

    assert declared == set(_capi.SIGNATURES), declared ^ set(_capi.SIGNATURES)
    assert _capi.abi_version() == 3
    assert "SPEX_E_ALIGN" in _capi.error_string(-3)


def test_ctypes_signatures_match_the_header_prototypes():
    """Every binding in _capi.SIGNATURES passes exactly the parameters include/spex_b200.h declares, with the
    same kind (pointer / 32-bit int / 64-bit int / float) in the same position: a drift between the two is
    undefined behaviour at the first call, not an import error."""
    from spex_b200 import _capi

    hdr = open(os.path.join(ROOT, "include", "spex_b200.h")).read()
    hdr = re.sub(r"/\*.*?\*/", "", hdr, flags=re.S)
    protos = dict(re.findall(r"\b(?:int|int64_t|const char\s*\*)\s+(spex_[a-z0-9_]+)\s*\(([^;]*?)\)\s*;", hdr, flags=re.S))
    assert set(protos) == set(_capi.SIGNATURES)

    def kind_c(param):
        param = " ".join(param.split())
        if "*" in param:
            return "p"
        base = param.rsplit(" ", 1)[0] if " " in param else param
        return {"int32_t": "i32", "int": "i32", "uint32_t": "i32", "int64_t": "i64", "uint64_t": "i64",
                "float": "f"}[base.replace("const ", "").strip()]

    def kind_py(t):
        if t in (ctypes.c_int32, ctypes.c_int, ctypes.c_uint32):
            return "i32"
        if t in (ctypes.c_int64, ctypes.c_uint64):
            return "i64"
        if t is ctypes.c_float:
            return "f"
        return "p"      # c_void_p, c_char_p, POINTER(...)

    for name, (_res, argtypes) in _capi.SIGNATURES.items():
        params = [p for p in protos[name].split(",") if p.strip() and p.strip() != "void"]
        assert [kind_c(p) for p in params] == [kind_py(t) for t in argtypes], name


# spex_spmm_epilogue rules.  The addresses are never dereferenced: with n_rows = 0 the library returns after its
# argument checks, so these run without a GPU.
_A, _B = 0x10000, 0x20000          # 16-byte aligned
_MIS = _A + 4                      # misaligned


def _peers(*p):
    return (ctypes.c_void_p * len(p))(*p)


_ADAM = dict(adam_p=_A, adam_m=_B, adam_v=_A + 0x100, lr=1e-3, beta1=0.9, beta2=0.999, eps=1e-8, step=1)
_BADARG, _ALIGN = -1, -3
_EPILOGUE_CASES = [
    # one valid descriptor of each epilogue kind
    ("plain", dict(Y=_A, addend=_B, addend_scale=1.0, Z=_B, z_scale=0.5), 0),
    ("y_peers", dict(Z=_B, out_row_offset=7, y_peers_host=_peers(_A, _B), n_y_peers=2), 0),
    ("y_mcast", dict(Z=_B, out_row_offset=7, y_mcast=_A), 0),
    ("publish_peers", dict(Z=_B, pub_src=_A, pub_peers_host=_peers(_A, _B), n_pub_peers=2), 0),
    ("publish_mcast", dict(Z=_B, pub_src=_A, pub_mcast=_B), 0),
    ("adam", dict(_ADAM), 0),
    ("adam_publish_peers", dict(_ADAM, pub_peers_host=_peers(_A), n_pub_peers=1), 0),
    ("adam_publish_mcast", dict(_ADAM, Z=_B, pub_mcast=_B), 0),
    # one violating descriptor per rule
    ("negative_out_row_offset", dict(Z=_B, y_mcast=_A, out_row_offset=-1), _BADARG),
    ("y_mcast_and_peers", dict(Z=_B, y_mcast=_A, y_peers_host=_peers(_A), n_y_peers=1), _BADARG),
    ("y_peers_negative", dict(Z=_B, y_peers_host=_peers(_A), n_y_peers=-1), _BADARG),
    ("y_peers_over_8", dict(Z=_B, y_peers_host=_peers(*[_A] * 9), n_y_peers=9), _BADARG),
    ("y_peers_null_array", dict(Z=_B, n_y_peers=1), _BADARG),
    ("y_peers_null_peer", dict(Z=_B, y_peers_host=_peers(_A, None), n_y_peers=2), _BADARG),
    ("pub_peers_over_8", dict(Z=_B, pub_src=_A, pub_peers_host=_peers(*[_A] * 9), n_pub_peers=9), _BADARG),
    ("pub_peers_null_peer", dict(Z=_B, pub_src=_A, pub_peers_host=_peers(None), n_pub_peers=1), _BADARG),
    ("pub_src_without_destination", dict(Z=_B, pub_src=_A), _BADARG),
    ("pub_src_with_two_destinations", dict(Z=_B, pub_src=_A, pub_mcast=_B, pub_peers_host=_peers(_A),
                                           n_pub_peers=1), _BADARG),
    ("pub_mcast_without_source", dict(Z=_B, pub_mcast=_B), _BADARG),
    ("pub_peers_without_source", dict(Z=_B, pub_peers_host=_peers(_A), n_pub_peers=1), _BADARG),
    ("pub_src_with_adam", dict(_ADAM, pub_src=_A, pub_mcast=_B), _BADARG),
    ("adam_partial", dict(_ADAM, adam_v=None), _BADARG),
    ("adam_step_0", dict(_ADAM, step=0), _BADARG),
    ("misaligned_Y", dict(Y=_MIS), _ALIGN),
    ("misaligned_addend", dict(Z=_B, addend=_MIS), _ALIGN),
    ("misaligned_Z", dict(Z=_MIS), _ALIGN),
    ("misaligned_y_mcast", dict(Z=_B, y_mcast=_MIS), _ALIGN),
    ("misaligned_y_peer", dict(Z=_B, y_peers_host=_peers(_A, _MIS), n_y_peers=2), _ALIGN),
    ("misaligned_pub_src", dict(Z=_B, pub_src=_MIS, pub_mcast=_B), _ALIGN),
    ("misaligned_pub_mcast", dict(Z=_B, pub_src=_A, pub_mcast=_MIS), _ALIGN),
    ("misaligned_pub_peer", dict(Z=_B, pub_src=_A, pub_peers_host=_peers(_MIS), n_pub_peers=1), _ALIGN),
    ("misaligned_adam_p", dict(_ADAM, adam_p=_MIS), _ALIGN),
    ("misaligned_adam_m", dict(_ADAM, adam_m=_MIS), _ALIGN),
    ("misaligned_adam_v", dict(_ADAM, adam_v=_MIS), _ALIGN),
]


@pytest.mark.parametrize("fields,expected", [c[1:] for c in _EPILOGUE_CASES], ids=[c[0] for c in _EPILOGUE_CASES])
@pytest.mark.parametrize("n_sel", [-1, 0], ids=["all_rows", "empty_subset"])
def test_spmm_layer_validates_the_epilogue_descriptor(fields, expected, n_sel):
    """spex_spmm_layer_f32 checks every spex_spmm_epilogue rule before anything else, also for an empty row list."""
    from spex_b200 import _capi

    ep = _capi.SpmmEpilogue(**fields)
    rc = _capi.lib.spex_spmm_layer_f32(_A, _A, _A, _A, 0, 64, _A if n_sel == 0 else None, n_sel, None, 0, None, 0,
                                       None, ctypes.byref(ep), None, None)
    assert rc == expected, _capi.error_string(rc)
    assert _capi.lib.spex_spmm_layer_f32(_A, _A, _A, _A, 0, 64, None, -1, None, 0, None, 0, None, None, None,
                                         None) == _BADARG      # no descriptor


def test_product_path_refuses_cpu():
    from helpers import make_args
    from spex_b200.dataloader import SyntheticDataset
    from spex_b200.model import LightGCN

    ds = SyntheticDataset(50, 40, 400, seed=1)
    model = LightGCN(make_args(), ds)
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        model.computer()
    # the fused table backs both embeddings
    assert model.embedding_item.weight.data_ptr() == model._table.data_ptr() + 51 * 64 * 4
    # same RNG stream as the reference constructor => same initial weights under a shared seed
    torch.manual_seed(3)
    a = LightGCN(make_args(), ds).embedding_item.weight.detach().clone()
    torch.manual_seed(3)
    eu = torch.nn.Embedding(51, 64)
    ei = torch.nn.Embedding(40, 64)
    torch.nn.init.xavier_uniform_(eu.weight, gain=1)
    torch.nn.init.xavier_uniform_(ei.weight, gain=1)
    assert torch.equal(a, ei.weight.detach())


def test_no_product_module_imports_the_oracle():
    pkg = os.path.join(ROOT, "spex_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                src = open(os.path.join(dirpath, f)).read()
                assert not re.search(r"^\s*(from|import)\s+oracle", src, flags=re.M), f


def test_rebalance_equalises_modelled_cost():
    from spex_b200.graph import build_norm_adj, partition_rows_by_nnz, rebalance_bounds

    u, i = random_graph(3000, 400, 60000, 5)
    g = build_norm_adj(u, i, 3001, 400)
    b = partition_rows_by_nnz(g.rowptr, 4)
    # pretend the last two parts (item rows) are 1.5x slower per unit of work
    work = lambda a, c: (g.rowptr[c] - g.rowptr[a]) + 2 * (c - a)
    dens = [1.0, 1.0, 1.5, 1.5]
    times = [work(b[p], b[p + 1]) * dens[p] for p in range(4)]
    nb = rebalance_bounds(g.rowptr, b, times)
    assert nb[0] == 0 and nb[-1] == g.n_rows and all(nb[k] <= nb[k + 1] for k in range(4))
    # modelled cost of the new parts (same densities by old block) is equal within a few rows
    def cost(a, c):
        tot = 0.0
        for p in range(4):
            lo, hi = max(a, b[p]), min(c, b[p + 1])
            if hi > lo:
                tot += work(lo, hi) * dens[p]
        return tot
    costs = [cost(nb[p], nb[p + 1]) for p in range(4)]
    assert max(costs) - min(costs) <= 0.02 * sum(costs) / 4 + 3 * g.degrees().max()
    assert max(costs) < max(times)


def test_epoch_batches_follow_dataloader_shuffle():
    from torch.utils.data import DataLoader, TensorDataset

    from spex_b200.main_rec import epoch_batches

    ds = TensorDataset(torch.arange(1000))
    torch.manual_seed(5)
    ref = [b[0] for b in DataLoader(ds, batch_size=256, shuffle=True)]
    ref2 = [b[0] for b in DataLoader(ds, batch_size=256, shuffle=True)]
    torch.manual_seed(5)
    mine, mine2 = epoch_batches(1000, 256), epoch_batches(1000, 256)
    assert all(torch.equal(a, b) for a, b in zip(ref, mine)) and len(ref) == len(mine)
    assert all(torch.equal(a, b) for a, b in zip(ref2, mine2))


def test_ngcf_adjacency_builder_edge_cases():
    """D^-1 (A + I) (NGCF_SPEX/code/utility/load_data.py:122-166): duplicates collapse (dok
    assignment), isolated nodes keep their self loop with weight 1, rows sum to 1, and the scipy
    hand-off used by Model_Wrapper(data_config['norm_adj']) round-trips."""
    import scipy.sparse as sp

    from spex_b200.ngcf import build_ngcf_norm_adj, csr_from_scipy

    nu, ni = 5, 4
    users = np.array([0, 0, 0, 2, 2, 4])
    items = np.array([1, 1, 3, 0, 3, 3])          # (0,1) twice; user 1, user 3, item 2 isolated
    g = build_ngcf_norm_adj(users, items, nu, ni)
    A = sp.dok_matrix((nu + ni, nu + ni), dtype=np.float32)
    for u, i in zip(users, items):
        A[u, nu + i] = 1.0
        A[nu + i, u] = 1.0
    A = (A.tocsr() + sp.eye(nu + ni)).tocsr()
    want = sp.diags(1.0 / np.asarray(A.sum(1)).ravel()).dot(A).tocsr().astype(np.float32)
    want.sort_indices()
    assert np.array_equal(g.rowptr, want.indptr) and np.array_equal(g.col, want.indices)
    assert np.array_equal(g.val, want.data)
    rows = g.rows_of_entries()
    assert np.allclose(np.bincount(rows, weights=g.val, minlength=g.n_rows), 1.0)
    for node in (1, 3, nu + 2):                     # isolated: only the self loop, weight 1
        assert g.rowptr[node + 1] - g.rowptr[node] == 1 and g.val[g.rowptr[node]] == 1.0
    assert np.array_equal(rows[g.tpos], g.col) and np.array_equal(g.col[g.tpos], rows)
    h = csr_from_scipy(want)
    assert np.array_equal(h.rowptr, g.rowptr) and np.array_equal(h.col, g.col) and np.array_equal(h.val, g.val)
    assert np.array_equal(h.tpos, g.tpos)
    with pytest.raises(ValueError):
        build_ngcf_norm_adj(np.array([5]), np.array([0]), nu, ni)


def test_bench_reference_arm_contract_and_no_cpu_fallback():
    """bench.py --impl reference (the reference's CPU path, oracle port) prints ONE JSON line with
    the keys the driver reads; the product arm refuses to run without a GPU instead of falling back."""
    import json
    import subprocess
    import sys

    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    env = dict(os.environ, CUDA_VISIBLE_DEVICES="")
    out = subprocess.run([sys.executable, "bench.py", "--impl", "reference", "--steps", "1", "--warmup", "1",
                          "--cpu-sample-scale", "0.001"], cwd=root, env=env, capture_output=True, text=True,
                         timeout=600)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1
    j = json.loads(lines[0])
    assert j["impl"] == "reference" and j["metric"] == "lightgcn_propagation_gedges_per_s"
    assert j["unit"] == "GEdges/s" and j["higher_is_better"] is True and j["value"] > 0
    assert j["cpu_baseline"]["kind"] == "port" and j["cpu_baseline"]["cores"] >= 1 and j["cpu_baseline"]["sample"]
    assert j["cpu_baseline"]["value"] == j["value"] == j["e2e"]["value"]
    assert j["e2e"]["h2d_bytes_per_step"] == 0 and j["e2e"]["d2h_bytes_per_step"] == 0
    assert j["gpu_launches"] == 0 and "workload" in j["config"]
    ours = subprocess.run([sys.executable, "bench.py", "--steps", "1", "--warmup", "1"], cwd=root, env=env,
                          capture_output=True, text=True, timeout=600)
    assert ours.returncode != 0 and "no CPU fallback" in (ours.stderr + ours.stdout)


def test_bpr_triple_sampler():
    """uniform_sample_bpr (upstream-LightGCN semantics for the north-star bpr_loss): positives are
    training items of the user, negatives are not, users without interactions never appear, the
    draw is deterministic in the seed and roughly uniform over active users."""
    from spex_b200.dataloader import uniform_sample_bpr

    nu, m = 200, 60
    u, i = random_graph(nu, m, 3000, 5)
    keep = u != 7                                    # user 7 has no interactions
    u, i = u[keep], i[keep]
    S = uniform_sample_bpr(u, i, nu, m, n_samples=20000, seed=1)
    assert S.dtype == np.int64 and S.shape[1] == 3 and 19000 < S.shape[0] <= 20000
    train = set(zip(u.tolist(), i.tolist()))
    assert all((a, b) in train for a, b, _ in S[:2000].tolist())
    assert not any((a, c) in train for a, _, c in S.tolist())
    assert 7 not in set(S[:, 0].tolist())
    assert 0 <= S[:, 2].min() and S[:, 2].max() < m
    assert np.array_equal(S, uniform_sample_bpr(u, i, nu, m, n_samples=20000, seed=1))
    assert not np.array_equal(S, uniform_sample_bpr(u, i, nu, m, n_samples=20000, seed=2))
    counts = np.bincount(S[:, 0], minlength=nu)
    active = np.unique(u)
    assert counts[active].min() > 40 and counts[active].max() < 170      # ~100 each
    assert uniform_sample_bpr(u, i, nu, m).shape[0] <= u.size


def test_parser_keeps_the_reference_namespace():
    """Flag names, types and defaults of /root/reference/LightGCN_SPEX/code/lg_parser.py:3-24."""
    from spex_b200.lg_parser import parse_args_r

    want = {"cuda_id": "0", "data_path": "../data/", "dataset": "twitter", "nb_heads": 3, "recdim": 64,
            "layer": 3, "lr": 0.001, "dropout": 0, "keepprob": 0.6, "a_fold": 100, "epochs": 50,
            "seed": 2020, "A_split": 0, "batch_size": 256, "batchSize": 256, "hiddenSize": 64,
            "nonhybrid": False, "act": 1}
    got = vars(parse_args_r([]))
    assert got == want and all(type(got[k]) is type(v) for k, v in want.items())
    a = parse_args_r(["--dataset", "epinion2", "--layer", "2", "--nonhybrid", "--keepprob", "0.3", "--A_split", "1"])
    assert (a.dataset, a.layer, a.nonhybrid, a.keepprob, a.A_split) == ("epinion2", 2, True, 0.3, 1)
