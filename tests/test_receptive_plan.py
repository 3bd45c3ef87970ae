"""ops.receptive_plan on CPU tensors: the rows each layer of a training step's propagation computes, for the
single-GPU model and the row-partitioned trainer alike.  The graph queries are written here over a small torch
CSR with hub rows; the sets are checked against their definition evaluated with scipy."""
import numpy as np
import pytest
import scipy.sparse as sp
import torch

from helpers import random_graph


def _graph():
    from spex_b200.graph import build_norm_adj

    u, i = random_graph(300, 120, 3000, 21, hub_items=2, hub_degree=200)
    return build_norm_adj(u, i, 301, 120)


def _queries(g, r0=0):
    """degree_sum / neighbors over the CSR `g` whose rows are the global rows [r0, r0 + g.n_rows); rows outside
    that range are ignored, as a rank ignores the rows it does not own."""
    rowptr = torch.from_numpy(g.rowptr)
    col = torch.from_numpy(g.col.astype(np.int64))
    row_of_edge = torch.repeat_interleave(torch.arange(g.n_rows), rowptr[1:] - rowptr[:-1])

    def own(rows):
        return rows[(rows >= r0) & (rows < r0 + g.n_rows)] - r0

    def degree_sum(rows):
        rows = own(rows)
        return int((rowptr[rows + 1] - rowptr[rows]).sum())

    def neighbors(rows):
        keep = torch.zeros(g.n_rows, dtype=torch.bool)
        keep[own(rows)] = True
        return torch.unique(col[keep[row_of_edge]])

    return degree_sum, neighbors


def _counted(fn, calls, key):
    def f(rows):
        calls[key] += 1
        return fn(rows)
    return f


def _batch_rows(g):
    """A few user rows and non-hub item rows: small enough to expand twice under wide limits."""
    deg = np.diff(g.rowptr)
    users = [3, 17, 101, 250]
    items = [301 + k for k in range(10, 120) if deg[301 + k] < 40][:3]
    return torch.tensor(sorted(users + items), dtype=torch.int64)


def _chain(g, S, K):
    """S = F[K], F[k] = S | N(F[k+1]) with no limit, and the edge count of every F[k] (index 0 unused)."""
    A = sp.csr_matrix((g.val, g.col, g.rowptr), shape=(g.n_rows, g.n_cols))
    F, E = [None] * (K + 1), [None] * (K + 1)
    F[K] = S.numpy()
    for k in range(K - 1, 0, -1):
        F[k] = np.union1d(F[K], A[F[k + 1]].indices)
    for k in range(1, K + 1):
        E[k] = int(A[F[k]].nnz)
    return F, E


def _same(a, b):
    return (a is None and b is None) or (a is not None and b is not None and torch.equal(a, b))


# (K, rule, stop): which limit refuses a set, and the first refused set k = K - stop
_STOPS = [(K, r, 0) for K in (1, 2, 3) for r in ("defaults", "none", "subset_S")] + \
         [(K, r, s) for r in ("expand", "subset_cand") for K in (2, 3) for s in range(1, K)]


@pytest.mark.parametrize("K,rule,stop", _STOPS)
def test_sets_match_the_definition_and_each_stop_rule(K, rule, stop, monkeypatch):
    """R[K] = S, R[k] = S | N(R[k+1]) against scipy; each limit refuses the set it is set to refuse, and the
    graph is queried once per set (a refused expansion gathers nothing)."""
    from spex_b200 import ops

    g = _graph()
    S = _batch_rows(g)
    F, E = _chain(g, S, K)
    assert all(E[k] > E[k + 1] for k in range(1, K))        # strictly growing sets: every threshold separates
    nnz = g.nnz
    sub, exp = 1.0, 1.0
    if rule == "subset_S":
        sub = (E[K] - 0.5) / nnz
    elif rule == "expand":
        exp = (E[K - stop + 1] - 0.5) / nnz
    elif rule == "subset_cand":
        sub = (E[K - stop] - 0.5) / nnz
    if rule == "defaults":
        sub, exp = ops.SUBSET_MAX_EDGE_FRAC, ops.EXPAND_MAX_EDGE_FRAC
    else:
        monkeypatch.setattr(ops, "SUBSET_MAX_EDGE_FRAC", sub)
        monkeypatch.setattr(ops, "EXPAND_MAX_EDGE_FRAC", exp)

    calls = {"degree_sum": 0, "neighbors": 0}
    degree_sum, neighbors = _queries(g)
    plan = ops.receptive_plan(S, K, nnz, _counted(degree_sum, calls, "degree_sum"),
                              _counted(neighbors, calls, "neighbors"))

    # the sets F[k] the limits accept, and the candidates F[k], k < K, that get built at all
    accepted, n_cand = [False] * (K + 1), 0
    if E[K] <= sub * nnz:
        accepted[K] = True
        for k in range(K - 1, 0, -1):
            if E[k + 1] > exp * nnz:
                break
            n_cand += 1
            if E[k] > sub * nnz:
                break
            accepted[k] = True
    if rule != "defaults":
        assert sum(accepted) == {"none": K, "subset_S": 0}.get(rule, stop)
    assert len(plan.R) == K + 1 and plan.R[0] is None and plan.edges[0] is None
    for k in range(1, K + 1):
        if accepted[k]:
            assert np.array_equal(plan.R[k].numpy(), F[k]) and plan.edges[k] == E[k]
        else:
            assert plan.R[k] is None and plan.edges[k] is None
    # one degree sum for S and one per candidate, one neighbour gather per candidate
    assert calls == {"degree_sum": 1 + n_cand, "neighbors": n_cand}


@pytest.mark.parametrize("P", [1, 2, 3])
@pytest.mark.parametrize("wide", [False, True])
def test_partitioned_queries_give_the_single_graph_plan(P, wide, monkeypatch):
    """The plan over P row blocks of graph.partition_rows_by_nnz - degree sums added up, neighbour lists
    concatenated, as the ranks of the partitioned trainer do - has the sets and edge counts of the whole graph."""
    from spex_b200 import ops
    from spex_b200.graph import partition_rows_by_nnz

    if wide:
        monkeypatch.setattr(ops, "SUBSET_MAX_EDGE_FRAC", 1.0)
        monkeypatch.setattr(ops, "EXPAND_MAX_EDGE_FRAC", 1.0)
    g = _graph()
    K = 3
    hub = 301 + int(np.argmax(np.diff(g.rowptr)[301:]))
    for S in (_batch_rows(g), torch.unique(torch.cat([_batch_rows(g), torch.tensor([hub])]))):
        one = ops.receptive_plan(S, K, g.nnz, *_queries(g))
        bounds = partition_rows_by_nnz(g.rowptr, P)
        blocks = [_queries(g.row_block(bounds[p], bounds[p + 1]), bounds[p]) for p in range(P)]
        part = ops.receptive_plan(S, K, g.nnz, lambda rows: sum(ds(rows) for ds, _ in blocks),
                                  lambda rows: torch.cat([nb(rows) for _, nb in blocks]))
        assert part.edges == one.edges
        assert all(_same(a, b) for a, b in zip(part.R, one.R))
        if wide:
            assert all(r is not None for r in one.R[1:])


def _backward_table_of_the_layer_loop(R, K, degree_sum, nnz, frac):
    """The backward row sets and sparse inputs as the restricted backward loop derived them before the plan
    answered them: layer j writes R[K-j] (j < K), its input is non-zero only on the rows the previous layer
    wrote (R[K] for j = 1), masked while those rows hold at most `frac` of nnz."""
    rows_tab, mask_tab = [None] * (K + 1), [None] * (K + 1)
    x_rows = R[K]
    for j in range(1, K + 1):
        sub = R[K - j] if j < K else None
        if x_rows is not None and degree_sum(x_rows) <= frac * nnz:
            mask_tab[j] = x_rows
        rows_tab[j] = sub
        x_rows = sub
    return rows_tab, mask_tab


@pytest.mark.parametrize("K", [1, 2, 3])
@pytest.mark.parametrize("sets", ["all", "last", "none"])
@pytest.mark.parametrize("sparse", ["never", "first", "always"])
def test_backward_layers_match_the_layer_loop(K, sets, sparse, monkeypatch):
    """plan.backward_layer(j) for every j = the table of the loop it replaces, with every set, only R[K], or no
    set restricted, and the sparse-input limit below, between and above the sets' edge counts (read when the
    question is asked, not when the plan is built)."""
    from spex_b200 import ops

    g = _graph()
    S = _batch_rows(g)
    _, E = _chain(g, S, K)
    nnz = g.nnz
    degree_sum, neighbors = _queries(g)
    monkeypatch.setattr(ops, "SUBSET_MAX_EDGE_FRAC", 1.0 if sets != "none" else (E[K] - 0.5) / nnz)
    monkeypatch.setattr(ops, "EXPAND_MAX_EDGE_FRAC", 1.0 if sets == "all" else (E[K] - 0.5) / nnz)
    plan = ops.receptive_plan(S, K, nnz, degree_sum, neighbors)
    assert sum(r is not None for r in plan.R) == {"all": K, "last": 1, "none": 0}[sets]
    frac = {"never": 0.0, "always": 1.0,
            "first": (E[K] + 0.5) / nnz if K == 1 else (E[K] + E[K - 1]) / 2 / nnz}[sparse]
    monkeypatch.setattr(ops, "SPARSE_INPUT_MAX_EDGE_FRAC", frac)
    rows_tab, mask_tab = _backward_table_of_the_layer_loop(plan.R, K, degree_sum, nnz, frac)
    for j in range(1, K + 1):
        rows, x_rows = plan.backward_layer(j)
        assert _same(rows, rows_tab[j]) and _same(x_rows, mask_tab[j]), j
    n_masks = sum(m is not None for m in mask_tab)
    if sets == "none" or sparse == "never":
        assert n_masks == 0
    elif sparse == "first":
        assert n_masks == 1 and mask_tab[1] is not None
    else:
        assert n_masks == (K if sets == "all" else 1)
