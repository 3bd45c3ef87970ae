"""Column-blocked long rows, several segments per warp (spmm_seg_runs_kernel: hub cells at the default L2 priority,
mid-row segments evict_first) against the one-segment-per-CTA kernel (spmm_seg_list_kernel), which the row-list
entry point runs for every segment when every row is listed.  Only cache priorities and scheduling differ, so every
output must be bit-identical."""
import numpy as np
import pytest
import torch

from oracle import lightgcn_oracle as O

pytestmark = pytest.mark.gpu

HUB_RUN = 8   # kHubRun in spex_b200/csrc/spmm.cu: hub cells per warp


def _graph(dev, seg_len):
    """A small graph whose plan holds hub cells and mid-row segments (the column-blocked list forced on a small
    table): item rows of graded degree next to a random bipartite graph."""
    from spex_b200 import ops
    from spex_b200.graph import build_norm_adj

    nu, m, seed = 900, 500, 18
    degs = (70, 150, 300, 500, 700, 850)
    u, i = O.random_bipartite(nu, m, 12000, seed)
    rng = np.random.default_rng(seed + 1)
    hu = np.concatenate([rng.choice(nu, d, replace=False) for d in degs])
    hi = np.repeat(np.arange(len(degs)), degs)
    key = np.unique(np.concatenate([u * m + i, hu * m + hi]))
    return ops.DeviceGraph.from_host(build_norm_adj(key // m, key % m, nu + 1, m), dev, seg_len=seg_len)


@pytest.mark.parametrize("hot", [False, True])
@pytest.mark.parametrize("seg_len", [32, 64])
def test_seg_runs_bit_identical_to_one_segment_per_cta(cuda_device, seg_len, hot, monkeypatch):
    from spex_b200 import ops

    # seg_len 32: single-batch cells, 1 edge to seg_len; seg_len 64: cells of several 32-edge batches
    monkeypatch.setattr(ops.DeviceGraph, "L2_WINDOW_BYTES", (16 if seg_len == 32 else 64) * 1024)
    monkeypatch.setattr(ops.DeviceGraph, "MIN_CB_COLS", 48)
    monkeypatch.setattr(ops.DeviceGraph, "HUB_EDGES_PER_BLOCK", 10 if seg_len == 32 else 100)
    g = _graph(cuda_device, seg_len)
    H = g.n_hub_seg
    assert 0 < H < g.n_seg
    assert H % HUB_RUN != 0 and g.n_seg % HUB_RUN != 0            # runs cut short at both list boundaries
    cnt = g.seg_count.cpu()
    assert bool((cnt[:H] > 0).all()) and bool((cnt <= seg_len).all())
    if seg_len == 32:
        assert bool((cnt == 1).any()) and bool((cnt[:H] == seg_len).any()) and bool((cnt[H:] == seg_len).any())
    else:
        assert bool((cnt[:H] > 32).any()) and bool((cnt[H:] > 32).any())
    if hot:
        assert g.mark_hot_columns(64, budget_bytes=16 * 1024) > 0
    N = g.n_rows
    torch.manual_seed(0)
    X = {D: torch.randn(N, D, device=cuda_device) for D in (32, 64, 128)}
    W = torch.randn(N, 64, device=cuda_device)
    long_rows = g.long_rows.long()
    sel = torch.cat([long_rows[::2], torch.arange(0, N, 7, device=cuda_device)]).unique()
    subset = g.row_subset(sel)
    assert subset[1] is not None and subset[1].numel() > 0
    act = torch.arange(0, N, 5, device=cuda_device)           # X is zero outside these rows
    Xs = torch.zeros_like(X[64])
    Xs[act] = X[64][act]

    def run():
        r = {f"spmm{D}": ops.spmm(g, x) for D, x in X.items()}
        E = (X[64] * 0.1).requires_grad_(True)
        out = ops.propagate_mean(E, g, 3)
        (out * W).sum().backward()
        r["mean"], r["grad"] = out.detach(), E.grad
        Yall = torch.zeros_like(X[64])
        ops.spmm_rows(g, X[64], None, Y=Yall)                     # all rows through the row-list entry point
        r["all_rows"] = Yall
        Ysub = torch.zeros_like(X[64])
        ops.spmm_rows(g, X[64], subset, Y=Ysub)                   # row subset (one segment per CTA in both arms)
        r["subset"] = Ysub
        Ymask = torch.zeros_like(X[64])
        ops.spmm_rows(g, Xs, None, Y=Ymask, x_nonzero=ops.nonzero_mask(N, act))   # sparse-input layer
        r["masked"] = Ymask
        r["dense_of_sparse"] = ops.spmm(g, Xs)
        torch.cuda.synchronize()
        return r

    every_row = g.row_subset(torch.arange(N, device=cuda_device))

    def one_segment_per_cta():
        """The same outputs with every row listed, so that every segment takes spmm_seg_list_kernel."""
        def layer(x, Y=None, **kw):
            if Y is None and kw.get("Z") is None:
                Y = torch.zeros_like(x)
            ops.spmm_rows(g, x, every_row, Y=Y, **kw)
            return Y

        r = {f"spmm{D}": layer(x) for D, x in X.items()}
        # the K=3 mean and its backward layer by layer, with the epilogues of spex_propagate_mean_f32 / _bwd_f32
        E0 = X[64] * 0.1
        out, grad = torch.empty_like(E0), torch.empty_like(E0)
        tmp = [torch.empty_like(E0), torch.empty_like(E0)]
        x = E0
        for k in range(3):
            last = k == 2
            layer(x, Y=None if last else tmp[k & 1], addend=E0 if k == 0 else out, Z=out, z_scale=0.25 if last else 1.0)
            x = tmp[k & 1]
        x = W                                                     # d sum(out * W) / d out
        for j in range(1, 4):
            last = j == 3
            layer(x, addend=W, Z=grad if last else tmp[(j - 1) & 1], z_scale=0.25 if last else 1.0)
            x = tmp[(j - 1) & 1]
        r["mean"], r["grad"] = out, grad
        r["all_rows"] = r["spmm64"]
        r["subset"] = torch.zeros_like(X[64])
        r["subset"][sel] = r["spmm64"][sel]
        r["masked"] = layer(Xs, x_nonzero=ops.nonzero_mask(N, act))
        r["dense_of_sparse"] = layer(Xs)
        torch.cuda.synchronize()
        return r

    new = run()
    ref = one_segment_per_cta()
    assert set(new) == set(ref)
    for k in new:
        assert torch.equal(new[k], ref[k]), k
    # the row subset and the sparse-input layer keep the one-segment kernel: their rows equal the new full layer's
    assert torch.equal(new["subset"][sel], new["spmm64"][sel])
    assert torch.equal(new["masked"], new["dense_of_sparse"])
    assert torch.equal(new["all_rows"], new["spmm64"])
    A = g.to_sparse_coo()
    assert float((new["spmm64"] - torch.sparse.mm(A, X[64])).abs().max()) < 1e-5 * float(new["spmm64"].abs().max())
