"""The added gradient of the SpMM layer epilogue (spex_spmm_layer_zadd_f32): on every kernel that writes Z - short rows,
the long-row fix-up, row subsets, sparse-input layers, 128-bit and 256-bit loads, the generic-D kernel - the flagged rows
get z_add's row after the scale, bit-equal to spex_spmm_layer_f32 followed by an fp32 add of those rows (and
spex_adam_f32 on that gradient where Adam is fused); unflagged rows never read z_add (it holds NaN there)."""
import ctypes as C

import numpy as np
import pytest
import torch

from test_gpu_spmm_edges import E_ALIGN, E_BADARG, SENT, Csr, _capi, _cols, _ep, _layer, _lib, _p, _st, _table

pytestmark = pytest.mark.gpu


def _zadd_layer(h, X, ep, z_add, flags, subset=None, nz=None):
    rows, slots, segs = subset if subset is not None else (None, None, None)
    g = h.g
    return _lib().spex_spmm_layer_zadd_f32(_p(g.rowptr), _p(g.col), _p(g.val), _p(X), g.n_rows, X.shape[1], _p(rows),
                                           -1 if rows is None else rows.numel(), _p(slots),
                                           0 if slots is None else slots.numel(), _p(segs),
                                           0 if segs is None else segs.numel(), _p(nz), C.byref(ep), _p(z_add),
                                           _p(flags), h.plan(X.shape[1]), _st())


def _graph(dev, seed, n=300):
    """Short rows and rows far above seg_len = 32 (the long-row pass), square so that X and Z share a row count."""
    rng = np.random.default_rng(seed)
    degs = rng.integers(0, 20, n)
    degs[::23] = rng.integers(70, 260, degs[::23].size)
    return Csr(_cols(rng, degs, n), n, rng, dev, seg_len=32), rng


def _inputs(h, D, dev, rng, align=32):
    n = h.n_rows
    X = _table(n, D, dev, align, rng.standard_normal((n, D)).astype(np.float32))
    add = _table(n, D, dev, 32, rng.standard_normal((n, D)).astype(np.float32))
    flags = torch.from_numpy((rng.random(n) < 0.4).astype(np.uint8)).to(dev)
    za = rng.standard_normal((n, D)).astype(np.float32)
    za[flags.cpu().numpy() == 0] = np.nan           # an unflagged row that read z_add would turn NaN
    return X, add, _table(n, D, dev, 32, za), flags


def _plus(Z, z_add, flags, rows=None):
    """Z with z_add added to its flagged rows (the listed ones) by torch: one fp32 add per element."""
    want = Z.clone()
    m = flags.bool()
    if rows is not None:
        keep = torch.zeros_like(m)
        keep[rows.long()] = True
        m &= keep
    want[m] = Z[m] + z_add[m]
    return want


CASES = [(32, "dense", 32), (64, "dense", 32), (128, "dense", 32), (64, "dense", 16), (128, "dense", 16),
         (64, "subset", 32), (32, "subset", 16), (64, "sparse_input", 32), (128, "sparse_input", 32), (48, "dense", 16)]


@pytest.mark.parametrize("D,kind,align", CASES, ids=[f"D{d}-{k}-ld{256 if a == 32 else 128}" for d, k, a in CASES])
def test_z_add_equals_layer_plus_torch_add(cuda_device, D, kind, align):
    h, rng = _graph(cuda_device, D + len(kind) + align)
    n = h.n_rows
    X, add, za, flags = _inputs(h, D, cuda_device, rng, align)
    sub = nz = rows = None
    if kind == "subset":
        rows = torch.from_numpy(rng.permutation(n)[: n // 2].astype(np.int64)).to(cuda_device)
        sub = h.g.row_subset(rows)
        assert sub[1] is not None and sub[1].numel() > 0          # long rows among the listed ones
    if kind == "sparse_input":
        keep = rng.random(n) < 0.2
        X[torch.from_numpy(~keep).to(cuda_device)] = 0.0
        nz = torch.from_numpy(keep.astype(np.uint8)).to(cuda_device)
    Zr = _table(n, D, cuda_device, fill=SENT)
    assert _layer(h, X, _ep(addend=add, Z=Zr, z_s=0.25), subset=sub, nz=nz) == 0
    Z = _table(n, D, cuda_device, fill=SENT)
    assert _zadd_layer(h, X, _ep(addend=add, Z=Z, z_s=0.25), za, flags, subset=sub, nz=nz) == 0
    want = _plus(Zr, za, flags, rows)
    assert torch.equal(Z, want)
    assert not torch.isnan(Z).any()
    if rows is not None:                                          # unlisted rows untouched
        unl = torch.ones(n, dtype=torch.bool, device=cuda_device)
        unl[rows] = False
        assert bool((Z[unl] == SENT).all())
    # z_add NULL: the new entry point is the old one
    Z0 = _table(n, D, cuda_device, fill=SENT)
    assert _zadd_layer(h, X, _ep(addend=add, Z=Z0, z_s=0.25), None, None, subset=sub, nz=nz) == 0
    assert torch.equal(Z0, Zr)


@pytest.mark.parametrize("D", [32, 64, 128])
@pytest.mark.parametrize("with_z", [False, True])
@pytest.mark.parametrize("subset", [False, True])
def test_z_add_reaches_the_fused_adam(cuda_device, D, with_z, subset):
    """Adam + publish: the gradient of a flagged row is Z + z_add, the same bits spex_adam_f32 gets from the layer's
    Z plus a torch add; the published rows are the updated p rows."""
    h, rng = _graph(cuda_device, 7 * D + with_z + 2 * subset)
    n = h.n_rows
    X, add, za, flags = _inputs(h, D, cuda_device, rng)
    rows = sub = None
    if subset:
        rows = torch.from_numpy(rng.permutation(n)[: n // 2].astype(np.int64)).to(cuda_device)
        sub = h.g.row_subset(rows)
    p0 = rng.standard_normal((n, D)).astype(np.float32)
    m0 = (rng.standard_normal((n, D)) * 0.1).astype(np.float32)
    v0 = (rng.random((n, D)) * 0.01).astype(np.float32)
    hyper = dict(lr=1e-3, b1=0.9, b2=0.999, eps=1e-8, step=3)
    p, m, v = (_table(n, D, cuda_device, 32, a) for a in (p0, m0, v0))
    Z = _table(n, D, cuda_device, fill=SENT) if with_z else None
    pub = _table(n, D, cuda_device, fill=SENT)
    ep = _ep(Z=Z, addend=add, z_s=0.25, pub_peers=[pub], adam=dict(p=p, m=m, v=v, **hyper))
    assert _zadd_layer(h, X, ep, za, flags, subset=sub) == 0
    # reference: the layer's Z over all rows, the flagged rows plus z_add, spex_adam_f32 on the whole table
    Zr = _table(n, D, cuda_device, fill=SENT)
    assert _layer(h, X, _ep(addend=add, Z=Zr, z_s=0.25)) == 0
    grad = _plus(Zr, za, flags)
    pe, me, ve = (_table(n, D, cuda_device, 32, a) for a in (p0, m0, v0))
    _capi().call("spex_adam_f32", _p(pe), _p(grad.contiguous()), _p(me), _p(ve), n * D, hyper["lr"], hyper["b1"],
                 hyper["b2"], hyper["eps"], hyper["step"], _st())
    sel = torch.ones(n, dtype=torch.bool, device=cuda_device)
    if subset:
        sel[:] = False
        sel[rows] = True
    for got, new, old in ((p, pe, p0), (m, me, m0), (v, ve, v0)):
        old = torch.from_numpy(old).to(cuda_device)
        assert torch.equal(got[sel], new[sel]) and torch.equal(got[~sel], old[~sel])
    assert torch.equal(pub[sel], pe[sel]) and bool((pub[~sel] == SENT).all())
    if with_z:
        assert torch.equal(Z[sel], grad[sel]) and bool((Z[~sel] == SENT).all())
    assert not torch.isnan(p).any()


def test_z_add_refusals_write_nothing(cuda_device):
    h, rng = _graph(cuda_device, 3)
    n, D = h.n_rows, 64
    X, add, za, flags = _inputs(h, D, cuda_device, rng)
    Y = _table(n, D, cuda_device, fill=SENT)
    Z = _table(n, D, cuda_device, fill=SENT)
    mis = _table(n + 1, D, cuda_device, fill=0.0).view(-1)[1: 1 + n * D].view(n, D)    # 4 bytes past alignment
    for ep, z, f, code in ((_ep(addend=add, Z=Z), za, None, E_BADARG),       # z_add without its flags
                           (_ep(addend=add, Z=Z), None, flags, E_BADARG),    # flags without z_add
                           (_ep(Y=Y), za, flags, E_BADARG),                  # neither Z nor Adam to add to
                           (_ep(addend=add, Z=Z), mis, flags, E_ALIGN)):
        assert _zadd_layer(h, X, ep, z, f) == code
    torch.cuda.synchronize()
    assert bool((Y == SENT).all()) and bool((Z == SENT).all())
