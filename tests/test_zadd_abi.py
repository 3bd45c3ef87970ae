"""spex_spmm_layer_zadd_f32's argument rules, checked before anything runs (n_rows = 0: the library returns after its
checks, so these run without a GPU; the addresses are never dereferenced)."""
import ctypes

import pytest

_A, _B = 0x10000, 0x20000          # 16-byte aligned
_MIS = _A + 4
_BADARG, _ALIGN = -1, -3
_ADAM = dict(adam_p=_A, adam_m=_B, adam_v=_A + 0x100, lr=1e-3, beta1=0.9, beta2=0.999, eps=1e-8, step=1)

_CASES = [
    ("no_z_add", dict(Z=_B), None, None, 0),
    ("z", dict(Z=_B), _A, _B, 0),
    ("adam", dict(_ADAM), _A, _B, 0),
    ("z_add_without_rows", dict(Z=_B), _A, None, _BADARG),
    ("rows_without_z_add", dict(Z=_B), None, _B, _BADARG),
    ("y_only", dict(Y=_A), _A, _B, _BADARG),
    ("misaligned_z_add", dict(Z=_B), _MIS, _B, _ALIGN),
    ("bad_descriptor_first", dict(Z=_MIS), _A, _B, _ALIGN),
]


@pytest.mark.parametrize("fields,z_add,rows,expected", [c[1:] for c in _CASES], ids=[c[0] for c in _CASES])
@pytest.mark.parametrize("n_sel", [-1, 0], ids=["all_rows", "empty_subset"])
def test_spmm_layer_zadd_validates_before_running(fields, z_add, rows, expected, n_sel):
    from spex_b200 import _capi

    ep = _capi.SpmmEpilogue(**fields)
    rc = _capi.lib.spex_spmm_layer_zadd_f32(_A, _A, _A, _A, 0, 64, _A if n_sel == 0 else None, n_sel, None, 0, None,
                                            0, None, ctypes.byref(ep), z_add, rows, None, None)
    assert rc == expected, _capi.error_string(rc)
