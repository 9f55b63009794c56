"""als_wrmf with several devices in options["devices"], without a GPU: the same buffer checks as the
one-device path (same exception types and messages, raised before any native call), the dispatch to
train_als_wrmf_multi, and the native entry point's argument checks that need no device."""
import numpy as np
import pytest

from mfrec_b200 import _native
from mfrec_b200.lib import als_implicit


@pytest.fixture
def calls(monkeypatch):
    """Replaces the native entry points with recorders; restores options["devices"] afterwards."""
    seen = []
    monkeypatch.setattr(_native, "train_als_wrmf", lambda *a, **kw: seen.append(("one", a, kw)))
    monkeypatch.setattr(_native, "train_als_wrmf_multi", lambda *a, **kw: seen.append(("multi", a, kw)))
    monkeypatch.setattr(_native, "default_context", lambda device=-1: None)
    monkeypatch.setitem(als_implicit.options, "devices", list(als_implicit.options["devices"]))
    return seen


def _args(k=4, nu=5, ni=3):
    rng = np.random.default_rng(0)
    row = np.array([0, 1, 1], np.int32)
    col = np.array([0, 1], np.int32)
    return dict(nbr_epochs=2, dim=k, u=rng.random((k, ni)), v=rng.random((k, nu)), m=None, m_inv=None,
                ratings_users_row=row, ratings_users_col=col, ratings_items_row=row.copy(),
                ratings_items_col=col.copy(), nbr_users=nu, nbr_items=ni)


def _bad_cases():
    yield "u as a list", dict(u=[[0.0]])
    yield "u float32", dict(u=np.zeros((4, 3), np.float32))
    yield "v 1-d", dict(v=np.zeros(20))
    yield "u not C-contiguous", dict(u=np.asfortranarray(np.zeros((4, 3))))
    ro = np.zeros((4, 3))
    ro.setflags(write=False)
    yield "u read-only", dict(u=ro)
    yield "col int64", dict(ratings_users_col=np.array([0, 1], np.int64))
    yield "row 2-d", dict(ratings_items_row=np.zeros((1, 3), np.int32))
    yield "dim mismatch", dict(dim=5)
    yield "nbr_items mismatch", dict(nbr_items=4)
    yield "nbr_users mismatch", dict(nbr_users=6)


@pytest.mark.parametrize("name,override", list(_bad_cases()), ids=[n for n, _ in _bad_cases()])
def test_multi_path_validates_like_the_one_device_path(calls, name, override):
    errors = []
    for devices in ([], [0, 1], [0, 0, 0]):
        als_implicit.options["devices"] = devices
        a = _args()
        a.update(override)
        with pytest.raises(Exception) as ei:
            als_implicit.als_wrmf(**a)
        errors.append((type(ei.value), str(ei.value)))
    assert errors[1] == errors[0] and errors[2] == errors[0], (name, errors)
    assert errors[0][0] in (TypeError, ValueError)
    assert not calls


def test_dispatch(calls):
    als_implicit.options["devices"] = [1]
    a = _args()
    als_implicit.als_wrmf(**a)
    als_implicit.options["devices"] = [0, 1]
    als_implicit.als_wrmf(**a)
    als_implicit.options["devices"] = [2, 2, 2]
    als_implicit.als_wrmf(**a)
    assert [c[0] for c in calls] == ["one", "multi", "multi"]
    assert list(calls[1][1][0]) == [0, 1] and list(calls[2][1][0]) == [2, 2, 2]
    assert calls[1][1][1:3] == (2, 4) and calls[1][1][3] is a["u"] and calls[1][1][4] is a["v"]


def test_native_entry_point_checks_without_a_device():
    """Checks that come before any device is touched: an empty list, a NULL argument, bad sizes."""
    import os
    if not os.path.exists(_native.LIB_PATH):
        pytest.fail("libmfrec_b200.so is not built: run __graft_entry__.build()")
    a = _args()
    u, v = a["u"].copy(), a["v"].copy()
    row, col = a["ratings_users_row"], a["ratings_users_col"]
    with pytest.raises(ValueError, match="no devices"):
        _native.train_als_wrmf_multi([], 1, 4, u, v, row, col, row, col, 5, 3)
    with pytest.raises(ValueError, match="k=0"):
        _native.train_als_wrmf_multi([0, 1], 1, 0, u, v, row, col, row, col, 5, 3)
    with pytest.raises(IndexError, match="more rows"):
        _native.train_als_wrmf_multi([0, 1], 1, 4, u, v, np.zeros(9, np.int32), col, row, col, 5, 3)
    with pytest.raises(_native.MfrecError) as ei:
        _native.train_als_wrmf_multi([0] * 17, 1, 4, u, v, row, col, row, col, 5, 3)
    assert ei.value.code == _native.ERR_UNSUPPORTED
    assert np.array_equal(u, a["u"]) and np.array_equal(v, a["v"])
