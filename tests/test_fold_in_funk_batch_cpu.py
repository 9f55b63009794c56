"""Batched Funk-SVD fold-in without a GPU: GDRecommender.retrain_users / retrain_items check their
arguments before anything is drawn, changed or handed to the library, and the C entry point is
declared, exported and bound."""
import copy
import os
import re

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture()
def rec(monkeypatch):
    from mfrec_b200.lib import gd_estimator
    from mfrec_b200.recommendation import GDRecommender

    def no_native_call(*a, **kw):
        raise AssertionError("reached the native call")

    monkeypatch.setattr(gd_estimator, "fold_in", no_native_call)
    r = GDRecommender(20, 15, {'nbr_features': 6})
    rng = np.random.default_rng(0)
    r.svd_u, r.svd_v = rng.normal(0, 0.1, (6, 15)), rng.normal(0, 0.1, (6, 20))
    r.items_bias, r.users_bias = rng.normal(0, 0.1, 15), rng.normal(0, 0.1, 20)
    r.overall_bias = 3.5
    return r


def _ratings():
    rng = np.random.default_rng(1)
    idx = np.stack([rng.integers(0, 20, 100), rng.integers(0, 15, 100)], axis=1).astype(np.int32)
    return idx, rng.integers(1, 6, 100).astype(np.float64)


def _check_untouched(rec, before, call, exc):
    np.random.seed(3)
    want = np.random.random(2)
    np.random.seed(3)
    with pytest.raises(exc):
        call()
    assert np.array_equal(np.random.random(2), want)      # nothing drawn
    for name in ('svd_u', 'svd_v', 'items_bias', 'users_bias'):
        assert np.array_equal(getattr(rec, name), getattr(before, name)), name


def test_validation_raises_before_any_draw_or_native_call(rec):
    idx, r = _ratings()
    bad_item = idx.copy()
    bad_item[bad_item[:, 0] == 4, 1] = 15
    bad_user = idx.copy()
    bad_user[bad_user[:, 1] == 2, 0] = -1
    no_user_4 = idx[:, 0] != 4
    no_item_2 = idx[:, 1] != 2
    before = copy.deepcopy(rec)
    cases = [
        (ValueError, lambda: rec.retrain_users([1, 4, 1], idx, r)),
        (ValueError, lambda: rec.retrain_items([0, 0], idx, r)),
        (IndexError, lambda: rec.retrain_users([20], idx, r)),
        (IndexError, lambda: rec.retrain_users([-1], idx, r)),
        (IndexError, lambda: rec.retrain_items([3, 15], idx, r)),
        (IndexError, lambda: rec.retrain_users([4], bad_item, r)),
        (IndexError, lambda: rec.retrain_items([2], bad_user, r)),
        (ValueError, lambda: rec.retrain_users([4], idx.astype(np.int64), r)),      # int32 buffers, like retrain_user
        (ValueError, lambda: rec.retrain_items([4], idx, r.astype(np.float32))),
        # a listed row without ratings: refused up front (the loop would train the rows before it)
        (ValueError, lambda: rec.retrain_users([1, 4], np.ascontiguousarray(idx[no_user_4]),
                                               np.ascontiguousarray(r[no_user_4]))),
        (ValueError, lambda: rec.retrain_items([2], np.ascontiguousarray(idx[no_item_2]),
                                               np.ascontiguousarray(r[no_item_2]))),
    ]
    for exc, call in cases:
        _check_untouched(rec, before, call, exc)


def test_empty_batches_are_no_ops(rec):
    idx, r = _ratings()
    before = copy.deepcopy(rec)
    np.random.seed(3)
    want = np.random.random(2)
    np.random.seed(3)
    rec.retrain_users([], idx, r)
    rec.retrain_items(np.zeros(0, dtype=np.int64), idx, r)
    assert np.array_equal(np.random.random(2), want)
    for name in ('svd_u', 'svd_v', 'items_bias', 'users_bias'):
        assert np.array_equal(getattr(rec, name), getattr(before, name)), name


def test_the_recommender_hands_the_rows_in_list_order(monkeypatch):
    """The one native call gets the listed rows in list order, only their ratings in input order,
    and the features drawn in list order."""
    from mfrec_b200 import _native
    from mfrec_b200.lib import gd_estimator
    from mfrec_b200.recommendation import GDRecommender
    calls = []
    monkeypatch.setattr(gd_estimator, "fold_in", lambda *a: calls.append(a))
    rec = GDRecommender(20, 15, {'nbr_features': 6})
    rec.svd_u, rec.svd_v = np.zeros((6, 15)), np.zeros((6, 20))
    rec.items_bias, rec.users_bias, rec.overall_bias = np.zeros(15), np.zeros(20), 3.5
    idx, r = _ratings()
    users = [7, 2, 11]
    np.random.seed(5)
    rec.retrain_users(users, idx, r)
    (side, *_rest), = calls
    assert side == _native.FOLD_USERS
    got_idx, got_r, rows = calls[0][10], calls[0][11], calls[0][14]
    m = np.isin(idx[:, 0], users)
    assert np.array_equal(got_idx, idx[m]) and np.array_equal(got_r, r[m])
    assert list(rows) == users
    np.random.seed(5)
    for u in users:
        assert np.array_equal(rec.svd_v[:, u], np.random.normal(0.0, 0.1, 6))


def test_entry_point_is_declared_and_bound():
    from mfrec_b200 import _native
    with open(os.path.join(ROOT, "include", "mfrec_b200.h")) as f:
        header = f.read()
    assert re.search(r"\bint mfrec_fold_in_funk\s*\(", header)
    assert int(re.search(r"#define MFREC_B200_ABI_VERSION (\d+)", header).group(1)) >= 5
    assert "mfrec_fold_in_funk" in _native.EXPORTS
    assert (_native.FOLD_USERS, _native.FOLD_ITEMS) == (0, 1)
