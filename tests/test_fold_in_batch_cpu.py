"""Batched fold-in without a GPU: KMFRecommender.add_users / retrain_users / retrain_items check
their arguments before anything is drawn, changed or handed to the library, and the C entry point
is declared, exported and bound."""
import copy
import os
import re

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture()
def rec(monkeypatch):
    from mfrec_b200.lib import kmf_train
    from mfrec_b200.recommendation import KMFRecommender

    def no_native_call(*a, **kw):
        raise AssertionError("reached the native call")

    monkeypatch.setattr(kmf_train, "fold_in", no_native_call)
    r = KMFRecommender(20, 15, {'nbr_features': 6})
    rng = np.random.default_rng(0)
    r.svd_u, r.svd_v = rng.normal(0, 0.1, (6, 15)), rng.normal(0, 0.1, (6, 20))
    r.items_bias, r.users_bias = np.zeros(15), np.zeros(20)
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
    assert rec.users_index == before.users_index and rec.users_label == before.users_label


def test_validation_raises_before_any_draw_or_native_call(rec):
    from mfrec_b200.recommendation.base import Error
    idx, r = _ratings()
    bad_item = idx.copy()
    bad_item[bad_item[:, 0] == 4, 1] = 15
    bad_user = idx.copy()
    bad_user[bad_user[:, 1] == 2, 0] = -1
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
        (ValueError, lambda: rec.retrain_users([4], idx, r.astype(np.float32))),
        (KeyError, lambda: rec.retrain_users([4], idx, r, kernel='train_cubic_kernel')),
        (IndexError, lambda: rec.add_users(['a', 'b'], [[1, 2], [3, 15]], [[5.0, 4.0], [3.0, 1.0]])),
        (IndexError, lambda: rec.add_users(['a'], [[-2]], [[5.0]])),
        (Error, lambda: rec.add_users(['a', 'b'], [[1, 2], [3]], [[5.0, 4.0], [3.0, 1.0]])),
        (ValueError, lambda: rec.add_users(['a', 'b'], [[1, 2]], [[5.0, 4.0]])),
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
    assert rec.add_users([], [], []) == []
    assert np.array_equal(np.random.random(2), want)
    for name in ('svd_u', 'svd_v', 'items_bias', 'users_bias'):
        assert np.array_equal(getattr(rec, name), getattr(before, name)), name


def test_entry_point_is_declared_and_bound():
    from mfrec_b200 import _native
    with open(os.path.join(ROOT, "include", "mfrec_b200.h")) as f:
        header = f.read()
    assert re.search(r"\bint mfrec_fold_in_kmf\s*\(", header)
    assert int(re.search(r"#define MFREC_B200_ABI_VERSION (\d+)", header).group(1)) >= 4
    assert "mfrec_fold_in_kmf" in _native.EXPORTS
    assert (_native.FOLD_USERS, _native.FOLD_ITEMS) == (0, 1)
