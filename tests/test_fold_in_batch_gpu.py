"""Batched fold-in (KMFRecommender.add_users / retrain_users / retrain_items, mfrec_fold_in_kmf): one
device call leaves the recommender exactly as the loop of add_user / retrain_user / retrain_item over
the same rows -- factors, biases, index / label maps, the numpy RNG, bit for bit."""
import contextlib
import copy
import io

import numpy as np
import pytest

from mfrec_b200 import _native, synth

pytestmark = pytest.mark.gpu

KERNELS = ('train_logistic_kernel', 'train_linear_kernel')
_TRAINED = {}


def _trained(k):
    """A small trained model (the set-up of test_fold_in_a_new_user) and its shuffled ratings."""
    from mfrec_b200.recommendation import KMFRecommender
    if k not in _TRAINED:
        nu, ni, nnz = 60, 40, 1500
        rec = KMFRecommender(nu, ni, {'nbr_epochs': 8, 'nbr_features': k})
        d = synth.make_ratings(nu, ni, nnz, seed=0)
        rec.set_ratings(d["idx"], d["r"])
        np.random.seed(4)
        rec.train(kernel='train_linear_kernel')
        _TRAINED[k] = (rec, d)
    rec, d = _TRAINED[k]
    return copy.deepcopy(rec), d


def _random_model(nu, ni, k, epochs, seed=0):
    """Random factors and biases (fold-in needs no trained model): for k the stratified trainer
    does not take, and for large shapes."""
    from mfrec_b200.recommendation import KMFRecommender
    rec = KMFRecommender(nu, ni, {'nbr_epochs': epochs, 'nbr_features': k})
    rng = np.random.default_rng(seed)
    rec.svd_u = rng.normal(0.0, 0.1, (k, ni))
    rec.svd_v = rng.normal(0.0, 0.1, (k, nu))
    rec.items_bias = rng.normal(0.0, 0.1, ni)
    rec.users_bias = rng.normal(0.0, 0.1, nu)
    return rec


def _new_users(n, ni, seed, lo=1, hi=12, common=None):
    rng = np.random.default_rng(seed)
    items, ratings = [], []
    for _ in range(n):
        c = int(rng.integers(lo, hi + 1))
        it = rng.choice(ni, c, replace=False)
        if common is not None and common not in it:
            it = np.r_[it[1:], common] if c else np.array([common])
        items.append(it.astype(np.int64))
        ratings.append(rng.integers(1, 6, it.shape[0]).astype(np.float64))
    return items, ratings


def _add_user_loop(rec, label, items, ratings, kernel):
    """add_user (kmf.py:149-172); its body with the other kernel for train_linear_kernel."""
    if kernel == 'train_logistic_kernel':
        return rec.add_user(label, items, ratings)
    new_id = rec._get_new_user_id()
    rec.users_index[label] = new_id
    rec.users_label[new_id] = label
    rec.svd_v = np.ascontiguousarray(np.c_[rec.svd_v, np.zeros(rec.dimensionality)])
    rec.users_bias = np.r_[rec.users_bias, 0.0]
    ratings_index = np.zeros([ratings.shape[0], 2], dtype=np.int32)
    ratings_index[:, 0] = new_id
    ratings_index[:, 1] = items
    rec.retrain_user(new_id, ratings_index, np.asarray(ratings, dtype=np.float64), kernel=kernel)
    return new_id


def _assert_same(a, b):
    for name in ('svd_u', 'svd_v', 'items_bias', 'users_bias'):
        x, y = getattr(a, name), getattr(b, name)
        assert x.shape == y.shape, name
        assert np.array_equal(x, y), name
    assert a.users_index == b.users_index
    assert a.users_label == b.users_label


def _run_both(rec, loop, batch, seed=11):
    """Runs loop(copy) and batch(copy) from the same RNG state; checks they end identical, printed the
    same and leave the RNG and kmf_train.last_rmse in the same state.  Returns (loop, batch) copies."""
    from mfrec_b200.lib import kmf_train
    a, b = copy.deepcopy(rec), copy.deepcopy(rec)
    outs = []
    for r, fn in ((a, loop), (b, batch)):
        np.random.seed(seed)
        buf = io.StringIO()
        with contextlib.redirect_stdout(buf):
            fn(r)
        outs.append((buf.getvalue(), np.random.random(4), None if kmf_train.last_rmse is None
                     else kmf_train.last_rmse.copy()))
    _assert_same(a, b)
    assert outs[0][0] == outs[1][0]
    assert np.array_equal(outs[0][1], outs[1][1])       # the next RNG draw
    assert np.array_equal(outs[0][2], outs[1][2], equal_nan=True)
    return a, b


@pytest.mark.parametrize("k", [8, 40, 128])
@pytest.mark.parametrize("kernel", KERNELS)
def test_add_users_equals_the_add_user_loop(kernel, k):
    rec, _ = _trained(k)
    items, ratings = _new_users(50, rec.nbr_items, seed=k)
    labels = ['new%d' % j for j in range(50)]
    a, b = _run_both(rec,
                     lambda r: [_add_user_loop(r, l, i, x, kernel) for l, i, x in zip(labels, items, ratings)],
                     lambda r: r.add_users(labels, items, ratings, kernel=kernel))
    assert b.nbr_users == rec.nbr_users + 50 and b.users_index['new7'] == rec.nbr_users + 7


@pytest.mark.parametrize("k", [8, 40, 128])
@pytest.mark.parametrize("kernel", KERNELS)
def test_retrain_users_equals_the_retrain_user_loop(kernel, k):
    rec, d = _trained(k)
    users = np.random.default_rng(1).permutation(rec.nbr_users)[:25]
    _run_both(rec,
              lambda r: [r.retrain_user(u, d["idx"], d["r"], kernel=kernel) for u in users],
              lambda r: r.retrain_users(users, d["idx"], d["r"], kernel=kernel))


@pytest.mark.parametrize("k", [8, 40, 128])
@pytest.mark.parametrize("kernel", KERNELS)
def test_retrain_items_equals_the_retrain_item_loop(kernel, k):
    rec, d = _trained(k)
    items = np.random.default_rng(2).permutation(rec.nbr_items)[:15]
    _run_both(rec,
              lambda r: [r.retrain_item(i, d["idx"], d["r"], kernel=kernel) for i in items],
              lambda r: r.retrain_items(items, d["idx"], d["r"], kernel=kernel))


@pytest.mark.parametrize("kernel", KERNELS)
def test_verbose_prints_what_the_loop_prints(kernel):
    rec, d = _trained(8)
    users = [3, 17, 5]
    keep = d["idx"][:, 0] != 17                       # user 17 has no ratings: the loop prints nothing for it
    idx, r = np.ascontiguousarray(d["idx"][keep]), np.ascontiguousarray(d["r"][keep])
    _run_both(rec,
              lambda x: [x.retrain_user(u, idx, r, verbose=True, kernel=kernel) for u in users],
              lambda x: x.retrain_users(users, idx, r, verbose=True, kernel=kernel))


def test_linear_rows_sharing_an_item_run_one_level_each():
    """Every new user rates item 3: with the linear kernel each fold-in writes b_3 and the next one
    reads it, so there is one row per level (one launch each) -- and still the loop's result."""
    rec, _ = _trained(40)
    items, ratings = _new_users(20, rec.nbr_items, seed=5, common=3)
    labels = ['c%d' % j for j in range(20)]
    ctx = _native.default_context()
    launches = []

    def batch(r):
        n0 = ctx.launch_count
        r.add_users(labels, items, ratings, kernel='train_linear_kernel')
        launches.append(ctx.launch_count - n0)

    _run_both(rec, lambda r: [_add_user_loop(r, l, i, x, 'train_linear_kernel')
                              for l, i, x in zip(labels, items, ratings)], batch)
    assert launches == [20]
    # the logistic kernel writes nothing of the frozen side: one launch for all rows
    b = copy.deepcopy(rec)
    n0 = ctx.launch_count
    b.add_users(labels, items, ratings)
    assert ctx.launch_count - n0 == 1


@pytest.mark.parametrize("kernel", KERNELS)
def test_rows_without_ratings(kernel):
    rec, d = _trained(40)
    items, ratings = _new_users(6, rec.nbr_items, seed=9)
    items[2], ratings[2] = np.zeros(0, np.int64), np.zeros(0)
    labels = ['e%d' % j for j in range(6)]
    _run_both(rec, lambda r: [_add_user_loop(r, l, i, x, kernel) for l, i, x in zip(labels, items, ratings)],
              lambda r: r.add_users(labels, items, ratings, kernel=kernel))
    keep = d["idx"][:, 0] != 9
    idx, r = np.ascontiguousarray(d["idx"][keep]), np.ascontiguousarray(d["r"][keep])
    _run_both(rec, lambda x: [x.retrain_user(u, idx, r, kernel=kernel) for u in (9, 4)],
              lambda x: x.retrain_users([9, 4], idx, r, kernel=kernel))
    # a batch whose rows have no ratings at all still draws their features, like the loop
    _run_both(rec, lambda x: x.retrain_user(9, idx, r, kernel=kernel),
              lambda x: x.retrain_users([9], idx, r, kernel=kernel))


@pytest.mark.parametrize("k", [1000, 29_100])
def test_wide_rows(k):
    """k = 1000: fewer than 32 lanes' rows fit in a block's shared memory; k = 29,100: not even one
    (the row stays in global memory).  Both still give the loop's result."""
    rec = _random_model(12, 10, k, epochs=2)
    d = synth.make_ratings(12, 10, 60, seed=3)
    for kernel in KERNELS:
        _run_both(rec, lambda r: [r.retrain_user(u, d["idx"], d["r"], kernel=kernel) for u in (4, 0, 7)],
                  lambda r: r.retrain_users([4, 0, 7], d["idx"], d["r"], kernel=kernel))
        _run_both(rec, lambda r: [r.retrain_item(i, d["idx"], d["r"], kernel=kernel) for i in (2, 9)],
                  lambda r: r.retrain_items([2, 9], d["idx"], d["r"], kernel=kernel))


def test_linear_batch_equals_the_oracle_per_row():
    """The reference's own arithmetic (oracle.cpu.kmf_train, float64, no FMA) run per row in list
    order, with the draws the recommender makes: bit for bit."""
    from oracle import cpu
    rec, d = _trained(8)
    users = [7, 30, 2, 51, 18]
    u0, v0, ib0, ub0 = rec.svd_u.copy(), rec.svd_v.copy(), rec.items_bias.copy(), rec.users_bias.copy()
    np.random.seed(6)
    rec.retrain_users(users, d["idx"], d["r"], kernel='train_linear_kernel')
    np.random.seed(6)
    for u in users:
        v0[:, u] = np.random.normal(0.0, 0.1, 8)
    for u in users:
        m = d["idx"][:, 0] == u
        cpu.kmf_train("linear", 8, 8, rec.learning_rate, rec.K_users, rec.K_items, rec.K_bias, u0, v0,
                      np.ascontiguousarray(d["idx"][m]), np.ascontiguousarray(d["r"][m]), ib0, ub0, 1, 0)
    assert np.array_equal(rec.svd_u, u0)
    assert np.array_equal(rec.svd_v, v0)
    assert np.array_equal(rec.items_bias, ib0)
    assert np.array_equal(rec.users_bias, ub0)


@pytest.mark.parametrize("kernel", KERNELS)
def test_frozen_side_and_unlisted_rows_stay_bit_identical(kernel):
    rec, d = _trained(40)
    # values float32 cannot hold: any float32 round trip would change them
    for name in ('svd_u', 'svd_v', 'items_bias', 'users_bias'):
        setattr(rec, name, getattr(rec, name) + 1e-12)
    u0, v0, ib0, ub0 = rec.svd_u.copy(), rec.svd_v.copy(), rec.items_bias.copy(), rec.users_bias.copy()
    users = np.array([12, 40, 3, 33])
    rec.retrain_users(users, d["idx"], d["r"], kernel=kernel)
    others = ~np.isin(np.arange(rec.nbr_users), users)
    assert np.array_equal(rec.svd_u, u0)
    assert np.array_equal(rec.svd_v[:, others], v0[:, others])
    assert np.array_equal(rec.users_bias[others], ub0[others])
    rated = np.isin(np.arange(rec.nbr_items), d["idx"][np.isin(d["idx"][:, 0], users), 1])
    if kernel == 'train_logistic_kernel':
        assert np.array_equal(rec.items_bias, ib0)
    else:   # the reference updates the item biases of the rated items too (kmf_train.pyx, SURVEY 8(a) A1)
        assert np.array_equal(rec.items_bias[~rated], ib0[~rated])
    assert not np.array_equal(rec.svd_v[:, users], v0[:, users])


def test_errors_change_nothing():
    rec, d = _trained(8)
    before = copy.deepcopy(rec)

    def unchanged():
        _assert_same(rec, before)
        assert np.array_equal(np.random.random(3), after)

    cases = [
        (ValueError, lambda: rec.retrain_users([3, 5, 3], d["idx"], d["r"])),
        (ValueError, lambda: rec.retrain_items([1, 1], d["idx"], d["r"])),
        (IndexError, lambda: rec.retrain_users([3, rec.nbr_users], d["idx"], d["r"])),
        (IndexError, lambda: rec.retrain_items([-1], d["idx"], d["r"])),
        (IndexError, lambda: rec.add_users(['a', 'b'], [np.array([1, 2]), np.array([rec.nbr_items])],
                                           [np.array([4.0, 3.0]), np.array([5.0])])),
    ]
    bad = d["idx"].copy()
    bad[bad[:, 0] == 5, 1] = rec.nbr_items       # user 5 names an item that does not exist
    cases.append((IndexError, lambda: rec.retrain_users([2, 5], bad, d["r"])))
    for exc, call in cases:
        np.random.seed(8)
        after = np.random.random(3)
        np.random.seed(8)
        with pytest.raises(exc):
            call()
        unchanged()
    # empty batches are no-ops
    np.random.seed(8)
    after = np.random.random(3)
    np.random.seed(8)
    rec.retrain_users([], d["idx"], d["r"])
    rec.retrain_items(np.zeros(0, np.int64), d["idx"], d["r"])
    assert rec.add_users([], [], []) == []
    unchanged()


def test_native_entry_point_validates_before_writing():
    """mfrec_fold_in_kmf itself: duplicate rows -> ValueError, a row or a listed row's rating index
    out of range -> IndexError; the arrays are untouched.  Ratings naming no listed row are ignored
    even when their indices are out of range."""
    k, nu, ni = 8, 30, 20
    rng = np.random.default_rng(0)
    u, v = rng.normal(0, 0.1, (k, ni)), rng.normal(0, 0.1, (k, nu))
    ib, ub = rng.normal(0, 0.1, ni), rng.normal(0, 0.1, nu)
    idx = np.array([[1, 3], [2, 4], [1, 5], [99, 99], [2, -7]], dtype=np.int32)
    r = np.array([4.0, 2.0, 5.0, 1.0, 3.0])
    saved = [a.copy() for a in (u, v, ib, ub)]
    args = (_native.KERNEL_LINEAR, _native.FOLD_USERS, 3, k, 0.01, 0.1, 0.1, 0.007, u, v, idx, r, ib, ub)
    with pytest.raises(ValueError):
        _native.fold_in_kmf(*args, np.array([1, 1]))
    with pytest.raises(IndexError):
        _native.fold_in_kmf(*args, np.array([1, nu]))
    with pytest.raises(IndexError):
        _native.fold_in_kmf(*args, np.array([1, 2]))           # rating 4 names item -7 for user 2
    for a, b in zip((u, v, ib, ub), saved):
        assert np.array_equal(a, b)
    rm = _native.fold_in_kmf(*args, np.array([1, 0]))           # user 0 has no rating
    assert rm.shape == (2, 3) and np.isfinite(rm[0]).all() and np.isnan(rm[1]).all()
    # against the single-row call
    u2, v2, ib2, ub2 = saved
    want = _native.train_kmf(_native.KERNEL_LINEAR, 3, k, 0.01, 0.1, 0.1, 0.007, u2, v2,
                             np.ascontiguousarray(idx[[0, 2]]), np.ascontiguousarray(r[[0, 2]]), ib2, ub2,
                             1, 0, schedule=_native.SCHED_SEQUENTIAL)
    assert np.array_equal(rm[0], want)
    for a, b in zip((u, v, ib, ub), (u2, v2, ib2, ub2)):
        assert np.array_equal(a, b)


@pytest.mark.parametrize("kernel", KERNELS)
def test_500_new_users_on_an_ml20m_shaped_model(kernel):
    """ML-20M shape (138k users x 27k items, k = 64), 500 new users with 20-200 ratings drawn by
    item popularity: the batch equals the add_user loop."""
    nu, ni, _nnz, k = synth.SHAPES["ml20m"]
    rec = _random_model(nu, ni, k, epochs=20, seed=1)
    _wu, wi = synth.marginals(nu, ni)
    rng = np.random.default_rng(2)
    items, ratings = [], []
    for _ in range(500):
        it = rng.choice(ni, int(rng.integers(20, 201)), replace=False, p=wi)
        items.append(it)
        ratings.append(rng.integers(1, 6, it.shape[0]).astype(np.float64))
    labels = ['m%d' % j for j in range(500)]
    _run_both(rec, lambda r: [_add_user_loop(r, l, i, x, kernel) for l, i, x in zip(labels, items, ratings)],
              lambda r: r.add_users(labels, items, ratings, kernel=kernel))
