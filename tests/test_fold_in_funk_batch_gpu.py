"""Batched Funk-SVD fold-in (GDRecommender.retrain_users / retrain_items, mfrec_fold_in_funk): one
device call leaves the recommender exactly as the loop of retrain_user / retrain_item over the same
rows under the sequential schedule -- factors, biases, the numpy RNG, what verbose prints and
gd_estimator.last_feature_*, bit for bit -- and every row equals the reference's arithmetic."""
import contextlib
import copy
import io

import numpy as np
import pytest

from mfrec_b200 import _native, synth

pytestmark = pytest.mark.gpu

# few epochs, a learning rate at which the improvement per epoch falls below min_improvement
# after a row-dependent number of epochs
PARAMS = {'min_epochs': 2, 'min_improvement': 1e-4, 'learning_rate': 0.05}


def _random_model(nu, ni, k, seed=0, extra=0, params=PARAMS, std=0.3):
    """Random factors ([k + extra] feature rows) and biases: a fold-in needs no trained model."""
    from mfrec_b200.recommendation import GDRecommender
    rec = GDRecommender(nu, ni, dict(params, nbr_features=k))
    rng = np.random.default_rng(seed)
    rec.svd_u = rng.normal(0.0, std, (k + extra, ni))
    rec.svd_v = rng.normal(0.0, std, (k + extra, nu))
    rec.items_bias = rng.normal(0.0, 0.2, ni)
    rec.users_bias = rng.normal(0.0, 0.2, nu)
    rec.overall_bias = 3.6
    return rec


@contextlib.contextmanager
def _sequential():
    from mfrec_b200.lib import gd_estimator
    saved = gd_estimator.options["schedule"]
    gd_estimator.options["schedule"] = "sequential"
    try:
        yield
    finally:
        gd_estimator.options["schedule"] = saved


def _assert_same(a, b):
    for name in ('svd_u', 'svd_v', 'items_bias', 'users_bias'):
        x, y = getattr(a, name), getattr(b, name)
        assert x.shape == y.shape, name
        assert np.array_equal(x, y), name


def _run_both(rec, loop, batch, seed=11):
    """Runs loop(copy) under the sequential schedule and batch(copy) from the same RNG state; checks
    they end identical, printed the same and leave the RNG and gd_estimator.last_feature_* in the same
    state.  Returns (loop, batch) copies."""
    from mfrec_b200.lib import gd_estimator
    a, b = copy.deepcopy(rec), copy.deepcopy(rec)
    outs = []
    for r, fn, sched in ((a, loop, _sequential), (b, batch, contextlib.nullcontext)):
        np.random.seed(seed)
        gd_estimator.last_feature_epochs = gd_estimator.last_feature_rmse = None
        buf = io.StringIO()
        with contextlib.redirect_stdout(buf), sched():
            fn(r)
        outs.append((buf.getvalue(), np.random.random(4), gd_estimator.last_feature_epochs,
                     gd_estimator.last_feature_rmse))
    _assert_same(a, b)
    assert outs[0][0] == outs[1][0]
    assert np.array_equal(outs[0][1], outs[1][1])       # the next RNG draw
    assert outs[0][2].dtype == outs[1][2].dtype
    assert np.array_equal(outs[0][2], outs[1][2])
    assert np.array_equal(outs[0][3], outs[1][3])
    return a, b


def _loop(method, rows, idx, r, epochs=None, **kw):
    """The single-row loop; collects every row's feature_epochs into `epochs`."""
    from mfrec_b200.lib import gd_estimator

    def run(rec):
        for x in rows:
            getattr(rec, method)(x, idx, r, **kw)
            if epochs is not None:
                epochs.append(gd_estimator.last_feature_epochs.copy())
    return run


def _assert_epochs_vary(epochs):
    """The rows stopped after different numbers of epochs: some feature has rows with different
    counts (at k = 300 the trailing term saturates the first features, which all stop at min_epochs)."""
    e = np.array(epochs)
    assert e.min() >= PARAMS['min_epochs'] and e.max() > e.min()
    assert (e != e[0]).any(axis=0).any()


@pytest.mark.parametrize("k", [1, 8, 40, 300])
def test_retrain_users_equals_the_sequential_loop(k):
    rec = _random_model(60, 40, k)
    d = synth.make_ratings(60, 40, 900, seed=1)
    users = np.random.default_rng(1).permutation(60)[:25]
    epochs = []
    _run_both(rec, _loop('retrain_user', users, d["idx"], d["r"], epochs),
              lambda x: x.retrain_users(users, d["idx"], d["r"]))
    _assert_epochs_vary(epochs)


@pytest.mark.parametrize("k", [1, 8, 40, 300])
def test_retrain_items_equals_the_sequential_loop(k):
    rec = _random_model(60, 40, k, seed=2)
    d = synth.make_ratings(60, 40, 900, seed=2)
    items = np.random.default_rng(2).permutation(40)[:15]
    epochs = []
    _run_both(rec, _loop('retrain_item', items, d["idx"], d["r"], epochs),
              lambda x: x.retrain_items(items, d["idx"], d["r"]))
    _assert_epochs_vary(epochs)


def test_verbose_prints_what_the_loop_prints():
    rec = _random_model(60, 40, 4)
    d = synth.make_ratings(60, 40, 900, seed=1)
    _run_both(rec, _loop('retrain_user', [3, 17, 5], d["idx"], d["r"], verbose=True),
              lambda x: x.retrain_users([3, 17, 5], d["idx"], d["r"], verbose=True))
    _run_both(rec, _loop('retrain_item', [9, 0], d["idx"], d["r"], verbose=True),
              lambda x: x.retrain_items([9, 0], d["idx"], d["r"], verbose=True))


def _oracle_row(rec, side, row, idx, r, u0, v0):
    """oracle.cpu.funk_train('with_bias_dev') on one row's ratings, from the factors u0 / v0 (the
    row's drawn initial features included): (row's factors [dim], epochs [dim], rmse [dim])."""
    from oracle import cpu
    dim = rec.dimensionality
    col = 0 if side == _native.FOLD_USERS else 1
    m = idx[:, col] == row
    u, v = np.ascontiguousarray(u0[:dim]), np.ascontiguousarray(v0[:dim])
    _, fe, fr = cpu.funk_train('with_bias_dev', rec.min_epochs, rec.min_improvement, dim, rec.feature_init,
                               rec.learning_rate, rec.K, u, v, np.ascontiguousarray(idx[m]),
                               np.ascontiguousarray(r[m]), rec.overall_bias, rec.items_bias, rec.users_bias,
                               1 if col == 0 else 0, 0 if col == 0 else 1)
    return (v[:, row] if col == 0 else u[:, row]), fe, fr


@pytest.mark.parametrize("side", [_native.FOLD_USERS, _native.FOLD_ITEMS])
def test_every_row_equals_the_oracle(side):
    """The reference's arithmetic (oracle.cpu.funk_train, pinned by tests/test_oracle.py) per row,
    from the features the recommender drew: factors, epochs and rmse, bit for bit."""
    from mfrec_b200.lib import gd_estimator
    rec = _random_model(60, 40, 8, seed=3)
    d = synth.make_ratings(60, 40, 900, seed=3)
    rows = [7, 30, 2, 11, 18] if side == _native.FOLD_USERS else [5, 0, 33]
    np.random.seed(6)
    init = rec.init_user_features if side == _native.FOLD_USERS else rec.init_item_features
    for x in rows:
        init(x)
    u0, v0 = rec.svd_u.copy(), rec.svd_v.copy()
    col = 0 if side == _native.FOLD_USERS else 1
    idx, r = d["idx"][np.isin(d["idx"][:, col], rows)], d["r"][np.isin(d["idx"][:, col], rows)]
    fe, fr = gd_estimator.fold_in(side, rec.min_epochs, rec.min_improvement, 8, rec.feature_init,
                                  rec.learning_rate, rec.K, rec.overall_bias, rec.svd_u, rec.svd_v,
                                  np.ascontiguousarray(idx), np.ascontiguousarray(r), rec.items_bias,
                                  rec.users_bias, rows)
    for p, x in enumerate(rows):
        want, fe_o, fr_o = _oracle_row(rec, side, x, d["idx"], d["r"], u0, v0)
        got = rec.svd_v[:, x] if side == _native.FOLD_USERS else rec.svd_u[:, x]
        assert np.array_equal(got, want)
        assert np.array_equal(fe[p], fe_o)
        assert np.array_equal(fr[p], fr_o)


def test_one_rating_rows_and_the_most_popular_item():
    """Rows with a single rating, and an item with thousands of ratings (the longest chain) retrained
    with items that have few."""
    nu, ni = 3000, 50
    rec = _random_model(nu, ni, 8, seed=4)
    rng = np.random.default_rng(4)
    # every user rates item 0; users < 40 rate nothing else, the others two more items
    pairs = [(u, 0) for u in range(nu)]
    pairs += [(u, int(i)) for u in range(40, nu) for i in rng.choice(np.arange(1, ni), 2, replace=False)]
    idx = np.array(pairs, dtype=np.int32)[rng.permutation(len(pairs))]
    r = rng.integers(1, 6, idx.shape[0]).astype(np.float64)
    users = [3, 17, 39, 0, 25]                      # one rating each
    _run_both(rec, _loop('retrain_user', users, idx, r), lambda x: x.retrain_users(users, idx, r))
    items = [4, 0, 31]                              # item 0: 3,000 ratings
    _run_both(rec, _loop('retrain_item', items, idx, r), lambda x: x.retrain_items(items, idx, r))


def test_rows_rating_one_common_item_run_in_one_launch():
    """Every user rates item 3: the rows share a frozen row but no written state, so they run in
    one launch, in no particular order -- and still give the loop's result."""
    rec = _random_model(60, 40, 8, seed=5)
    d = synth.make_ratings(60, 40, 900, seed=5)
    users = np.arange(0, 60, 3)
    extra = np.array([[u, 3] for u in users if not ((d["idx"][:, 0] == u) & (d["idx"][:, 1] == 3)).any()],
                     dtype=np.int32).reshape(-1, 2)
    idx = np.ascontiguousarray(np.r_[d["idx"], extra].astype(np.int32))
    r = np.r_[d["r"], np.full(extra.shape[0], 4.0)]
    assert set(users) <= set(idx[idx[:, 1] == 3, 0])
    ctx = _native.default_context()
    launches = []

    def batch(x):
        n0 = ctx.launch_count
        x.retrain_users(users, idx, r)
        launches.append(ctx.launch_count - n0)
    _run_both(rec, _loop('retrain_user', users, idx, r), batch)
    assert launches == [1]


@pytest.mark.parametrize("side", [_native.FOLD_USERS, _native.FOLD_ITEMS])
def test_feature_rows_beyond_dim_are_untouched(side):
    """gd_estimator.fold_in on factor arrays with more feature rows than dim (the recommender's own
    draws need exactly `dimensionality` rows): the sequential estimator_loop_with_bias_dev loop's
    result, and rows dim.. stay as they were."""
    from mfrec_b200.lib import gd_estimator
    dim, extra, nu, ni = 6, 3, 60, 40
    rng = np.random.default_rng(6)
    u0, v0 = rng.normal(0, 0.3, (dim + extra, ni)), rng.normal(0, 0.3, (dim + extra, nu))
    ib, ub = rng.normal(0, 0.2, ni), rng.normal(0, 0.2, nu)
    d = synth.make_ratings(nu, ni, 900, seed=6)
    col = 0 if side == _native.FOLD_USERS else 1
    rows = [4, 9, 31]
    hp = (PARAMS['min_epochs'], PARAMS['min_improvement'], dim, 0.1, PARAMS['learning_rate'], 0.05, 3.6)
    u1, v1 = u0.copy(), v0.copy()
    with _sequential():
        for x in rows:
            m = d["idx"][:, col] == x
            gd_estimator.estimator_loop_with_bias_dev(
                hp[0], hp[0], hp[1], dim, hp[3], hp[4], hp[4], hp[4], hp[5], hp[6], u1, v1,
                np.ascontiguousarray(d["idx"][m]), np.ascontiguousarray(d["r"][m]), ib, ub, nu, ni,
                1 - col, col)
    u2, v2 = u0.copy(), v0.copy()
    gd_estimator.fold_in(side, hp[0], hp[1], dim, hp[3], hp[4], hp[5], hp[6], u2, v2, d["idx"], d["r"], ib, ub,
                         rows)
    assert np.array_equal(u1, u2) and np.array_equal(v1, v2)
    assert np.array_equal(u2[dim:], u0[dim:]) and np.array_equal(v2[dim:], v0[dim:])
    assert not np.array_equal((v2 if col == 0 else u2)[:dim], (v0 if col == 0 else u0)[:dim])


@pytest.mark.parametrize("side", [_native.FOLD_USERS, _native.FOLD_ITEMS])
def test_frozen_side_unlisted_rows_and_biases_stay_bit_identical(side):
    rec = _random_model(60, 40, 8, seed=7)
    d = synth.make_ratings(60, 40, 900, seed=7)
    for name in ('svd_u', 'svd_v', 'items_bias', 'users_bias'):   # values float32 cannot hold
        setattr(rec, name, getattr(rec, name) + 1e-12)
    u0, v0, ib0, ub0 = rec.svd_u.copy(), rec.svd_v.copy(), rec.items_bias.copy(), rec.users_bias.copy()
    if side == _native.FOLD_USERS:
        rows = np.array([12, 40, 3, 33])
        rec.retrain_users(rows, d["idx"], d["r"])
        trained, t0, frozen, f0, n = rec.svd_v, v0, rec.svd_u, u0, 60
    else:
        rows = np.array([12, 0, 39])
        rec.retrain_items(rows, d["idx"], d["r"])
        trained, t0, frozen, f0, n = rec.svd_u, u0, rec.svd_v, v0, 40
    others = ~np.isin(np.arange(n), rows)
    assert np.array_equal(frozen, f0)
    assert np.array_equal(trained[:, others], t0[:, others])
    assert np.array_equal(rec.items_bias, ib0) and np.array_equal(rec.users_bias, ub0)
    assert not np.array_equal(trained[:, rows], t0[:, rows])


def test_errors_change_nothing_and_draw_nothing():
    rec = _random_model(60, 40, 8, seed=8)
    d = synth.make_ratings(60, 40, 900, seed=8)
    before = copy.deepcopy(rec)
    bad = d["idx"].copy()
    bad[bad[:, 0] == 5, 1] = 40                      # user 5 names an item that does not exist
    keep = d["idx"][:, 0] != 9                       # user 9 has no ratings
    idx9, r9 = np.ascontiguousarray(d["idx"][keep]), np.ascontiguousarray(d["r"][keep])
    cases = [
        (ValueError, lambda: rec.retrain_users([3, 5, 3], d["idx"], d["r"])),
        (ValueError, lambda: rec.retrain_items([1, 1], d["idx"], d["r"])),
        (IndexError, lambda: rec.retrain_users([3, 60], d["idx"], d["r"])),
        (IndexError, lambda: rec.retrain_items([-1], d["idx"], d["r"])),
        (IndexError, lambda: rec.retrain_users([2, 5], bad, d["r"])),
        (ValueError, lambda: rec.retrain_users([2], d["idx"].astype(np.int64), d["r"])),
        (ValueError, lambda: rec.retrain_items([2], d["idx"], d["r"].astype(np.float32))),
        (ValueError, lambda: rec.retrain_users([4, 9], idx9, r9)),
    ]
    for exc, call in cases:
        np.random.seed(8)
        after = np.random.random(3)
        np.random.seed(8)
        with pytest.raises(exc):
            call()
        assert np.array_equal(np.random.random(3), after)
        _assert_same(rec, before)
    np.random.seed(8)
    after = np.random.random(3)
    np.random.seed(8)
    rec.retrain_users([], d["idx"], d["r"])
    rec.retrain_items(np.zeros(0, np.int64), d["idx"], d["r"])
    assert np.array_equal(np.random.random(3), after)
    _assert_same(rec, before)


def test_native_entry_point_validates_before_writing():
    """mfrec_fold_in_funk itself: duplicate rows or a row without ratings -> ValueError, a row or a
    listed row's rating index out of range -> IndexError; the arrays are untouched.  Ratings naming
    no listed row are ignored even when their indices are out of range."""
    k, nu, ni = 8, 30, 20
    rng = np.random.default_rng(0)
    u, v = rng.normal(0, 0.1, (k, ni)), rng.normal(0, 0.1, (k, nu))
    ib, ub = rng.normal(0, 0.1, ni), rng.normal(0, 0.1, nu)
    idx = np.array([[1, 3], [2, 4], [1, 5], [99, 99], [2, -7]], dtype=np.int32)
    r = np.array([4.0, 2.0, 5.0, 1.0, 3.0])
    saved = [a.copy() for a in (u, v, ib, ub)]
    args = (_native.FOLD_USERS, 3, 1e-4, k, 0.1, 0.01, 0.05, 3.6, u, v, idx, r, ib, ub)
    for exc, rows in ((ValueError, [1, 1]), (IndexError, [1, nu]), (IndexError, [1, 2]), (ValueError, [1, 0])):
        with pytest.raises(exc):
            _native.fold_in_funk(*args, np.array(rows))
        for a, b in zip((u, v, ib, ub), saved):
            assert np.array_equal(a, b)
    fe, fr = _native.fold_in_funk(*args, np.array([1]))
    assert fe.shape == fr.shape == (1, k)
    u2, v2, ib2, ub2 = saved
    want = _native.train_funk(_native.FUNK_WITH_BIAS_DEV, 3, 3, 1e-4, k, 0.1, 0.01, 0.05, 3.6, u2, v2,
                              np.ascontiguousarray(idx[[0, 2]]), np.ascontiguousarray(r[[0, 2]]), ib2, ub2,
                              1, 0, schedule=_native.SCHED_SEQUENTIAL)
    assert np.array_equal(fe[0], want[0]) and np.array_equal(fr[0], want[1])
    for a, b in zip((u, v, ib, ub), (u2, v2, ib2, ub2)):
        assert np.array_equal(a, b)


def test_2000_users_on_an_ml20m_shaped_model():
    """ML-20M shape (138k users x 27k items), k = 40 and GDRecommender's default epochs: 2,000 users
    with 20-200 ratings drawn by item popularity retrained in one call.  20 sampled rows equal the
    per-row oracle; every other row is untouched."""
    from oracle import cpu
    nu, ni, _nnz, _k = synth.SHAPES["ml20m"]
    k = 40
    rec = _random_model(nu, ni, k, seed=9, params={}, std=0.1)
    _wu, wi = synth.marginals(nu, ni)
    rng = np.random.default_rng(9)
    users = rng.choice(nu, 2000, replace=False)
    idx = []
    for x in users:
        it = rng.choice(ni, int(rng.integers(20, 201)), replace=False, p=wi)
        idx.append(np.stack([np.full(it.shape[0], x), it], axis=1))
    idx = np.concatenate(idx).astype(np.int32)
    perm = rng.permutation(idx.shape[0])
    idx = np.ascontiguousarray(idx[perm])
    r = rng.integers(1, 6, idx.shape[0]).astype(np.float64)
    u0, v0 = rec.svd_u.copy(), rec.svd_v.copy()
    np.random.seed(10)
    rec.retrain_users(users, idx, r)
    np.random.seed(10)
    for x in users:
        v0[:, x] = np.random.normal(0.0, 0.1, k)
    assert np.array_equal(rec.svd_u, u0)
    others = np.ones(nu, bool)
    others[users] = False
    assert np.array_equal(rec.svd_v[:, others], v0[:, others])
    for x in rng.choice(users, 20, replace=False):
        m = idx[:, 0] == x
        one = np.ascontiguousarray(idx[m])
        one[:, 0] = 0
        v_row = np.ascontiguousarray(v0[:, [x]])
        cpu.funk_train('with_bias_dev', rec.min_epochs, rec.min_improvement, k, rec.feature_init,
                       rec.learning_rate, rec.K, u0.copy(), v_row, one, np.ascontiguousarray(r[m]),
                       rec.overall_bias, rec.items_bias, rec.users_bias[[x]], 1, 0)
        assert np.array_equal(rec.svd_v[:, x], v_row[:, 0])
