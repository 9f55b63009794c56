"""Top-N, predictions and similarity served from several shards of one process
(mfrec_model_topn_sweep_multi, mfrec_model_predict_multi, _native.ModelSet) against the one-device
calls: items, scores and counts must be EQUAL, not close.  Shards that share the test GPU run the
whole split path (one context, stream and model copy per shard, one host thread each); the last test
uses every GPU of the process."""
import numpy as np
import pytest

from mfrec_b200 import synth

pytestmark = pytest.mark.gpu


def _device():
    import torch
    return torch.cuda.current_device()


def _factors(nu, ni, k, seed):
    u, v = synth.init_factors(nu, ni, k, seed=seed)
    rng = np.random.default_rng(seed)
    return u, v, rng.normal(0, 0.2, ni), rng.normal(0, 0.2, nu)


def _models(devices, k, ni, nu, u, v, ib, ub):
    from mfrec_b200 import _native
    one = _native.Model(k, ni, nu, u, v, ib, ub, ctx=_native.default_context(devices[0]))
    return one, _native.ModelSet(devices, k, ni, nu, u, v, ib, ub)


def _rated_csr(users, ni, per_user, seed):
    """Rated-items CSR of a user list; a user listed twice gets the same list both times."""
    rng = np.random.default_rng(seed)
    lists = {int(x): np.sort(rng.choice(ni, int(rng.integers(0, 2 * per_user)), replace=False)) for x in set(users.tolist())}
    parts = [lists[int(x)] for x in users]
    indptr = np.zeros(len(users) + 1, np.int64)
    indptr[1:] = np.cumsum([len(p) for p in parts])
    return indptr, (np.concatenate(parts) if parts else np.zeros(0)).astype(np.int32)


def _same(a, b, sweep=True):
    (i0, s0, c0, st0), (i1, s1, c1, st1) = a, b
    assert np.array_equal(i1, i0) and np.array_equal(s1, s0) and np.array_equal(c1, c0)
    # users redone, FLOPs, overflows, padded K and z are exact; the rest are means / times
    for j in (0, 3, 4, 5, 6):
        assert st1[j] == st0[j], (j, st0, st1)
    assert abs(st1[1] - st0[1]) <= 1e-12 * max(1.0, abs(st0[1]))
    assert (st0[3] > 0) == sweep


def _both(one, ms, predictor, users, nc, indptr, rated, N, mu=3.4):
    a = one.topn(predictor, users, nc, indptr, rated, N, mu, 1.0, 5.0, sweep=True)
    b = ms.topn(predictor, users, nc, indptr, rated, N, mu, 1.0, 5.0, sweep=True)
    return a, b


# KB = ceil((k + bias column) / 64): 20 -> 1, 64 + bias -> 2, 128 + bias -> 3, 250 -> 4, 250 + bias -> 4 with
# the covariance read through L2 (ka > 240)
CASES = [(20, "predict_rating"), (64, "predict_rating_with_bias"), (128, "predict_logistic"), (250, "predict_dot"),
         (250, "predict_rating_with_bias")]


@pytest.mark.parametrize("shards", [2, 3, 5])
@pytest.mark.parametrize("k,predictor", CASES)
def test_all_users_equal_one_device(k, predictor, shards):
    """users = NULL (all users), 1,300 users: not a multiple of 512; 2 shards cut at 512, 3 and 5 evenly."""
    d = _device()
    nu, ni, N = 1300, 3000, 25
    one, ms = _models([d] * shards, k, ni, nu, *_factors(nu, ni, k, seed=k))
    indptr, rated = _rated_csr(np.arange(nu), ni, 30, seed=1)
    a, b = _both(one, ms, predictor, None, ni, indptr, rated, N)
    _same(a, b)


@pytest.mark.parametrize("shards", [2, 3, 5])
def test_user_list_in_any_order_with_a_duplicate(shards):
    d = _device()
    nu, ni, k, N = 2000, 2100, 96, 17
    one, ms = _models([d] * shards, k, ni, nu, *_factors(nu, ni, k, seed=5))
    rng = np.random.default_rng(2)
    users = rng.permutation(nu)[:1100].astype(np.int32)
    users = np.insert(users, 700, users[3])                   # listed twice, in different shares
    indptr, rated = _rated_csr(users, ni, 20, seed=3)
    a, b = _both(one, ms, "predict_linear", users, 2050, indptr, rated, N)
    _same(a, b)
    assert np.array_equal(a[0][3], a[0][700])


def test_shares_below_128_users_keep_the_sweep():
    """300 users over 3 and 5 shards: every share is under the 128 users below which a one-device
    call takes the exact path, but the whole call is not, so every share sweeps."""
    d = _device()
    nu, ni, k, N = 300, 2000, 64, 20
    for shards in (3, 5):
        one, ms = _models([d] * shards, k, ni, nu, *_factors(nu, ni, k, seed=shards))
        indptr, rated = _rated_csr(np.arange(nu), ni, 10, seed=4)
        a, b = _both(one, ms, "predict_dot", None, ni, indptr, rated, N)
        _same(a, b)


def test_a_call_under_128_users_is_exact_on_every_shard():
    d = _device()
    nu, ni, k, N = 1000, 2000, 64, 20
    one, ms = _models([d] * 3, k, ni, nu, *_factors(nu, ni, k, seed=6))
    users = np.arange(0, 1000, 8, dtype=np.int32)[:127]
    indptr, rated = _rated_csr(users, ni, 10, seed=5)
    a, b = _both(one, ms, "predict_rating_with_bias", users, ni, indptr, rated, N)
    _same(a, b, sweep=False)
    # and the exact path is what the one-device call gives those users
    wi, ws, wc = one.topn("predict_rating_with_bias", users, ni, indptr, rated, N, 3.4, 1.0, 5.0)
    assert np.array_equal(b[0], wi) and np.array_equal(b[1], ws) and np.array_equal(b[2], wc)


def test_more_shards_than_users():
    d = _device()
    nu, ni, k, N = 50, 400, 20, 5
    one, ms = _models([d] * 5, k, ni, nu, *_factors(nu, ni, k, seed=7))
    users = np.array([9, 2, 40], np.int32)
    indptr, rated = _rated_csr(users, ni, 5, seed=6)
    a, b = _both(one, ms, "predict_rating", users, ni, indptr, rated, N)
    _same(a, b, sweep=False)


def test_heavy_tailed_scores_take_the_exact_fallback():
    """A few huge item rows: thresholds misjudge, some users are redone exactly in both calls."""
    d = _device()
    nu, ni, k, N = 1500, 3000, 32, 30
    u, v, ib, ub = _factors(nu, ni, k, seed=8)
    u[:, :40] *= 25.0
    one, ms = _models([d] * 3, k, ni, nu, u, v, ib, ub)
    a, b = _both(one, ms, "predict_dot", None, ni, None, None, N)
    _same(a, b)
    assert a[3][0] > 0 and b[3][0] > 0


@pytest.mark.parametrize("shards", [2, 3, 5])
def test_predict_equals_one_device(shards):
    d = _device()
    nu, ni, k = 900, 700, 40
    one, ms = _models([d] * shards, k, ni, nu, *_factors(nu, ni, k, seed=9))
    rng = np.random.default_rng(3)
    for n in (10001, 3):
        pairs = np.c_[rng.integers(0, nu, n), rng.integers(0, ni, n)].astype(np.int32)
        real = rng.uniform(1, 5, n)
        real[::7] = np.nan                                    # dropped from the sums
        for predictor in ("predict_rating_with_bias", "predict_logistic", "predict_dot"):
            o0, s0 = one.predict(predictor, pairs, real, 3.4, 1.0, 5.0, want_stats=True)
            o1, s1 = ms.predict(predictor, pairs, real, 3.4, 1.0, 5.0, want_stats=True)
            assert np.array_equal(o1, o0)
            np.testing.assert_allclose(s1, s0, rtol=1e-12, atol=0)
            assert s1[2] == s0[2]


@pytest.fixture()
def serve_devices():
    """Sets options["devices"] for the test and restores it afterwards."""
    from mfrec_b200.lib._buffers import options
    saved = list(options["devices"])

    def use(devices):
        options["devices"] = list(devices)

    yield use
    options["devices"] = saved


def _evaluate(rec, held, predictor):
    from mfrec_b200.recommendation import metrics
    np.random.seed(0)
    pr = metrics.precision_recall(rec, held, nbr_recommendations=10, predictor=predictor)
    users = np.unique(held[:, 0]).astype(np.int32)
    top = rec.find_recommended_items_batch(users, 10, predictor)
    stats = np.array(rec.last_topn_stats)
    sim = rec.similar_items_batch(np.arange(rec.nbr_items), nbr_recommendations=6)
    rmse, errors = metrics.test_predict_rating(rec, held, nbr_samples=held.shape[0], predictor=predictor)
    one_user = rec.find_recommended_items(user_index=int(users[0]), nbr_recommendations=10, predictor=predictor)
    return pr, top, stats, sim, rmse, errors, one_user


def _check_recommender(rec, held, predictor, serve_devices):
    from mfrec_b200 import _native
    d = _device()
    serve_devices([])
    want = _evaluate(rec, held, predictor)
    assert isinstance(rec._resident_model(), _native.Model)
    serve_devices([d, d, d])
    got = _evaluate(rec, held, predictor)
    assert isinstance(rec._resident_model(), _native.ModelSet) and len(rec._resident_model().models) == 3
    assert got[0] == want[0]
    for a, b in zip(got[1], want[1]):
        assert np.array_equal(a, b)
    assert got[2][3] == want[2][3] > 0 and got[2][0] == want[2][0]   # merged stats: the sweep ran on the shards
    for a, b in zip(got[3], want[3]):
        assert np.array_equal(a, b)
    assert got[4] == want[4] and np.array_equal(got[5], want[5])
    assert got[6] == want[6]


def test_kmf_recommender_on_three_shards(serve_devices):
    from mfrec_b200.recommendation import KMFRecommender
    nu, ni, k = 1500, 800, 24
    d = synth.make_ratings(nu, ni, 40000, seed=4, shuffle_seed=None)
    rec = KMFRecommender(nu, ni, {'nbr_epochs': 5, 'nbr_features': k})
    rec.set_ratings(d["idx"], d["r"])
    serve_devices([])
    np.random.seed(1)
    rec.train(kernel='train_linear_kernel')
    rng = np.random.default_rng(3)
    held = np.c_[rng.integers(0, nu, 3000), rng.integers(0, ni, 3000), rng.integers(1, 6, 3000)].astype(np.float64)
    assert np.unique(held[:, 0]).shape[0] >= 128
    _check_recommender(rec, held, 'predict_linear', serve_devices)


def test_wrmf_recommender_on_three_shards(serve_devices):
    from mfrec_b200.recommendation import WRMFRecommender
    nu, ni, k = 1400, 700, 32
    d = synth.make_ratings(nu, ni, 30000, seed=6, shuffle_seed=None)
    rec = WRMFRecommender(nu, ni, {'nbr_epochs': 3, 'nbr_features': k})
    rec.set_ratings(d["idx"], np.ones(d["idx"].shape[0]))
    serve_devices([])
    rec.train()
    rng = np.random.default_rng(4)
    held = np.c_[rng.integers(0, nu, 2500), rng.integers(0, ni, 2500), np.ones(2500)]
    _check_recommender(rec, held, 'predict', serve_devices)


def test_errors_change_nothing():
    from mfrec_b200 import _native
    d = _device()
    nu, ni, k, N = 1200, 2000, 32, 10
    u, v, ib, ub = _factors(nu, ni, k, seed=11)
    _one, ms = _models([d] * 3, k, ni, nu, u, v, ib, ub)
    ok = np.arange(nu, dtype=np.int32)
    users = ok.copy()
    users[-1] = nu                                            # the last share holds the bad id
    out = (np.full((nu, N), -7, np.int32), np.full((nu, N), -7.0), np.full(nu, -7, np.int32))
    with pytest.raises(IndexError):
        ms.topn("predict_dot", users, ni, None, None, N, sweep=True, out=out)
    assert (out[0] == -7).all() and (out[1] == -7.0).all() and (out[2] == -7).all()
    # models that do not match: another k, another item count, one context twice
    good = ms.models
    pairs = np.c_[np.arange(100) % nu, np.arange(100) % ni].astype(np.int32)
    for bad in (_native.Model(k + 40, ni, nu, np.zeros((k + 40, ni)), np.zeros((k + 40, nu)), ctx=good[1].ctx),
                _native.Model(k, ni - 1, nu, u[:, :-1], v, ctx=good[1].ctx)):
        ms.models = (good[0], bad, good[2])
        with pytest.raises(ValueError):
            ms.topn("predict_dot", ok, ni, None, None, N, sweep=True, out=out)
        assert (out[0] == -7).all() and (out[1] == -7.0).all() and (out[2] == -7).all()
        pred = np.full(100, -7.0)
        with pytest.raises(ValueError):
            _predict_into(ms, pairs, pred)
        assert (pred == -7.0).all()
    ms.models = (good[0], good[0], good[2])
    with pytest.raises(ValueError):
        ms.topn("predict_dot", ok, ni, None, None, N, sweep=True, out=out)
    assert (out[0] == -7).all()
    ms.models = good
    # the set still works after the refusals
    items, scores, counts, stats = ms.topn("predict_dot", ok, ni, None, None, N, sweep=True)
    assert stats[3] > 0 and (counts == N).all()


def _predict_into(ms, pairs, out):
    import ctypes as C
    from mfrec_b200 import _native
    _native._check(_native.lib().mfrec_model_predict_multi(
        _native._handles([m.ctx for m in ms.models]), _native._handles(ms.models), C.c_int(len(ms.models)),
        C.c_int(_native.PREDICTORS["predict_dot"]), _native._ptr(pairs), None, C.c_int(0), C.c_int64(pairs.shape[0]),
        C.c_double(0.0), C.c_double(1.0), C.c_double(5.0), _native._ptr(out), None), ms.ctx.handle)


def test_all_gpus_of_the_process():
    import torch
    n = torch.cuda.device_count()
    if n < 2:
        pytest.skip("needs at least 2 GPUs")
    nu, ni, k, N = 5000, 4000, 128, 50
    u, v, ib, ub = _factors(nu, ni, k, seed=12)
    indptr, rated = _rated_csr(np.arange(nu), ni, 30, seed=7)
    for devices in (list(range(n)), [x for x in range(n) for _ in range(2)][:16]):
        one, ms = _models(devices, k, ni, nu, u, v, ib, ub)
        _same(*_both(one, ms, "predict_logistic", None, ni, indptr, rated, N))
        pairs = np.c_[np.arange(20000) % nu, (np.arange(20000) * 7) % ni].astype(np.int32)
        o0, _ = one.predict("predict_logistic", pairs, None, 3.4, 1.0, 5.0)
        o1, _ = ms.predict("predict_logistic", pairs, None, 3.4, 1.0, 5.0)
        assert np.array_equal(o1, o0)
