"""ALS-WRMF split over several shards (mfrec_train_als_wrmf_multi) against the one-device call: the
factors must be EQUAL, not close.  Shards that share one device run the whole split-and-exchange path
(separate contexts, streams and copies, stores into the other shards' copies, event barriers) on a
single GPU; the last tests use every GPU of the process."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu


def _implicit_matrix(nu, ni, n, seed, hot=0):
    """Popularity-skewed implicit feedback; `hot` users also rate item 0; the last user and the
    last item stay without neighbours."""
    from scipy.sparse import lil_matrix
    rng = np.random.default_rng(seed)
    m = lil_matrix((nu, ni))
    pop = 1.0 / (np.arange(ni - 1) + 5.0)
    pop /= pop.sum()
    for u, i in zip(rng.integers(0, nu - 1, n), rng.choice(ni - 1, n, p=pop)):
        m[int(u), int(i)] = 1.0
    for u in rng.choice(nu - 1, hot, replace=False):
        m[int(u), 0] = 1.0
    return m


def _structures(m):
    """The reference's arrays, with every user and item active (the trailing empty ones too)."""
    from mfrec_b200.lib.datasets import create_bool_sparse_col, create_bool_sparse_row
    nu, ni = m.shape
    ur, uc = create_bool_sparse_row(m)
    ir, ic = create_bool_sparse_col(m)
    ur = np.r_[ur, np.zeros(nu + 1 - ur.shape[0])].astype(np.int32)
    ir = np.r_[ir, np.zeros(ni + 1 - ir.shape[0])].astype(np.int32)
    return ur, uc, ir, ic


def _device():
    import torch
    return torch.cuda.current_device()


def _one_and_multi(devices, k, nu, ni, st, epochs, seed):
    from mfrec_b200 import _native
    ur, uc, ir, ic = st
    rng = np.random.default_rng(seed)
    u0, v0 = rng.normal(0, 0.1, (k, ni)), rng.normal(0, 0.1, (k, nu))
    u1, v1 = u0.copy(), v0.copy()
    _native.train_als_wrmf(epochs, k, u0, v0, ur, uc, ir, ic, nu, ni, 1, 0.015,
                           ctx=_native.default_context(devices[0]))
    _native.train_als_wrmf_multi(devices, epochs, k, u1, v1, ur, uc, ir, ic, nu, ni, 1, 0.015)
    return (u0, v0), (u1, v1)


# 20: the reference's k; 64: the measured one-CTA case; 165 / 166: the last one-CTA k and the first
# cluster k on a 227 KB device; 203: no tile, block or CTA split divides it; 256: the top of the range
@pytest.mark.parametrize("shards", [2, 3])
@pytest.mark.parametrize("k", [20, 64, 165, 166, 203, 256])
def test_shards_on_one_device_bit_identical(k, shards):
    d = _device()
    nu, ni = 400, 300
    m = _implicit_matrix(nu, ni, 9000, seed=k + shards, hot=250)
    st = _structures(m)
    assert st[0][-1] == 0 and st[2][-1] == 0 and st[2][1] >= 250
    (u0, v0), (u1, v1) = _one_and_multi([d] * shards, k, nu, ni, st, 3, seed=k)
    assert np.isfinite(u0).all() and np.isfinite(v0).all()
    assert np.array_equal(u1, u0) and np.array_equal(v1, v0)


@pytest.mark.parametrize("k", [20, 200])
def test_more_shards_than_active_rows(k):
    """5 shards, 3 active users and 4 active items (of 10 and 8): most shards get an empty range on
    one side or both."""
    d = _device()
    nu, ni = 10, 8
    ur = np.array([0, 3, 1, 2], np.int32)                 # users 0..2
    uc = np.array([0, 2, 5, 1, 0, 7], np.int32)
    ir = np.array([0, 2, 1, 0, 3], np.int32)              # items 0..3 (item 2 without neighbours)
    ic = np.array([0, 2, 1, 4, 5, 9], np.int32)
    (u0, v0), (u1, v1) = _one_and_multi([d] * 5, k, nu, ni, (ur, uc, ir, ic), 3, seed=3)
    assert np.array_equal(u1, u0) and np.array_equal(v1, v0)


def _recommender(m, k, epochs):
    from mfrec_b200.recommendation import WRMFRecommender
    nu, ni = m.shape
    rec = WRMFRecommender(nu, ni, {'nbr_epochs': epochs, 'nbr_features': k, 'neighborhood': ni})
    rows, cols = m.nonzero()
    for u, i in zip(rows, cols):
        rec.set_item_by_id(int(u), int(i), 1.0)
    return rec


def _train_with_devices(rec, devices, **kw):
    from mfrec_b200.lib import als_implicit
    saved = list(als_implicit.options["devices"])
    als_implicit.options["devices"] = list(devices)
    try:
        rec.train(**kw)
    finally:
        als_implicit.options["devices"] = saved


def test_reference_constant_initialisation_20_epochs():
    """WRMFRecommender.train with initialize_model=True: all features start equal and round-off
    breaks the symmetry; the runs are bit-identical, so they do not drift apart."""
    d = _device()
    m = _implicit_matrix(400, 300, 9000, seed=21, hot=100)
    one, multi = _recommender(m, 20, 20), _recommender(m, 20, 20)
    _train_with_devices(one, [d])
    _train_with_devices(multi, [d, d, d])
    assert np.array_equal(multi.svd_u, one.svd_u) and np.array_equal(multi.svd_v, one.svd_v)
    assert np.array_equal(multi.svd_u.T @ multi.svd_v, one.svd_u.T @ one.svd_v)


@pytest.mark.parametrize("k", [64, 256])
def test_all_gpus_of_the_process(k):
    import torch
    n = torch.cuda.device_count()
    if n < 2:
        pytest.skip("needs at least 2 GPUs")
    m = _implicit_matrix(400, 300, 9000, seed=k, hot=250)
    rng = np.random.default_rng(k)
    u0, v0 = rng.normal(0, 0.1, (k, 300)), rng.normal(0, 0.1, (k, 400))
    one, multi = _recommender(m, k, 3), _recommender(m, k, 3)
    one.svd_u, one.svd_v = u0.copy(), v0.copy()
    multi.svd_u, multi.svd_v = u0.copy(), v0.copy()
    _train_with_devices(one, [0], initialize_model=False)
    _train_with_devices(multi, list(range(n)), initialize_model=False)
    assert np.array_equal(multi.svd_u, one.svd_u) and np.array_equal(multi.svd_v, one.svd_v)
    # the same split, each device listed twice
    twice = _recommender(m, k, 3)
    twice.svd_u, twice.svd_v = u0.copy(), v0.copy()
    _train_with_devices(twice, [x for x in range(n) for _ in range(2)][:16], initialize_model=False)
    assert np.array_equal(twice.svd_u, one.svd_u) and np.array_equal(twice.svd_v, one.svd_v)


def test_errors_change_nothing():
    import torch
    from mfrec_b200 import _native
    d = _device()
    nu, ni = 40, 30
    ur, uc, ir, ic = _structures(_implicit_matrix(nu, ni, 300, seed=3))
    rng = np.random.default_rng(2)

    def check(exc, devices, k, cols=None, code=None):
        u, v = rng.normal(0, 0.1, (k, ni)), rng.normal(0, 0.1, (k, nu))
        u0, v0 = u.copy(), v.copy()
        with pytest.raises(exc) as ei:
            _native.train_als_wrmf_multi(devices, 1, k, u, v, ur, uc if cols is None else cols, ir, ic, nu, ni)
        assert np.array_equal(u, u0) and np.array_equal(v, v0)
        if code is not None:
            assert ei.value.code == code
        return ei

    check(ValueError, [], 20)
    check(ValueError, [d, torch.cuda.device_count()], 20)
    check(ValueError, [d, -1], 20)
    ei = check(_native.MfrecError, [d, d], 257, code=_native.ERR_UNSUPPORTED)
    assert "256" in str(ei.value)
    bad = uc.copy()
    bad[len(bad) // 2] = ni + 5
    check(IndexError, [d, d], 20, cols=bad)
    check(IndexError, [d, d], 200, cols=bad)
    u, v = rng.normal(0, 0.1, (20, ni)), rng.normal(0, 0.1, (20, nu))
    u0, v0 = u.copy(), v.copy()
    _native.train_als_wrmf_multi([d, d], 0, 20, u, v, ur, uc, ir, ic, nu, ni)
    assert np.array_equal(u, u0) and np.array_equal(v, v0)
    # the library still works after the refusals
    (a0, b0), (a1, b1) = _one_and_multi([d, d], 20, nu, ni, (ur, uc, ir, ic), 1, seed=9)
    assert np.array_equal(a1, a0) and np.array_equal(b1, b0)


@pytest.mark.parametrize("k", [64, 203])
def test_repeated_calls_equal_one_call(k):
    """2 epochs then 1 epoch on the same arrays == 3 epochs in one call: nothing (streams, events,
    peer mappings, pooled scratch) carries over from one call to the next."""
    from mfrec_b200 import _native
    d = _device()
    nu, ni = 400, 300
    ur, uc, ir, ic = _structures(_implicit_matrix(nu, ni, 9000, seed=31, hot=200))
    rng = np.random.default_rng(4)
    u0, v0 = rng.normal(0, 0.1, (k, ni)), rng.normal(0, 0.1, (k, nu))
    u1, v1 = u0.copy(), v0.copy()
    _native.train_als_wrmf_multi([d, d], 3, k, u0, v0, ur, uc, ir, ic, nu, ni)
    _native.train_als_wrmf_multi([d, d], 2, k, u1, v1, ur, uc, ir, ic, nu, ni)
    _native.train_als_wrmf_multi([d, d], 1, k, u1, v1, ur, uc, ir, ic, nu, ni)
    assert np.array_equal(u1, u0) and np.array_equal(v1, v0)
