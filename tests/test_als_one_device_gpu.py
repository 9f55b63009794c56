"""mfrec_train_als_wrmf on the caller's context: the call borrows it (it neither destroys nor keeps
it), counts its launches there, and reports its refusals there, with u / v untouched; the context
keeps working for ALS and for other calls afterwards."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu
PREFIX = "mfrec_train_als_wrmf: "


def _problem(nu=60, ni=40, seed=0):
    """The reference's arrays ([0, counts...] and neighbour ids in row order) of a random implicit matrix."""
    m = np.random.default_rng(seed).random((nu, ni)) < 0.15
    ur, ir = np.r_[0, m.sum(1)].astype(np.int32), np.r_[0, m.sum(0)].astype(np.int32)
    uc, ic = np.nonzero(m)[1].astype(np.int32), np.nonzero(m.T)[1].astype(np.int32)
    return nu, ni, ur, uc, ir, ic


def _factors(k, nu, ni, seed):
    rng = np.random.default_rng(seed)
    return rng.normal(0, 0.1, (k, ni)), rng.normal(0, 0.1, (k, nu))


def _device():
    import torch
    return torch.cuda.current_device()


def _context():
    from mfrec_b200 import _native
    return _native.default_context(_device())


def _train(ctx, epochs, k, u, v, p, users_row=None, users_col=None):
    from mfrec_b200 import _native
    nu, ni, ur, uc, ir, ic = p
    _native.train_als_wrmf(epochs, k, u, v, ur if users_row is None else users_row, uc if users_col is None else users_col,
                           ir, ic, nu, ni, 1, 0.015, ctx=ctx)


def _predict_on(ctx, u, v):
    from mfrec_b200 import _native
    from oracle import cpu
    pairs = np.stack([np.arange(30), np.arange(30)[::-1]], axis=1).astype(np.int32)
    got = _native.predict_pairs("predict_rating", u, v, pairs, ctx=ctx)
    np.testing.assert_allclose(got, cpu.predict_pairs("predict_rating", u, v, pairs), rtol=1e-5, atol=1e-5)


@pytest.mark.parametrize("k", [20, 200])   # one CTA per row / a cluster per row
def test_the_context_keeps_working(k):
    ctx = _context()
    p = _problem(seed=k)
    u0, v0 = _factors(k, p[0], p[1], seed=1)
    u1, v1 = u0.copy(), v0.copy()
    n0 = ctx.launch_count
    _train(ctx, 3, k, u0, v0, p)
    n1 = ctx.launch_count
    assert n1 > n0 and np.isfinite(u0).all() and np.isfinite(v0).all()
    # the same context again: 2 epochs then 1 equal 3 in one call
    _train(ctx, 2, k, u1, v1, p)
    _train(ctx, 1, k, u1, v1, p)
    assert np.array_equal(u1, u0) and np.array_equal(v1, v0)
    n2 = ctx.launch_count
    assert n2 > n1
    _predict_on(ctx, u0, v0)
    assert ctx.launch_count > n2


def test_refusals_report_on_the_context_and_change_nothing():
    from mfrec_b200 import _native
    ctx = _context()
    p = _problem(seed=3)
    nu, ni, ur, uc, ir, ic = p
    bad_col = uc.copy()
    bad_col[len(bad_col) // 2] = ni + 5
    bad_row = ur.copy()
    bad_row[0] = -1   # a first count below 0 would start the first row before the column array

    def refused(exc, k, **kw):
        u, v = _factors(k, nu, ni, seed=k)
        u0, v0 = u.copy(), v.copy()
        with pytest.raises(exc) as ei:
            _train(ctx, 1, k, u, v, p, **kw)
        assert np.array_equal(u, u0) and np.array_equal(v, v0)
        msg = _native.lib().mfrec_last_error(ctx.handle).decode()
        assert msg.startswith(PREFIX) and str(ei.value).endswith(msg), (msg, str(ei.value))
        return ei.value, msg

    e, msg = refused(_native.MfrecError, 257)
    assert e.code == _native.ERR_UNSUPPORTED and "256" in msg
    for k in (20, 200):
        assert "neighbour id out of range" in refused(IndexError, k, users_col=bad_col)[1]
        assert "negative count" in refused(ValueError, k, users_row=bad_row)[1]

    # still usable: the same factors as on a context of its own, and other calls run
    k = 20
    u0, v0 = _factors(k, nu, ni, seed=7)
    u1, v1 = u0.copy(), v0.copy()
    _train(ctx, 2, k, u0, v0, p)
    own = _native.Context(_device())
    try:
        _train(own, 2, k, u1, v1, p)
    finally:
        own.close()
    assert np.array_equal(u1, u0) and np.array_equal(v1, v0)
    _predict_on(ctx, u0, v0)
