"""The tensor-core top-N sweep at k where the per-user threshold's covariance ([ka][ka] floats,
ka = k + 1 with a bias column) no longer fits one CTA's shared memory (ka > 240 with 227 KB per
block), against the exact path."""
import numpy as np
import pytest

from mfrec_b200 import synth

pytestmark = pytest.mark.gpu

RTOL = 1e-5


def _rated_csr(nu, ni, per_user, seed):
    rng = np.random.default_rng(seed)
    lens = rng.integers(0, per_user * 2, nu)
    indptr = np.zeros(nu + 1, np.int64)
    indptr[1:] = np.cumsum(lens)
    rated = np.concatenate([np.sort(rng.choice(ni, n, replace=False)) for n in lens]).astype(np.int32)
    return indptr, rated


# ka = 240 (the last with the covariance in shared memory), 241, 251 and 256 (through L2)
@pytest.mark.parametrize("k,predictor", [(240, "predict_dot"), (241, "predict_dot"),
                                         (250, "predict_rating_with_bias"), (256, "predict_dot")])
def test_sweep_large_k_equals_exact_path(k, predictor):
    from mfrec_b200 import _native
    _native.default_context()
    nu, ni, N = 1500, 4000, 25
    u, v = synth.init_factors(nu, ni, k, seed=k)
    rng = np.random.default_rng(k)
    ib, ub = rng.normal(0, 0.2, ni), rng.normal(0, 0.2, nu)
    indptr, rated = _rated_csr(nu, ni, 30, seed=1)
    items, scores, counts, stats = _native.topn_sweep(predictor, u, v, None, ni, indptr, rated, N, 3.4, ib, ub)
    assert stats[3] == 2.0 * nu * ni * k           # the tensor-core path ran (not forwarded)
    assert stats[0] < 0.05 * nu, "too many users fell back to the exact path: %r" % (stats,)
    users = np.arange(nu, dtype=np.int32)
    wi, ws, wc = _native.topn(predictor, u, v, users, ni, indptr, rated, N, 3.4, ib, ub)
    for row in range(nu):
        m = int(wc[row])
        assert counts[row] == m
        np.testing.assert_allclose(scores[row][:m], ws[row][:m], rtol=RTOL, atol=RTOL)
        for j in range(m):
            if items[row][j] != wi[row][j]:
                near = [wi[row][i] for i in range(m) if abs(ws[row][i] - ws[row][j]) <= 3e-5 * max(1.0, abs(ws[row][j]))]
                assert items[row][j] in near or j >= m - 2, (row, j)
        assert (items[row][m:] == -1).all()
