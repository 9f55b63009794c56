"""ALS-WRMF above the single-CTA limit (k = 166..256: the cluster row solver of als.cu) against the
CPU oracle, across the switch from the one-CTA solver, end to end through WRMFRecommender, and at
the boundaries."""
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


def _run_pair(k, nu, ni, m, epochs, seed=1):
    from mfrec_b200.lib import als_implicit
    from oracle import cpu
    ur, uc, ir, ic = _structures(m)
    assert ur.shape[0] - 1 == nu and ir.shape[0] - 1 == ni
    rng = np.random.default_rng(seed)
    u0, v0 = rng.normal(0, 0.1, (k, ni)), rng.normal(0, 0.1, (k, nu))
    u1, v1 = u0.copy(), v0.copy()
    cpu.als_wrmf(epochs, k, u0, v0, ur, uc, ir, ic, 1, 0.015)
    als_implicit.als_wrmf(epochs, k, u1, v1, None, None, ur, uc, ir, ic, nu, ni, c_pos=1, k=0.015)
    return (u0, v0), (u1, v1), (ur, uc, ir, ic)


# 165: the last k of the one-CTA solver on a 227 KB device; 166: the first of the cluster solver;
# 203: no tile, block or CTA split divides it; 256: the top of the range
@pytest.mark.parametrize("k", [165, 166, 203, 256])
def test_als_large_k_matches_oracle(k):
    nu, ni = 400, 300
    m = _implicit_matrix(nu, ni, 9000, seed=k)
    (u0, v0), (u1, v1), (ur, _, ir, _) = _run_pair(k, nu, ni, m, 2)
    assert ur[-1] == 0 and ir[-1] == 0
    np.testing.assert_allclose(u1, u0, rtol=1e-8, atol=1e-11)
    np.testing.assert_allclose(v1, v0, rtol=1e-8, atol=1e-11)
    # rows without neighbours solve (HH + reg I) y = 0
    assert not u1[:, -1].any() and not v1[:, -1].any()


def test_als_large_k_hot_item_matches_oracle():
    """One item with more than 2,000 neighbours (many staging steps on every CTA of its cluster).
    One epoch: the oracle's Gauss-Jordan solve takes ~3 ms per row at this k."""
    k, nu, ni = 200, 2200, 300
    m = _implicit_matrix(nu, ni, 12000, seed=11, hot=2100)
    (u0, v0), (u1, v1), (ur, uc, ir, ic) = _run_pair(k, nu, ni, m, 1)
    assert ir[1] > 2000   # item 0
    np.testing.assert_allclose(u1, u0, rtol=1e-8, atol=1e-11)
    np.testing.assert_allclose(v1, v0, rtol=1e-8, atol=1e-11)


def test_wrmf_recommender_k256_end_to_end():
    """WRMFRecommender at k = 256 with the reference's constant initialisation: predictions after
    two epochs against the oracle (the rule and reason of test_als_gpu's end-to-end test), then
    precision / recall over the tensor-core sweep and the top-N lists."""
    from mfrec_b200.lib.datasets import create_bool_sparse_col, create_bool_sparse_row
    from mfrec_b200.recommendation import WRMFRecommender, metrics
    from oracle import cpu
    k, nu, ni = 256, 400, 300
    m = _implicit_matrix(nu, ni, 9000, seed=7)
    rec = WRMFRecommender(nu, ni, {'nbr_epochs': 2, 'nbr_features': k, 'neighborhood': ni})
    rows, cols = m.nonzero()
    for u, i in zip(rows, cols):
        rec.set_item_by_id(int(u), int(i), 1.0)
    rec.train()
    ur, uc = create_bool_sparse_row(rec.relationship_matrix)
    ir, ic = create_bool_sparse_col(rec.relationship_matrix)
    u0, v0 = np.zeros((k, ni)) + 0.1, np.zeros((k, nu)) + 0.1
    cpu.als_wrmf(2, k, u0, v0, ur, uc, ir, ic, 1, 0.015)
    np.testing.assert_allclose(rec.svd_u.T @ rec.svd_v, u0.T @ v0, rtol=1e-6, atol=1e-8)

    rng = np.random.default_rng(0)
    test_users = rng.choice(nu, 160, replace=False)
    held_out = np.c_[test_users, rng.integers(0, ni, 160), np.ones(160)]
    p, r, f = metrics.precision_recall(rec, held_out, nbr_recommendations=5)
    assert 0.0 <= p <= 1.0 and 0.0 <= r <= 1.0 and 0.0 <= f <= 1.0
    items, _scores, counts = rec.find_recommended_items_batch(test_users, 5)
    assert rec.last_topn_stats is not None
    dense = m.toarray()
    for j, user in enumerate(test_users):
        got = items[j, :counts[j]]
        assert counts[j] == 5 and not dense[user, got].any()
    for user in test_users[:8]:
        got, _ = rec.find_recommended_items(user_index=int(user), nbr_recommendations=5)
        assert len(got) == 5 and not dense[user, got].any()


def test_als_k257_still_refused():
    from mfrec_b200 import _native
    from mfrec_b200.lib import als_implicit
    k, nu, ni = 257, 40, 30
    ur, uc, ir, ic = _structures(_implicit_matrix(nu, ni, 300, seed=3))
    rng = np.random.default_rng(2)
    u, v = rng.normal(0, 0.1, (k, ni)), rng.normal(0, 0.1, (k, nu))
    u0, v0 = u.copy(), v.copy()
    with pytest.raises(_native.MfrecError) as ei:
        als_implicit.als_wrmf(1, k, u, v, None, None, ur, uc, ir, ic, nu, ni)
    assert ei.value.code == _native.ERR_UNSUPPORTED and "256" in str(ei.value)
    assert np.array_equal(u, u0) and np.array_equal(v, v0)


def test_als_large_k_bad_neighbour_id_writes_nothing():
    from mfrec_b200.lib import als_implicit
    k, nu, ni = 200, 5, 4
    rng = np.random.default_rng(4)
    u, v = rng.normal(0, 0.1, (k, ni)), rng.normal(0, 0.1, (k, nu))
    u0, v0 = u.copy(), v.copy()
    row = np.array([0, 1, 1], np.int32)
    with pytest.raises(IndexError):
        als_implicit.als_wrmf(1, k, u, v, None, None, row, np.array([0, 9], np.int32), row,
                              np.array([0, 1], np.int32), nu, ni)
    assert np.array_equal(u, u0) and np.array_equal(v, v0)


def test_als_large_k_deterministic():
    from mfrec_b200.lib import als_implicit
    k, nu, ni = 256, 400, 300
    ur, uc, ir, ic = _structures(_implicit_matrix(nu, ni, 9000, seed=5))
    rng = np.random.default_rng(6)
    u0, v0 = rng.normal(0, 0.1, (k, ni)), rng.normal(0, 0.1, (k, nu))
    out = []
    for _ in range(2):
        u, v = u0.copy(), v0.copy()
        als_implicit.als_wrmf(2, k, u, v, None, None, ur, uc, ir, ic, nu, ni, c_pos=1, k=0.015)
        out.append((u, v))
    assert np.array_equal(out[0][0], out[1][0]) and np.array_equal(out[0][1], out[1][1])
