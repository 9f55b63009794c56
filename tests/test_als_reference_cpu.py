"""CPU tests (no GPU) of oracle/als_systems.py, the float64 reference that tests/test_als_layouts_gpu.py
checks every ALS-WRMF row-solver layout against: it agrees with the C oracle, its checker rejects
the kernel bugs that matter, and its restatement of the device's layout choice is right."""
import numpy as np
import pytest

from oracle import als_systems as A
from oracle import cpu

B200_SMEM_PER_SM, B200_SMEM_OPTIN = 228 * 1024, 227 * 1024


def _problem(k, nu, ni, nnz, seed, ktile=8):
    edges = (0, 1, ktile - 1, ktile, ktile + 1, 2 * ktile, 2 * ktile + 1)
    return A.implicit_problem(k, nu, ni, nnz, seed, degrees=edges, hot=nu // 3, duplicate=True)


def _check_structure(p):
    nu, ni = p["nu"], p["ni"]
    assert p["ur"].shape[0] == nu and p["ir"].shape[0] == ni        # one inactive trailing row each
    assert p["ur"].sum() == p["uc"].shape[0] and p["ir"].sum() == p["ic"].shape[0]
    assert p["ir"][ni - 1] == 0                                      # an active item without neighbours
    assert not (p["uc"] == ni - 1).any() and not (p["ic"] == nu - 1).any()


@pytest.mark.parametrize("c_pos,reg", [(0, 1e-6), (1, 0.015), (40, 3.0)])
@pytest.mark.parametrize("k", [1, 7, 33, 130])
def test_reference_matches_c_oracle(k, c_pos, reg):
    """Two epochs of systems() + np.linalg.solve against the C oracle's Gauss-Jordan, at 1e-9."""
    p = _problem(k, 220, 160, 3500, seed=k * 7 + c_pos)
    _check_structure(p)
    u, v = p["u0"].copy(), p["v0"].copy()
    cpu.als_wrmf(2, k, u, v, p["ur"], p["uc"], p["ir"], p["ic"], c_pos, reg)
    ru, rv = A.als_wrmf(2, p["u0"], p["v0"], p["ur"], p["uc"], p["ir"], p["ic"], c_pos, reg)
    np.testing.assert_allclose(ru, u, rtol=1e-9, atol=1e-12)
    np.testing.assert_allclose(rv, v, rtol=1e-9, atol=1e-12)
    # the inactive trailing rows keep their initial values, rows without neighbours are zero
    assert np.array_equal(ru[:, -1], p["u0"][:, -1]) and np.array_equal(rv[:, -1], p["v0"][:, -1])
    assert not ru[:, -2].any()


def test_reference_matches_c_oracle_fewer_fixed_rows_than_k():
    """k = 130 with 100 users and 60 items: both Gram matrices HH are singular, reg keeps M definite."""
    k = 130
    p = A.implicit_problem(k, 100, 60, 900, seed=5, degrees=(0, 1, 7, 8, 9), hot=30, duplicate=True)
    u, v = p["u0"].copy(), p["v0"].copy()
    cpu.als_wrmf(2, k, u, v, p["ur"], p["uc"], p["ir"], p["ic"], 1, 0.015)
    ru, rv = A.als_wrmf(2, p["u0"], p["v0"], p["ur"], p["uc"], p["ir"], p["ic"], 1, 0.015)
    np.testing.assert_allclose(ru, u, rtol=1e-9, atol=1e-12)
    np.testing.assert_allclose(rv, v, rtol=1e-9, atol=1e-12)


def test_duplicated_neighbour_counts_twice():
    """A neighbour listed twice enters M and b twice, as in the reference's loop."""
    k = 5
    rng = np.random.default_rng(0)
    X = rng.normal(0, 0.1, (k, 4))
    row, col = np.array([0, 3], np.int32), np.array([2, 0, 2], np.int32)
    (_, deg, M, b), = list(A.systems(X, row, col, 40, 0.5))
    x0, x2 = X[:, 0], X[:, 2]
    assert deg == 3
    np.testing.assert_allclose(M, X @ X.T + 40 * (2 * np.outer(x2, x2) + np.outer(x0, x0)) + 0.5 * np.eye(k),
                               rtol=1e-14, atol=1e-16)
    np.testing.assert_allclose(b, 41 * (2 * x2 + x0), rtol=1e-14, atol=1e-16)


# ---- the checker against plausible kernel bugs ----------------------------------------------------------

def _half_pass(k, ktile, c_pos=1, reg=0.015):
    p = _problem(k, 260, 180, 4000, seed=k, ktile=ktile)
    X, Y0, row, col = p["u0"], p["v0"], p["ur"], p["uc"]
    return X, Y0, A.solve_half_pass(X, Y0, row, col, c_pos, reg), row, col, p["nu"]


def _row_of_degree(row, d):
    return int(np.nonzero(row[1:] == d)[0][0])


def _without(row, col, j, which):
    """The structure with row j's first (which = 0) or last (which = -1) neighbour left out."""
    starts = np.r_[0, np.cumsum(row[1:])]
    t = starts[j] + (0 if which == 0 else row[j + 1] - 1)
    row2 = row.copy()
    row2[j + 1] -= 1
    return row2, np.delete(col, t)


def _system(X, row, col, j, c_pos, reg):
    return next((M, b) for jj, _d, M, b in A.systems(X, row, col, c_pos, reg) if jj == j)


@pytest.mark.parametrize("k", [33, 72, 220])
def test_checker_rejects_kernel_bugs(k):
    """Each mutation touches one row (or one value) of an exact solution; the checker must reject it.
    kTile is the one the B200 layout uses at this k, and the mutated row's degree is 2 kTile: a kernel
    that drops the last row of a full staging step computes exactly the 'last neighbour' mutation."""
    c_pos, reg = 1, 0.015
    ktile = A.als_layout(k, B200_SMEM_PER_SM, B200_SMEM_OPTIN)[1]
    X, Y0, Y1, row, col, n = _half_pass(k, ktile, c_pos, reg)
    diag = A.check_half_pass(X, Y0, Y1, row, col, c_pos, reg, n)   # the unmutated solution passes
    assert diag["eta"].max() <= 1e-15 and np.nanmax(diag["fwd"]) <= 1e-3
    j = _row_of_degree(row, 2 * ktile)
    M, b = _system(X, row, col, j, c_pos, reg)

    def mutated(y):
        Y = Y1.copy()
        Y[:, j] = y
        return Y

    cases = {}
    for name, which in (("drop the last neighbour", -1), ("drop the first neighbour", 0)):
        r2, c2 = _without(row, col, j, which)
        cases[name] = mutated(np.linalg.solve(*_system(X, r2, c2, j, c_pos, reg)))
    M2 = M.copy()
    M2[k - 1, k - 1] -= reg
    cases["no reg on the last diagonal entry"] = mutated(np.linalg.solve(M2, b))
    cases["c_pos instead of 1 + c_pos in b"] = mutated(np.linalg.solve(M, b * c_pos / (1.0 + c_pos)))
    y = Y1[:, j].copy()
    f, g = int(np.argmax(np.abs(y))), int(np.argmin(np.abs(y)))
    y[[f, g]] = y[[g, f]]
    cases["two features swapped"] = mutated(y)
    Y = Y1.copy()
    Y[0, n - 1] = np.nextafter(Y[0, n - 1], np.inf)
    cases["an inactive row written"] = Y
    Y = Y1.copy()
    Y[k - 1, _row_of_degree(row, 0)] = 1e-300
    cases["a row without neighbours not zero"] = Y
    Y = Y1.copy()
    Y[k // 2, j] = np.nan
    cases["a NaN"] = Y
    accepted = []
    for name, Y in cases.items():
        try:
            A.check_half_pass(X, Y0, Y, row, col, c_pos, reg, n)
            accepted.append(name)
        except AssertionError:
            pass
    assert not accepted, "the checker accepted: %s" % accepted


def test_dropped_neighbour_is_far_above_the_bound():
    """The margin the bound leaves: a row that loses one of its neighbours has a backward error
    many orders above 8 (k + deg + n) eps, at every degree class of the edges."""
    k, c_pos, reg = 72, 1, 0.015
    X, Y0, Y1, row, col, n = _half_pass(k, 16, c_pos, reg)
    for d in (1, 15, 16, 17, 32, 33):
        j = _row_of_degree(row, d)
        M, b = _system(X, row, col, j, c_pos, reg)
        y = np.linalg.solve(*_system(X, *_without(row, col, j, -1), j, c_pos, reg))
        b_abs = next(s[4] for s in A._systems(X, row, col, c_pos, reg) if s[0] == j)
        eta = A.backward_error(M, y, b, b_abs)
        assert eta > 1e3 * A.eta_bound(k, d, X.shape[1]), (d, eta)


def test_checker_accepts_another_summation_order_of_b():
    """A correct solve whose b was summed in another order passes, even where the sum cancels: here
    the 11 neighbour features sum to ~1e-9 of their magnitudes, so relative to ||b||_inf that
    order's rounding alone is many times the bound."""
    rng = np.random.default_rng(3)
    X = rng.normal(0, 0.1, (1, 200))
    X[0, 10] -= X[0, :11].sum() - 1e-10               # neighbours 0..10 sum to about 1e-10
    row, col = np.array([0, 11], np.int32), np.arange(11, dtype=np.int32)
    (_, deg, M, b, b_abs), = list(A._systems(X, row, col, 1, 0.015))
    acc = 0.0
    for t in col[::-1]:                                # the other order: last neighbour first
        acc += X[0, t]
    y = np.array([2.0 * acc / M[0, 0]])
    textbook = abs(M[0, 0] * y[0] - b[0]) / (abs(M[0, 0] * y[0]) + abs(b[0]))
    assert textbook > 10 * A.eta_bound(1, deg, 200)
    assert A.backward_error(M, y, b, b_abs) <= A.eta_bound(1, deg, 200)
    A.check_half_pass(X, np.zeros((1, 2)), np.r_[y, 0.0].reshape(1, 2), row, col, 1, 0.015, 2)


# ---- the layout restatement -----------------------------------------------------------------------------

def test_layout_table_b200():
    """als_layout at the B200's 228 KB per SM and 227 KB opt-in per block.  Two boundaries move by one
    with the cluster kernel's static shared memory (0 or 1 KB)."""
    want = {
        0: [(1, 32, 1, 69), (1, 16, 70, 76), (1, 8, 77, 165), (2, 32, 166, 198), (2, 16, 199, 217),
            (2, 8, 218, 226), (3, 32, 227, 241), (3, 16, 242, 256)],
        1024: [(1, 32, 1, 69), (1, 16, 70, 76), (1, 8, 77, 165), (2, 32, 166, 198), (2, 16, 199, 216),
               (2, 8, 217, 226), (3, 32, 227, 240), (3, 16, 241, 256)],
    }
    for static, table in want.items():
        assert A.layout_table(B200_SMEM_PER_SM, B200_SMEM_OPTIN, static) == table
    assert A.als_layout(257, B200_SMEM_PER_SM, B200_SMEM_OPTIN) is None
    # every layout fits: the one-CTA kernel in one CTA's opt-in share, four per SM where kTile > 8,
    # the cluster kernel's share on each of its CTAs
    for k in range(1, 257):
        c, t = A.als_layout(k, B200_SMEM_PER_SM, B200_SMEM_OPTIN)
        if c == 1:
            assert A._one_cta_smem(k, t) <= B200_SMEM_OPTIN
            assert t == A.K_TILE_MIN or 4 * A._one_cta_smem(k, t) <= B200_SMEM_PER_SM
        else:
            assert A._cluster_smem(k, c, t) <= B200_SMEM_OPTIN
