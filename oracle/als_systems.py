"""The normal equations of one ALS-WRMF half-pass, in float64 NumPy -- TEST INFRASTRUCTURE ONLY.

``als_pass`` of ``mfrec_oracle.c`` (als_implicit.pyx:257-306) restated with BLAS, so that a test can
afford to build every row's system at many k and check the device's solution of it directly:

* ``row`` = ``[0, count_0, count_1, ...]`` holds counts, not offsets (``start += row[j]``), and only
  rows ``0 .. len(row) - 2`` are solved;
* ``HH = sum x x^T`` over ALL rows of the fixed side;
* row j: ``M = HH + c_pos * sum x x^T + reg * I`` and ``b = (1 + c_pos) * sum x`` over the listed
  neighbours, a neighbour listed twice counted twice.

Factors keep the reference's layout: feature-major ``[k, n]`` float64.

``als_layout`` restates the device's choice of row solver (``als_layout`` in
``mfrec_b200/csrc/als.cu``), so that tests can tell which kernel configuration a k runs.
"""
import numpy as np

EPS = 2.0 ** -53


def systems(X_fixed, row, col, c_pos, reg):
    """Yields ``(j, deg, M, b)`` for every active row j of the solved side, in row order.
    ``X_fixed`` is the fixed side's factors ``[k, n_fixed]``."""
    for j, deg, M, b, _b_abs in _systems(X_fixed, row, col, c_pos, reg):
        yield j, deg, M, b


def _systems(X_fixed, row, col, c_pos, reg):
    """``systems`` plus ``b_abs = (1 + c_pos) * sum |x|``, the scale of b's rounding error."""
    X = np.ascontiguousarray(np.asarray(X_fixed, dtype=np.float64).T)   # [n_fixed, k]
    k = X.shape[1]
    row = np.asarray(row, dtype=np.int64)
    col = np.asarray(col, dtype=np.int64)
    HH = X.T @ X
    start = 0
    for j in range(row.shape[0] - 1):
        start += int(row[j])
        deg = int(row[j + 1])
        XS = X[col[start:start + deg]]
        M = HH + c_pos * (XS.T @ XS)
        M[np.diag_indices(k)] += reg
        b = (1.0 + c_pos) * XS.sum(axis=0)
        yield j, deg, M, b, (1.0 + c_pos) * np.abs(XS).sum(axis=0)


def solve_half_pass(X_fixed, Y, row, col, c_pos, reg):
    """The half-pass's result: ``Y`` ``[k, n_rows]`` with every active row replaced by
    ``np.linalg.solve(M, b)``; the other rows are copied."""
    out = np.array(Y, dtype=np.float64, copy=True)
    for j, _deg, M, b in systems(X_fixed, row, col, c_pos, reg):
        out[:, j] = np.linalg.solve(M, b)
    return out


def als_wrmf(nbr_epochs, u, v, users_row, users_col, items_row, items_col, c_pos=1, reg=0.015):
    """``oracle.cpu.als_wrmf`` (u = item factors ``[k, ni]``, v = user factors ``[k, nu]``), returning
    new arrays: per epoch the user pass on u, then the item pass on the new v."""
    for _ in range(nbr_epochs):
        v = solve_half_pass(u, v, users_row, users_col, c_pos, reg)
        u = solve_half_pass(v, u, items_row, items_col, c_pos, reg)
    return u, v


def implicit_problem(k, nu, ni, nnz, seed, degrees=(), hot=0, duplicate=False):
    """A test problem in the reference's arrays: ``dict(u0 [k, ni], v0 [k, nu], ur, uc, ir, ic, nu, ni)``,
    random factors ``normal(0, 0.1)``, popularity-skewed implicit feedback.

    * The last user and the last item are inactive (outside ``ur`` / ``ir``) and have no neighbours;
      item ``ni - 2`` is active without neighbours.
    * Users ``nu - 1 - len(degrees) .. nu - 2`` have exactly ``degrees`` distinct items each.
    * ``hot`` other users also rate item 0.
    * ``duplicate``: the first user with two or more items lists its first item once more at the
      end, and likewise the first such item its first user.
    """
    rng = np.random.default_rng(seed)
    n_rand = nu - 1 - len(degrees)
    assert n_rand >= 1 and max(degrees, default=0) <= ni - 2
    pop = 1.0 / (np.arange(ni - 2) + 5.0)
    pop /= pop.sum()
    lists = [set() for _ in range(nu)]
    for u, i in zip(rng.integers(0, n_rand, nnz), rng.choice(ni - 2, nnz, p=pop)):
        lists[int(u)].add(int(i))
    for u in rng.choice(n_rand, hot, replace=False):
        lists[int(u)].add(0)
    for t, d in enumerate(degrees):
        lists[n_rand + t] = set(int(i) for i in rng.choice(ni - 2, d, replace=False))
    users = [sorted(s) for s in lists]
    items = [[] for _ in range(ni)]
    for u, s in enumerate(users):
        for i in s:
            items[i].append(u)
    if duplicate:
        for lst in (users, items):
            first = next(x for x in lst if len(x) >= 2)
            first.append(first[0])

    def arrays(lst):
        row = np.array([0] + [len(x) for x in lst[:-1]], dtype=np.int32)   # the last row stays inactive
        col = np.array([c for x in lst[:-1] for c in x], dtype=np.int32)
        return row, col

    ur, uc = arrays(users)
    ir, ic = arrays(items)
    return dict(u0=rng.normal(0, 0.1, (k, ni)), v0=rng.normal(0, 0.1, (k, nu)), ur=ur, uc=uc, ir=ir, ic=ic,
                nu=nu, ni=ni)


def eta_bound(k, deg, n_fixed):
    """The backward-error bound of a row solve: 8 (k + deg + n_fixed) eps.  It covers the Cholesky
    error and a different summation order of M and b (HH sums n_fixed terms, the neighbour Gram deg,
    the solve k)."""
    return 8.0 * (k + deg + n_fixed) * EPS


def backward_error(M, y, b, b_abs):
    """``||M y - b||_inf / (||M||_inf ||y||_inf + ||b_abs||_inf)``, 0 where both terms vanish.

    ``b_abs = (1 + c_pos) * sum |x|`` stands where the textbook normwise error has ``||b||_inf``: b's
    entries are sums of neighbour features that can cancel, and the rounding error of a sum scales
    with the magnitudes of its terms, not with the result.  Measured on a B200 with ``||b||_inf``: at
    k = 1, a row whose 11 features sum to 2.3e-4 from magnitudes summing to 0.93 gave 3.0e-14, and
    other orders of the same sum reach 1.5e-13 of that row's bound 1.9e-13."""
    den = np.abs(M).sum(axis=1).max() * np.abs(y).max() + np.abs(b_abs).max()
    return np.abs(M @ y - b).max() / den if den > 0 else 0.0


def check_half_pass(X_fixed, Y_before, Y_after, row, col, c_pos, reg, nbr_rows, cond_max=1e8):
    """Checks a half-pass's result ``Y_after`` (``[k, nbr_rows]``) against every row's system built
    from ``X_fixed`` (``[k, n_fixed]``), and returns per-row diagnostics
    ``{"row", "deg", "eta", "bound", "cond", "fwd"}`` (arrays over the active rows; ``fwd`` is the
    distance to ``np.linalg.solve`` in units of the forward error allowed below, NaN where not checked).

    Asserts, with a message naming the row:
      * every value of ``Y_after`` is finite;
      * rows outside ``0 .. len(row) - 2`` are bit-identical to ``Y_before``;
      * a row without neighbours is exactly zero;
      * the backward error of every solved row (``backward_error``, float64, from this module's M and
        b) is at most ``eta_bound``;
      * where ``cond_2(M) <= cond_max``, ``||y - y_ref||_inf <= bound * cond * (||y_ref||_inf +
        ||b_abs||_inf / ||M||_inf)`` with ``y_ref = np.linalg.solve(M, b)``: the forward error a
        backward error of ``bound`` allows (a failure lists the features that are off).
    """
    X_fixed = np.asarray(X_fixed, dtype=np.float64)
    Y_before = np.asarray(Y_before, dtype=np.float64)
    Y_after = np.asarray(Y_after, dtype=np.float64)
    k, n_fixed = X_fixed.shape
    assert Y_before.shape == (k, nbr_rows) and Y_after.shape == (k, nbr_rows), (Y_before.shape, Y_after.shape)
    bad = np.argwhere(~np.isfinite(Y_after))
    assert bad.shape[0] == 0, "non-finite values at (feature, row) %s" % bad[:8].tolist()
    n_active = len(row) - 1
    inactive = np.nonzero((Y_after[:, n_active:] != Y_before[:, n_active:]).any(axis=0)
                          | (np.signbit(Y_after[:, n_active:]) != np.signbit(Y_before[:, n_active:])).any(axis=0))[0]
    assert inactive.shape[0] == 0, "inactive rows written: %s" % (inactive[:8] + n_active).tolist()

    rows, degs, etas, bounds, conds, fwds = [], [], [], [], [], []
    for j, deg, M, b, b_abs in _systems(X_fixed, row, col, c_pos, reg):
        y = Y_after[:, j]
        bound = eta_bound(k, deg, n_fixed)
        if deg == 0:
            assert not y.any(), "row %d has no neighbours but is not zero: max |y| = %g" % (j, np.abs(y).max())
        eta = backward_error(M, y, b, b_abs)
        assert eta <= bound, "row %d (deg %d): backward error %.3g > %.3g" % (j, deg, eta, bound)
        w = np.linalg.eigvalsh(M)
        cond = w[-1] / w[0] if w[0] > 0 else np.inf
        fwd = np.nan
        if cond <= cond_max:
            y_ref = np.linalg.solve(M, b)
            scale = bound * cond * (np.abs(y_ref).max() + np.abs(b_abs).max() / np.abs(M).sum(axis=1).max())
            err = np.abs(y - y_ref)
            fwd = err.max() / scale if scale > 0 else (0.0 if not err.any() else np.inf)
            off = np.nonzero(err > scale)[0]
            assert off.shape[0] == 0, "row %d (deg %d, cond %.3g): features %s off by %s (allowed %.3g)" % (
                j, deg, cond, off[:8].tolist(), err[off[:8]].tolist(), scale)
        rows.append(j)
        degs.append(deg)
        etas.append(eta)
        bounds.append(bound)
        conds.append(cond)
        fwds.append(fwd)
    return {"row": np.array(rows, dtype=np.int64), "deg": np.array(degs, dtype=np.int64),
            "eta": np.array(etas), "bound": np.array(bounds), "cond": np.array(conds), "fwd": np.array(fwds)}


# ---- the device's row-solver layout ------------------------------------------------------------------
# A restatement of als_layout in mfrec_b200/csrc/als.cu (lines 480-508 when this was written) and of the
# sizes it uses (als_pitch, als_cluster_pitch, als_cluster_smem): from k and the device's shared memory
# it picks C, the CTAs per row (1: als_solve_kernel, more: als_cluster_solve_kernel), and kTile, the
# neighbour rows staged per step.  Keep the two in step.
K_TILE_MIN, K_TILE_MAX, CLUSTER_MAX, K_MAX = 8, 32, 8, 256


def _pitch(k):
    return (k + 7) // 8 * 8


def _cluster_pitch(k):
    return (k + 63) // 64 * 64


def _one_cta_smem(k, ktile):
    return (k * k + 2 * k + ktile * _pitch(k)) * 8


def _cluster_smem(k, c, ktile):
    nr = (k + c - 1) // c
    return (nr * k + nr + 2 * (k + 1) + 2 * k + k + ktile * _cluster_pitch(k)) * 8


def als_layout(k, smem_per_sm, smem_optin, cluster_static_smem=0):
    """``(C, kTile)`` of the row solver at k, or None where the device refuses k.  ``smem_per_sm`` and
    ``smem_optin`` are the device's shared memory per SM and opt-in per block; ``cluster_static_smem``
    is the cluster kernel's static shared memory (``cudaFuncAttributes.sharedSizeBytes``)."""
    ktile = K_TILE_MAX
    while ktile > K_TILE_MIN and _one_cta_smem(k, ktile) * 4 > smem_per_sm:
        ktile //= 2
    if _one_cta_smem(k, ktile) <= smem_optin:
        return 1, ktile
    if k > K_MAX:
        return None
    budget = max(smem_optin - cluster_static_smem, 0)
    c = 2
    while c < CLUSTER_MAX and _cluster_smem(k, c, K_TILE_MIN) > budget:
        c += 1
    ktile = K_TILE_MAX
    while ktile > K_TILE_MIN and _cluster_smem(k, c, ktile) > budget:
        ktile //= 2
    if _cluster_smem(k, c, ktile) > budget:
        return None
    return c, ktile


def layout_table(smem_per_sm, smem_optin, cluster_static_smem=0, k_max=K_MAX):
    """``[(C, kTile, k_first, k_last), ...]`` over k = 1 .. k_max, in k order (one entry per run of k
    with the same layout)."""
    out = []
    for k in range(1, k_max + 1):
        lay = als_layout(k, smem_per_sm, smem_optin, cluster_static_smem)
        if lay is None:
            break
        if out and out[-1][:2] == lay:
            out[-1] = (lay[0], lay[1], out[-1][2], k)
        else:
            out.append((lay[0], lay[1], k, k))
    return out
