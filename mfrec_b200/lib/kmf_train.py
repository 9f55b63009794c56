"""``mfrec.lib.kmf_train`` on a B200.

Same call signature as the reference's Cython functions (mfrec/lib/kmf_train.pyx:103-121 and
:195-213): 16 required positional arguments, ``update_users=1, update_items=1, verbose=0``;
``u`` (item factors ``[k, ni]``), ``v`` (user factors ``[k, nu]``), ``items_bias`` and
``users_bias`` are updated in place; returns ``None``.  As in the reference, ``f_init``,
``learning_rate_users``, ``learning_rate_items`` and ``overall_avg`` are accepted and unused
(kmf_train.pyx:159,250 pass a literal 0.0 for the overall average).
"""
import numpy as np

from mfrec_b200 import _native
from mfrec_b200.lib._buffers import buffer_arg, check_rating_arrays, native_opts, options

last_rmse = None  # rmse per epoch of the most recent call (the reference only prints it)


def _train(kernel, nbr_epochs, dim, learning_rate, K_users, K_items, K_bias, u, v, ratings_index,
           ratings, items_bias, users_bias, update_users, update_items, verbose):
    global last_rmse
    nbr_epochs, dim = int(nbr_epochs), int(dim)
    buffer_arg(u, "u", np.float64, 2)
    buffer_arg(v, "v", np.float64, 2)
    buffer_arg(ratings_index, "ratings_index", np.int32, 2, writable=False)
    buffer_arg(ratings, "ratings", np.float64, 1, writable=False)
    buffer_arg(items_bias, "items_bias", np.float64, 1)
    buffer_arg(users_bias, "users_bias", np.float64, 1)
    check_rating_arrays(u, v, ratings_index, ratings, items_bias, users_bias)
    if dim > u.shape[0] or dim > v.shape[0] or dim < 0:
        raise ValueError("dim=%d exceeds the factor arrays (%d, %d features)" % (dim, u.shape[0], v.shape[0]))
    if dim == 0 or ratings.shape[0] == 0 or nbr_epochs <= 0:
        last_rmse = np.full(max(nbr_epochs, 0), np.nan)
        return None
    if len(options["devices"]) > 1 and update_users and update_items and options["schedule"] == "stratified":
        opts = native_opts()
        opts.pop("schedule")
        last_rmse = _native.train_kmf_multi(
            options["devices"], kernel, nbr_epochs, dim, float(learning_rate), float(K_users), float(K_items),
            float(K_bias), u[:dim], v[:dim], ratings_index, ratings, items_bias, users_bias, **opts)
        _print_rmse(kernel, verbose)
        return None
    ctx = _native.default_context(options["device"])
    opts = native_opts()
    if not (update_users and update_items):
        opts["storage"] = 0   # fold-ins keep the frozen side bit-identical: float32 rows, rows gathered
    last_rmse = _native.train_kmf(
        kernel, nbr_epochs, dim, float(learning_rate), float(K_users), float(K_items),
        float(K_bias), u[:dim], v[:dim], ratings_index, ratings, items_bias, users_bias,
        1 if update_users else 0, 1 if update_items else 0, ctx=ctx, **opts)
    _print_rmse(kernel, verbose)
    return None


def _print_rmse(kernel, verbose, rmse_per_epoch=None):
    if verbose:
        for epoch, rmse in enumerate(last_rmse if rmse_per_epoch is None else rmse_per_epoch):
            if kernel == _native.KERNEL_LOGISTIC:
                print("EPOCHS: " + str(epoch + 1))
            print("RMSE: " + str(rmse) + "\n")


def fold_in(kernel, side, nbr_epochs, dim, learning_rate, K_users, K_items, K_bias, u, v, ratings_index,
            ratings, items_bias, users_bias, rows, verbose=0):
    """Many fold-ins in one device call (not in the reference): the same result as calling
    ``train_*_kernel`` once per listed row, in list order, on the ratings naming that row, with
    ``update_users, update_items = 1, 0`` (``side`` = ``_native.FOLD_USERS``) or ``0, 1``
    (``_native.FOLD_ITEMS``), under the sequential schedule -- what ``KMFRecommender.retrain_user``
    / ``retrain_item`` do.  ``verbose`` prints what those calls would, row by row, and ``last_rmse``
    is left as the last of them leaves it.  Returns the rmse per row and epoch."""
    global last_rmse
    nbr_epochs, dim = int(nbr_epochs), int(dim)
    buffer_arg(u, "u", np.float64, 2)
    buffer_arg(v, "v", np.float64, 2)
    buffer_arg(ratings_index, "ratings_index", np.int32, 2, writable=False)
    buffer_arg(ratings, "ratings", np.float64, 1, writable=False)
    buffer_arg(items_bias, "items_bias", np.float64, 1)
    buffer_arg(users_bias, "users_bias", np.float64, 1)
    check_rating_arrays(u, v, ratings_index, ratings, items_bias, users_bias)
    if dim > u.shape[0] or dim > v.shape[0] or dim < 0:
        raise ValueError("dim=%d exceeds the factor arrays (%d, %d features)" % (dim, u.shape[0], v.shape[0]))
    rows = np.ascontiguousarray(rows, dtype=np.int32).reshape(-1)
    if rows.shape[0] == 0:
        return np.zeros((0, max(nbr_epochs, 0)))
    if dim == 0 or nbr_epochs <= 0:
        rm = np.full((rows.shape[0], max(nbr_epochs, 0)), np.nan)
    else:
        rm = _native.fold_in_kmf(kernel, side, nbr_epochs, dim, float(learning_rate), float(K_users),
                                 float(K_items), float(K_bias), u[:dim], v[:dim], ratings_index, ratings,
                                 items_bias, users_bias, rows,
                                 ctx=_native.default_context(options["device"]))
        if verbose:   # a call without ratings prints nothing
            col = 0 if side == _native.FOLD_USERS else 1
            rated = np.isin(rows, ratings_index[:ratings.shape[0], col])
            for p in np.nonzero(rated)[0]:
                _print_rmse(kernel, verbose, rm[p])
    last_rmse = rm[-1].copy()
    return rm


def train_linear_kernel(nbr_epochs, dim, f_init, learning_rate, learning_rate_users,
                        learning_rate_items, K_users, K_items, K_bias, overall_avg, u, v,
                        ratings_index, ratings, items_bias, users_bias, update_users=1,
                        update_items=1, verbose=0):
    """SGD for kernel matrix factorisation, linear kernel (kmf_train.pyx:195-277)."""
    return _train(_native.KERNEL_LINEAR, nbr_epochs, dim, learning_rate, K_users, K_items, K_bias,
                  u, v, ratings_index, ratings, items_bias, users_bias, update_users,
                  update_items, verbose)


def train_logistic_kernel(nbr_epochs, dim, f_init, learning_rate, learning_rate_users,
                          learning_rate_items, K_users, K_items, K_bias, overall_avg, u, v,
                          ratings_index, ratings, items_bias, users_bias, update_users=1,
                          update_items=1, verbose=0):
    """SGD for kernel matrix factorisation, logistic kernel (kmf_train.pyx:103-189)."""
    return _train(_native.KERNEL_LOGISTIC, nbr_epochs, dim, learning_rate, K_users, K_items,
                  K_bias, u, v, ratings_index, ratings, items_bias, users_bias, update_users,
                  update_items, verbose)
