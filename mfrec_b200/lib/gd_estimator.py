"""``mfrec.lib.gd_estimator`` on a B200: the Funk-SVD per-feature SGD loops.

Signatures follow mfrec/lib/gd_estimator.pyx: ``estimator_loop_without_bias`` (:691-704),
``estimator_loop_with_bias`` (:489-507), ``estimator_loop_with_bias_dev`` (:588-608).  ``u`` and
``v`` are trained in place, biases are read-only, ``max_epochs`` / ``learning_rate_users`` /
``learning_rate_items`` / ``nbr_users`` / ``nbr_items`` are accepted and unused exactly like the
reference; returns ``None``.

The development variants (SURVEY.md section 8(a), priority A3) -- ``estimator_loop`` (:210-303),
``estimator_loop2`` (:308-395), ``estimator_subloop`` (:903-962, returns the rmse),
``predictor_subloop`` (:967-995) with their dense ``user + item * nbr_users`` cache, and the
learned-bias hybrid ``estimator_loop_with_learned_bias`` (:401-483) -- run on the device in the
reference's own order (one thread, float64: bit-identical to the reference, toy sizes like the
reference itself).  The implicit-feedback loop (:785-898) reuses its outer loop variable and
overwrites its own accumulator; it is not reproduced and raises NotImplementedError.
"""
import numpy as np

from mfrec_b200 import _native
from mfrec_b200.lib._buffers import buffer_arg, check_rating_arrays, native_opts, options

last_feature_epochs = None
last_feature_rmse = None


def _train(variant, min_epochs, max_epochs, min_improvement, dim, f_init, learning_rate, K,
           overall_avg, u, v, ratings_index, ratings, items_bias, users_bias, update_users,
           update_items, verbose):
    global last_feature_epochs, last_feature_rmse
    dim = int(dim)
    buffer_arg(u, "u", np.float64, 2)
    buffer_arg(v, "v", np.float64, 2)
    buffer_arg(ratings_index, "ratings_index", np.int32, 2, writable=False)
    buffer_arg(ratings, "ratings", np.float64, 1, writable=False)
    if variant != _native.FUNK_WITHOUT_BIAS:
        buffer_arg(items_bias, "items_bias", np.float64, 1, writable=False)
        buffer_arg(users_bias, "users_bias", np.float64, 1, writable=False)
    check_rating_arrays(u, v, ratings_index, ratings, items_bias, users_bias)
    if dim > u.shape[0] or dim > v.shape[0] or dim < 0:
        raise ValueError("dim=%d exceeds the factor arrays (%d, %d features)" % (dim, u.shape[0], v.shape[0]))
    if dim == 0:
        return None
    ctx = _native.default_context(options["device"])
    fe, fr = _native.train_funk(
        variant, int(min_epochs), int(max_epochs), float(min_improvement), dim, float(f_init),
        float(learning_rate), float(K), float(overall_avg), u[:dim], v[:dim], ratings_index,
        ratings, items_bias, users_bias, 1 if update_users else 0, 1 if update_items else 0,
        ctx=ctx, **native_opts())
    last_feature_epochs, last_feature_rmse = fe, fr
    if verbose:
        for f in range(dim):
            print("Training the feature " + str(f))
            print("RMSE: " + str(fr[f]) + "\n")
    return None


def fold_in(side, min_epochs, min_improvement, dim, f_init, learning_rate, K, overall_avg, u, v,
            ratings_index, ratings, items_bias, users_bias, rows, verbose=0):
    """Many fold-ins in one device call (not in the reference): the same result, bit for bit, as
    calling ``estimator_loop_with_bias_dev`` once per listed row, in list order, on the ratings naming
    that row, with ``update_users, update_items = 1, 0`` (``side`` = ``_native.FOLD_USERS``) or
    ``0, 1`` (``_native.FOLD_ITEMS``) under the sequential schedule -- what
    ``GDRecommender.retrain_user`` / ``retrain_item`` do.  The batch always runs the reference's order,
    whatever ``options["schedule"]`` says.  Every listed row needs at least one rating.  ``verbose``
    prints what those calls would, row by row, and ``last_feature_epochs`` / ``last_feature_rmse`` are
    left as the last of them leaves them.  Returns (feature_epochs [n_rows, dim], feature_rmse
    [n_rows, dim])."""
    global last_feature_epochs, last_feature_rmse
    dim = int(dim)
    buffer_arg(u, "u", np.float64, 2)
    buffer_arg(v, "v", np.float64, 2)
    buffer_arg(ratings_index, "ratings_index", np.int32, 2, writable=False)
    buffer_arg(ratings, "ratings", np.float64, 1, writable=False)
    buffer_arg(items_bias, "items_bias", np.float64, 1, writable=False)
    buffer_arg(users_bias, "users_bias", np.float64, 1, writable=False)
    check_rating_arrays(u, v, ratings_index, ratings, items_bias, users_bias)
    if dim > u.shape[0] or dim > v.shape[0] or dim < 0:
        raise ValueError("dim=%d exceeds the factor arrays (%d, %d features)" % (dim, u.shape[0], v.shape[0]))
    rows = np.ascontiguousarray(rows, dtype=np.int32).reshape(-1)
    if rows.shape[0] == 0 or dim == 0:
        return np.zeros((rows.shape[0], dim), dtype=np.int32), np.zeros((rows.shape[0], dim))
    fe, fr = _native.fold_in_funk(
        side, int(min_epochs), float(min_improvement), dim, float(f_init), float(learning_rate), float(K),
        float(overall_avg), u[:dim], v[:dim], ratings_index, ratings, items_bias, users_bias, rows,
        ctx=_native.default_context(options["device"]))
    last_feature_epochs, last_feature_rmse = fe[-1].copy(), fr[-1].copy()
    if verbose:
        for p in range(rows.shape[0]):
            for f in range(dim):
                print("Training the feature " + str(f))
                print("RMSE: " + str(fr[p, f]) + "\n")
    return fe, fr


def estimator_loop_without_bias(min_epochs, max_epochs, min_improvement, dim, f_init,
                                learning_rate, K, u, v, ratings_index, ratings, nbr_users,
                                nbr_items, verbose=0):
    return _train(_native.FUNK_WITHOUT_BIAS, min_epochs, max_epochs, min_improvement, dim, f_init,
                  learning_rate, K, 1.0, u, v, ratings_index, ratings, None, None, 1, 1, verbose)


def estimator_loop_with_bias(min_epochs, max_epochs, min_improvement, dim, f_init, learning_rate,
                             learning_rate_users, learning_rate_items, K, overall_avg, u, v,
                             ratings_index, ratings, items_bias, users_bias, nbr_users, nbr_items,
                             verbose=0):
    return _train(_native.FUNK_WITH_BIAS, min_epochs, max_epochs, min_improvement, dim, f_init,
                  learning_rate, K, overall_avg, u, v, ratings_index, ratings, items_bias,
                  users_bias, 1, 1, verbose)


def estimator_loop_with_bias_dev(min_epochs, max_epochs, min_improvement, dim, f_init,
                                 learning_rate, learning_rate_users, learning_rate_items, K,
                                 overall_avg, u, v, ratings_index, ratings, items_bias, users_bias,
                                 nbr_users, nbr_items, update_users=1, update_items=1, verbose=0):
    return _train(_native.FUNK_WITH_BIAS_DEV, min_epochs, max_epochs, min_improvement, dim, f_init,
                  learning_rate, K, overall_avg, u, v, ratings_index, ratings, items_bias,
                  users_bias, update_users, update_items, verbose)


def _dev_common(dim, u, v, ratings_index, ratings, nbr_users):
    dim = int(dim)
    buffer_arg(u, "u", np.float64, 2)
    buffer_arg(v, "v", np.float64, 2)
    buffer_arg(ratings_index, "ratings_index", np.int32, 2, writable=False)
    buffer_arg(ratings, "ratings", np.float64, 1, writable=False)
    check_rating_arrays(u, v, ratings_index, ratings)
    if dim > u.shape[0] or dim > v.shape[0] or dim < 0:
        raise ValueError("dim=%d exceeds the factor arrays (%d, %d features)" % (dim, u.shape[0], v.shape[0]))
    if nbr_users is not None and int(nbr_users) != v.shape[1]:
        raise ValueError("nbr_users=%d is not the width of v (%d): the dense rating cache is indexed "
                         "user + item * nbr_users" % (int(nbr_users), v.shape[1]))
    return dim


def estimator_loop(min_epochs, max_epochs, min_improvement, dim, f_init, learning_rate, K, u, v,
                   ratings_index, ratings, batch, rmse_hist, nbr_users, nbr_features, verbose=0):
    """gd_estimator.pyx:210-303: honours max_epochs, writes rmse_hist[epoch + f*max_epochs +
    batch*max_epochs*dim]."""
    global last_feature_epochs, last_feature_rmse
    dim = _dev_common(dim, u, v, ratings_index, ratings, nbr_users)
    buffer_arg(rmse_hist, "rmse_hist", np.float64, 1)
    max_epochs, batch = int(max_epochs), int(batch)
    if max_epochs < 0 or batch < 0 or rmse_hist.shape[0] < (batch + 1) * max_epochs * dim:
        raise ValueError("rmse_hist holds %d entries, (batch + 1) * max_epochs * dim = %d are addressed"
                         % (rmse_hist.shape[0], (batch + 1) * max(max_epochs, 0) * dim))
    if dim == 0:
        return None
    fe, fr = _native.funk_loop_dev(int(min_epochs), max_epochs, float(min_improvement), dim, float(f_init),
                                   float(learning_rate), float(K), u[:dim], v[:dim], ratings_index, ratings,
                                   batch, rmse_hist, ctx=_native.default_context(options["device"]))
    last_feature_epochs, last_feature_rmse = fe, fr
    if verbose:
        for f in range(dim):
            print("Training the feature " + str(f))
            print("Nbr. epoch: " + str(fe[f]))
            print("RMSE: " + str(fr[f]) + "\n")
    return None


def estimator_loop2(min_epochs, max_epochs, min_improvement, dim, f_init, learning_rate, K, u, v,
                    ratings_index, ratings, features_bias, nbr_users, nbr_features, verbose=0):
    """gd_estimator.pyx:308-395: estimator_loop with the control of estimator_loop_without_bias;
    max_epochs and features_bias are accepted and unused like in the reference."""
    global last_feature_epochs, last_feature_rmse
    dim = _dev_common(dim, u, v, ratings_index, ratings, nbr_users)
    if dim == 0:
        return None
    fe, fr = _native.funk_loop_dev(int(min_epochs), -1, float(min_improvement), dim, float(f_init),
                                   float(learning_rate), float(K), u[:dim], v[:dim], ratings_index, ratings,
                                   0, None, ctx=_native.default_context(options["device"]))
    last_feature_epochs, last_feature_rmse = fe, fr
    if verbose:
        for f in range(dim):
            print("Training the feature " + str(f))
            print("RMSE: " + str(fr[f]) + "\n")
    return None


def _dense_cache(rating_cache, u, v, writable):
    buffer_arg(rating_cache, "rating_cache", np.float64, 1, writable=writable)
    if rating_cache.shape[0] < u.shape[1] * v.shape[1]:
        raise ValueError("rating_cache holds %d entries, nbr_users * nbr_items = %d are addressed"
                         % (rating_cache.shape[0], u.shape[1] * v.shape[1]))


def estimator_subloop(f, epochs, min_improvement, dim, f_init, learning_rate, K, u, v, ratings_index,
                      ratings, rating_cache, nbr_users, nbr_features, verbose=0):
    """gd_estimator.pyx:903-962: ONE pass of feature f (epochs / min_improvement unused like in the
    reference); returns the rmse."""
    dim = _dev_common(dim, u, v, ratings_index, ratings, nbr_users)
    _dense_cache(rating_cache, u, v, False)
    f = int(f)
    if not 0 <= f < dim:
        raise IndexError("feature %d of %d" % (f, dim))
    return _native.funk_subloop(f, dim, float(f_init), float(learning_rate), float(K), u[:dim], v[:dim],
                                ratings_index, ratings, rating_cache,
                                ctx=_native.default_context(options["device"]))


def predictor_subloop(f, epochs, dim, f_init, u, v, ratings_index, ratings, rating_cache, nbr_users,
                      nbr_features):
    """gd_estimator.pyx:967-995: refresh the dense cache for feature f, in place."""
    dim = _dev_common(dim, u, v, ratings_index, ratings, nbr_users)
    _dense_cache(rating_cache, u, v, True)
    f = int(f)
    if not 0 <= f < dim:
        raise IndexError("feature %d of %d" % (f, dim))
    _native.funk_predictor_subloop(f, dim, float(f_init), u[:dim], v[:dim], ratings_index, rating_cache,
                                   ctx=_native.default_context(options["device"]))
    return None


def estimator_loop_with_learned_bias(min_epochs, max_epochs, min_improvement, dim, f_init, learning_rate,
                                     learning_rate_users, learning_rate_items, K_feature, K_bias,
                                     overall_avg, u, v, ratings_index, ratings, items_bias, users_bias,
                                     nbr_users, nbr_items, verbose=0, learning_mode=0):
    """gd_estimator.pyx:401-483: full clamped k-dot per rating, feature f and both biases are
    learned (items_bias / users_bias are written); max_epochs / learning_mode unused like in the
    reference."""
    global last_feature_epochs, last_feature_rmse
    dim = _dev_common(dim, u, v, ratings_index, ratings, None)
    buffer_arg(items_bias, "items_bias", np.float64, 1)
    buffer_arg(users_bias, "users_bias", np.float64, 1)
    check_rating_arrays(u, v, ratings_index, ratings, items_bias, users_bias)
    if u.shape[0] != dim or v.shape[0] != dim:
        # full_estimator sums over `dim` features of the arrays it is given (:141-142)
        raise ValueError("estimator_loop_with_learned_bias needs factor arrays of exactly dim rows")
    if dim == 0:
        return None
    fe, fr = _native.train_funk_learned_bias(
        int(min_epochs), float(min_improvement), dim, float(f_init), float(learning_rate),
        float(learning_rate_users), float(learning_rate_items), float(K_feature), float(K_bias),
        float(overall_avg), u, v, ratings_index, ratings, items_bias, users_bias,
        ctx=_native.default_context(options["device"]))
    last_feature_epochs, last_feature_rmse = fe, fr
    if verbose:
        for f in range(dim):
            print("Training the feature " + str(f))
            print("RMSE: " + str(fr[f]) + "\n")
    return None


def estimator_loop_with_implicit_feedback(*_a, **_k):
    raise NotImplementedError(
        "estimator_loop_with_implicit_feedback (gd_estimator.pyx:785-898) reuses its outer loop variable "
        "(:869, :879) and overwrites feedback_sum (:873): its results are an artefact of those bugs and it "
        "is not part of the B200 hot path; see DESIGN.md")
