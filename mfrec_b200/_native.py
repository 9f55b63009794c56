"""ctypes binding of ``libmfrec_b200.so`` (the C ABI declared in ``include/mfrec_b200.h``).

There is no CPU path: if the shared library is missing, or no sm_100 device is visible when
a compute call is made, an exception is raised -- nothing silently falls back.
"""
import atexit
import ctypes as C
import os
import threading

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
# MFREC_B200_LIB: another build of the same library (kernel experiments; see tools/README.md)
LIB_PATH = os.environ.get("MFREC_B200_LIB") or os.path.join(_HERE, "libmfrec_b200.so")

OK = 0
ERR_BAD_ARG, ERR_INDEX, ERR_OOM, ERR_CUDA, ERR_UNSUPPORTED = -1, -2, -3, -4, -5

KERNEL_LINEAR, KERNEL_LOGISTIC = 0, 1
FUNK_WITHOUT_BIAS, FUNK_WITH_BIAS, FUNK_WITH_BIAS_DEV = 0, 1, 2
SCHED_STRATIFIED, SCHED_SEQUENTIAL = 0, 1
FOLD_USERS, FOLD_ITEMS = 0, 1

PREDICTORS = {
    "predict_rating": 0,
    "predict_rating_with_bias": 1,
    "predict_linear": 2,
    "predict_logistic": 3,
    "predict_linear_neg": 4,
    "predict_dot": 5,
}

# every symbol include/mfrec_b200.h declares (tests check the library exports them all)
EXPORTS = (
    "mfrec_abi_version", "mfrec_ctx_create", "mfrec_ctx_destroy", "mfrec_last_error",
    "mfrec_ctx_stream", "mfrec_ctx_sync", "mfrec_ctx_launch_count", "mfrec_train_kmf",
    "mfrec_train_funk", "mfrec_funk_loop_dev", "mfrec_funk_subloop", "mfrec_funk_predictor_subloop",
    "mfrec_train_funk_learned_bias", "mfrec_train_als_wrmf", "mfrec_predict_pairs", "mfrec_rmse_pairs", "mfrec_topn", "mfrec_topn_sweep",
    "mfrec_bias_stats", "mfrec_ratings_pack", "mfrec_ratings_destroy", "mfrec_ratings_info",
    "mfrec_ratings_quad_types", "mfrec_ratings_perm", "mfrec_ratings_order", "mfrec_ratings_offsets", "mfrec_ratings_packed",
    "mfrec_ratings_slab_items", "mfrec_model_create", "mfrec_model_read", "mfrec_model_destroy",
    "mfrec_model_device_ptrs", "mfrec_sgd_epoch", "mfrec_model_predict",
    "mfrec_ring_create", "mfrec_ring_destroy", "mfrec_ring_handle", "mfrec_ring_connect",
    "mfrec_ring_connect_local", "mfrec_ring_epochs", "mfrec_ring_epochs_one_device", "mfrec_ring_wait",
    "mfrec_ring_sync_model", "mfrec_model_topn", "mfrec_model_topn_sweep", "mfrec_ratings_copies",
    "mfrec_train_kmf_multi", "mfrec_fold_in_kmf", "mfrec_fold_in_funk", "mfrec_train_als_wrmf_multi",
    "mfrec_model_topn_sweep_multi", "mfrec_model_predict_multi",
)


class MfrecError(RuntimeError):
    """Error reported by libmfrec_b200 (CUDA failure, OOM, unsupported size)."""

    def __init__(self, code, message):
        RuntimeError.__init__(self, "libmfrec_b200 error %d: %s" % (code, message))
        self.code = code


SPLIT_AUTO, SPLIT_ON, SPLIT_OFF = 0, 1, 2
STORAGE_F32, STORAGE_F16, STORAGE_BF16 = 0, 1, 2


class Opts(C.Structure):
    _fields_ = [("schedule", C.c_int32), ("row_blocks", C.c_int32), ("workers", C.c_int32),
                ("n_slabs", C.c_int32), ("keep_order", C.c_int32), ("k_hint", C.c_int32),
                ("seed", C.c_uint64), ("split", C.c_int32), ("split_min_copy", C.c_int32),
                ("storage", C.c_int32)]


_lib = None
_lib_lock = threading.Lock()


def lib():
    """Load the shared library (once).  Raises ImportError if it has not been built."""
    global _lib
    with _lib_lock:
        if _lib is None:
            if not os.path.exists(LIB_PATH):
                raise ImportError(
                    "%s is missing: build it with `make -C mfrec_b200/csrc` "
                    "(or __graft_entry__.build()); mfrec_b200 has no CPU fallback" % LIB_PATH)
            L = C.CDLL(LIB_PATH)
            L.mfrec_last_error.restype = C.c_char_p
            L.mfrec_last_error.argtypes = [C.c_void_p]
            L.mfrec_ctx_stream.restype = C.c_void_p
            L.mfrec_ctx_stream.argtypes = [C.c_void_p]
            L.mfrec_ctx_launch_count.restype = C.c_int64
            L.mfrec_ctx_launch_count.argtypes = [C.c_void_p]
            L.mfrec_ctx_destroy.restype = None
            L.mfrec_ctx_destroy.argtypes = [C.c_void_p]
            L.mfrec_ratings_destroy.restype = None
            L.mfrec_ratings_destroy.argtypes = [C.c_void_p]
            L.mfrec_model_destroy.restype = None
            L.mfrec_model_destroy.argtypes = [C.c_void_p]
            L.mfrec_ring_destroy.restype = None
            L.mfrec_ring_destroy.argtypes = [C.c_void_p]
            _lib = L
    return _lib


def _check(rc, ctx=None):
    if rc == OK:
        return
    msg = lib().mfrec_last_error(ctx)
    msg = msg.decode("utf-8", "replace") if msg else ""
    if rc == ERR_INDEX:
        raise IndexError(msg)
    if rc == ERR_BAD_ARG:
        raise ValueError(msg)
    if rc == ERR_OOM:
        raise MemoryError(msg)
    raise MfrecError(rc, msg)


def _ptr(a):
    return None if a is None else C.c_void_p(a.ctypes.data)


def _opts(schedule=0, row_blocks=0, workers=0, n_slabs=0, keep_order=0, k_hint=0, seed=0, split=0,
          split_min_copy=0, storage=0):
    return Opts(int(schedule), int(row_blocks), int(workers), int(n_slabs), int(keep_order),
                int(k_hint), int(seed), int(split), int(split_min_copy), int(storage))


class Context(object):
    """One CUDA device + stream (``mfrec_ctx``)."""

    def __init__(self, device=-1):
        self._h = C.c_void_p()
        _check(lib().mfrec_ctx_create(C.c_int(int(device)), C.byref(self._h)))

    def close(self):
        if getattr(self, "_h", None):
            lib().mfrec_ctx_destroy(self._h)
            self._h = None

    __del__ = close

    @property
    def handle(self):
        return self._h

    @property
    def stream(self):
        """Raw ``cudaStream_t`` the context launches on (int)."""
        return lib().mfrec_ctx_stream(self._h) or 0

    def sync(self):
        _check(lib().mfrec_ctx_sync(self._h), self._h)

    @property
    def launch_count(self):
        return int(lib().mfrec_ctx_launch_count(self._h))


_default_ctx = {}
_ctx_lock = threading.Lock()


def default_context(device=-1):
    with _ctx_lock:
        if device not in _default_ctx:
            _default_ctx[device] = Context(device)
        return _default_ctx[device]


# ---------------------------------------------------------------------------------------
# one-call drop-ins
# ---------------------------------------------------------------------------------------
def train_kmf(kernel, nbr_epochs, k, lr, K_users, K_items, K_bias, u, v, ratings_index, ratings,
              items_bias, users_bias, update_users=1, update_items=1, ctx=None, **opts):
    """In-place training; returns rmse per epoch (float64[nbr_epochs])."""
    ctx = ctx or default_context()
    rm = np.zeros(max(int(nbr_epochs), 1), dtype=np.float64)
    o = _opts(**opts)
    _check(lib().mfrec_train_kmf(
        ctx.handle, C.c_int(kernel), C.c_int(nbr_epochs), C.c_int(k), C.c_double(lr),
        C.c_double(K_users), C.c_double(K_items), C.c_double(K_bias), _ptr(u), _ptr(v),
        _ptr(ratings_index), _ptr(ratings), C.c_int64(ratings.shape[0]), C.c_int32(u.shape[1]),
        C.c_int32(v.shape[1]), _ptr(items_bias), _ptr(users_bias), C.c_int(update_users),
        C.c_int(update_items), C.byref(o), _ptr(rm)), ctx.handle)
    return rm[:max(int(nbr_epochs), 0)]


def fold_in_kmf(kernel, side, nbr_epochs, k, lr, K_users, K_items, K_bias, u, v, ratings_index, ratings,
                items_bias, users_bias, rows, ctx=None):
    """Many fold-ins in one call, in place (``mfrec_fold_in_kmf``): the same result as one
    sequential-schedule ``train_kmf`` per listed row, in list order, on that row's ratings.
    ``side`` = FOLD_USERS (rows are users) or FOLD_ITEMS.  Returns rmse [n_rows, nbr_epochs]."""
    ctx = ctx or default_context()
    rows = np.ascontiguousarray(rows, dtype=np.int32).reshape(-1)
    rm = np.zeros((rows.shape[0], max(int(nbr_epochs), 0)), dtype=np.float64)
    _check(lib().mfrec_fold_in_kmf(
        ctx.handle, C.c_int(kernel), C.c_int(side), C.c_int(nbr_epochs), C.c_int(k), C.c_double(lr),
        C.c_double(K_users), C.c_double(K_items), C.c_double(K_bias), _ptr(u), _ptr(v),
        _ptr(ratings_index), _ptr(ratings), C.c_int64(ratings.shape[0]), C.c_int32(u.shape[1]),
        C.c_int32(v.shape[1]), _ptr(items_bias), _ptr(users_bias), _ptr(rows), C.c_int32(rows.shape[0]),
        _ptr(rm) if rm.size else None), ctx.handle)
    return rm


def train_kmf_multi(devices, kernel, nbr_epochs, k, lr, K_users, K_items, K_bias, u, v, ratings_index, ratings,
                    items_bias, users_bias, **opts):
    """train_kmf on several GPUs of this process (DSGD ring over peer memory); in place, returns
    rmse per epoch."""
    dev = np.ascontiguousarray(devices, dtype=np.int32)
    rm = np.zeros(max(int(nbr_epochs), 1), dtype=np.float64)
    o = _opts(**opts)
    _check(lib().mfrec_train_kmf_multi(
        _ptr(dev), C.c_int(dev.shape[0]), C.c_int(kernel), C.c_int(nbr_epochs), C.c_int(k), C.c_double(lr),
        C.c_double(K_users), C.c_double(K_items), C.c_double(K_bias), _ptr(u), _ptr(v), _ptr(ratings_index),
        _ptr(ratings), C.c_int64(ratings.shape[0]), C.c_int32(u.shape[1]), C.c_int32(v.shape[1]),
        _ptr(items_bias), _ptr(users_bias), C.byref(o), _ptr(rm)), None)
    return rm[:max(int(nbr_epochs), 0)]


def train_funk(variant, min_epochs, max_epochs, min_improvement, k, f_init, lr, K, overall_avg, u,
               v, ratings_index, ratings, items_bias, users_bias, update_users=1, update_items=1,
               ctx=None, **opts):
    """In-place Funk-SVD training; returns (epochs_per_feature, rmse_per_feature)."""
    ctx = ctx or default_context()
    fe = np.zeros(k, dtype=np.int32)
    fr = np.zeros(k, dtype=np.float64)
    o = _opts(**opts)
    _check(lib().mfrec_train_funk(
        ctx.handle, C.c_int(variant), C.c_int(min_epochs), C.c_int(max_epochs),
        C.c_double(min_improvement), C.c_int(k), C.c_double(f_init), C.c_double(lr), C.c_double(K),
        C.c_double(overall_avg), _ptr(u), _ptr(v), _ptr(ratings_index), _ptr(ratings),
        C.c_int64(ratings.shape[0]), C.c_int32(u.shape[1]), C.c_int32(v.shape[1]),
        _ptr(items_bias), _ptr(users_bias), C.c_int(update_users), C.c_int(update_items),
        C.byref(o), _ptr(fe), _ptr(fr)), ctx.handle)
    return fe, fr


def fold_in_funk(side, min_epochs, min_improvement, k, f_init, lr, K, overall_avg, u, v, ratings_index,
                 ratings, items_bias, users_bias, rows, ctx=None):
    """Many Funk-SVD fold-ins in one call, in place (``mfrec_fold_in_funk``): the same result as one
    sequential-schedule ``train_funk(FUNK_WITH_BIAS_DEV, ...)`` per listed row, in list order, on that
    row's ratings.  ``side`` = FOLD_USERS (rows are users) or FOLD_ITEMS.  Returns (feature_epochs
    int32 [n_rows, k], feature_rmse [n_rows, k])."""
    ctx = ctx or default_context()
    rows = np.ascontiguousarray(rows, dtype=np.int32).reshape(-1)
    fe = np.zeros((rows.shape[0], k), dtype=np.int32)
    fr = np.zeros((rows.shape[0], k), dtype=np.float64)
    _check(lib().mfrec_fold_in_funk(
        ctx.handle, C.c_int(side), C.c_int(min_epochs), C.c_double(min_improvement), C.c_int(k),
        C.c_double(f_init), C.c_double(lr), C.c_double(K), C.c_double(overall_avg), _ptr(u), _ptr(v),
        _ptr(ratings_index), _ptr(ratings), C.c_int64(ratings.shape[0]), C.c_int32(u.shape[1]),
        C.c_int32(v.shape[1]), _ptr(items_bias), _ptr(users_bias), _ptr(rows), C.c_int32(rows.shape[0]),
        _ptr(fe) if fe.size else None, _ptr(fr) if fr.size else None), ctx.handle)
    return fe, fr


def funk_loop_dev(min_epochs, max_epochs, min_improvement, k, f_init, lr, K, u, v, ratings_index,
                  ratings, batch=0, rmse_hist=None, ctx=None):
    """estimator_loop (max_epochs >= 0, rmse_hist written) / estimator_loop2 (max_epochs < 0):
    gd_estimator.pyx:210-303 / :308-395, reference order.  Returns (epochs, rmse) per feature."""
    ctx = ctx or default_context()
    fe = np.zeros(k, dtype=np.int32)
    fr = np.zeros(k, dtype=np.float64)
    _check(lib().mfrec_funk_loop_dev(
        ctx.handle, C.c_int(min_epochs), C.c_int(max_epochs), C.c_double(min_improvement), C.c_int(k),
        C.c_double(f_init), C.c_double(lr), C.c_double(K), _ptr(u), _ptr(v), _ptr(ratings_index),
        _ptr(ratings), C.c_int64(ratings.shape[0]), C.c_int32(u.shape[1]), C.c_int32(v.shape[1]),
        C.c_int(batch), _ptr(rmse_hist) if rmse_hist is not None else None, _ptr(fe), _ptr(fr)), ctx.handle)
    return fe, fr


def funk_subloop(f, k, f_init, lr, K, u, v, ratings_index, ratings, rating_cache, ctx=None):
    """estimator_subloop (gd_estimator.pyx:903-962): one pass of feature f, returns its rmse."""
    ctx = ctx or default_context()
    out = C.c_double(0.0)
    _check(lib().mfrec_funk_subloop(
        ctx.handle, C.c_int(f), C.c_int(k), C.c_double(f_init), C.c_double(lr), C.c_double(K), _ptr(u),
        _ptr(v), _ptr(ratings_index), _ptr(ratings), C.c_int64(ratings.shape[0]), C.c_int32(u.shape[1]),
        C.c_int32(v.shape[1]), _ptr(rating_cache), C.byref(out)), ctx.handle)
    return float(out.value)


def funk_predictor_subloop(f, k, f_init, u, v, ratings_index, rating_cache, ctx=None):
    """predictor_subloop (gd_estimator.pyx:967-995): cache refresh of feature f, in place."""
    ctx = ctx or default_context()
    _check(lib().mfrec_funk_predictor_subloop(
        ctx.handle, C.c_int(f), C.c_int(k), C.c_double(f_init), _ptr(u), _ptr(v), _ptr(ratings_index),
        C.c_int64(ratings_index.shape[0]), C.c_int32(u.shape[1]), C.c_int32(v.shape[1]),
        _ptr(rating_cache)), ctx.handle)


def train_funk_learned_bias(min_epochs, min_improvement, k, f_init, lr, lr_users, lr_items, K_feature,
                            K_bias, overall_avg, u, v, ratings_index, ratings, items_bias, users_bias,
                            ctx=None):
    """estimator_loop_with_learned_bias (gd_estimator.pyx:401-483), reference order, in place."""
    ctx = ctx or default_context()
    fe = np.zeros(k, dtype=np.int32)
    fr = np.zeros(k, dtype=np.float64)
    _check(lib().mfrec_train_funk_learned_bias(
        ctx.handle, C.c_int(min_epochs), C.c_double(min_improvement), C.c_int(k), C.c_double(f_init),
        C.c_double(lr), C.c_double(lr_users), C.c_double(lr_items), C.c_double(K_feature),
        C.c_double(K_bias), C.c_double(overall_avg), _ptr(u), _ptr(v), _ptr(ratings_index), _ptr(ratings),
        C.c_int64(ratings.shape[0]), C.c_int32(u.shape[1]), C.c_int32(v.shape[1]), _ptr(items_bias),
        _ptr(users_bias), _ptr(fe), _ptr(fr)), ctx.handle)
    return fe, fr


def train_als_wrmf(nbr_epochs, k, u, v, users_row, users_col, items_row, items_col, nbr_users,
                   nbr_items, c_pos=1, reg=0.015, ctx=None):
    """In-place ALS-WRMF (als_implicit.pyx:208-352) on u [k, ni], v [k, nu]."""
    ctx = ctx or default_context()
    _check(lib().mfrec_train_als_wrmf(
        ctx.handle, C.c_int(nbr_epochs), C.c_int(k), _ptr(u), _ptr(v), _ptr(users_row),
        C.c_int64(users_row.shape[0]), _ptr(users_col), _ptr(items_row),
        C.c_int64(items_row.shape[0]), _ptr(items_col), C.c_int32(nbr_users), C.c_int32(nbr_items),
        C.c_int(int(c_pos)), C.c_double(float(reg))), ctx.handle)


def train_als_wrmf_multi(devices, nbr_epochs, k, u, v, users_row, users_col, items_row, items_col, nbr_users,
                         nbr_items, c_pos=1, reg=0.015):
    """train_als_wrmf over several shards, one per entry of ``devices`` (ids may repeat); in place,
    bit-identical to train_als_wrmf on ``devices[0]``."""
    dev = np.ascontiguousarray(devices, dtype=np.int32).reshape(-1)
    _check(lib().mfrec_train_als_wrmf_multi(
        _ptr(dev) if dev.size else None, C.c_int(dev.shape[0]), C.c_int(nbr_epochs), C.c_int(k), _ptr(u), _ptr(v),
        _ptr(users_row), C.c_int64(users_row.shape[0]), _ptr(users_col), _ptr(items_row),
        C.c_int64(items_row.shape[0]), _ptr(items_col), C.c_int32(nbr_users), C.c_int32(nbr_items),
        C.c_int(int(c_pos)), C.c_double(float(reg))), None)


def _as(a, dtype):
    return None if a is None else np.ascontiguousarray(a, dtype=dtype)


def predict_pairs(predictor, u, v, pairs, mu=0.0, items_bias=None, users_bias=None,
                  min_rating=1.0, max_rating=5.0, ctx=None):
    ctx = ctx or default_context()
    u, v = _as(u, np.float64), _as(v, np.float64)
    pairs = _as(pairs, np.int32).reshape(-1, 2)
    ib, ub = _as(items_bias, np.float64), _as(users_bias, np.float64)
    out = np.zeros(pairs.shape[0], dtype=np.float64)
    _check(lib().mfrec_predict_pairs(
        ctx.handle, C.c_int(PREDICTORS[predictor]), C.c_int(u.shape[0]), _ptr(u), _ptr(v),
        C.c_int32(u.shape[1]), C.c_int32(v.shape[1]), _ptr(pairs), C.c_int64(pairs.shape[0]),
        C.c_double(mu), _ptr(ib), _ptr(ub), C.c_double(min_rating), C.c_double(max_rating),
        _ptr(out)), ctx.handle)
    return out


def rmse_pairs(predictor, u, v, pairs, real, mu=0.0, items_bias=None, users_bias=None,
               min_rating=1.0, max_rating=5.0, ctx=None):
    """Returns (stats[4] = rmse, mae, var|e|, n_valid; errors[n])."""
    ctx = ctx or default_context()
    u, v = _as(u, np.float64), _as(v, np.float64)
    pairs = _as(pairs, np.int32).reshape(-1, 2)
    real = _as(real, np.float64)
    ib, ub = _as(items_bias, np.float64), _as(users_bias, np.float64)
    errs = np.zeros(pairs.shape[0], dtype=np.float64)
    stats = np.zeros(4, dtype=np.float64)
    _check(lib().mfrec_rmse_pairs(
        ctx.handle, C.c_int(PREDICTORS[predictor]), C.c_int(u.shape[0]), _ptr(u), _ptr(v),
        C.c_int32(u.shape[1]), C.c_int32(v.shape[1]), _ptr(pairs), _ptr(real),
        C.c_int64(pairs.shape[0]), C.c_double(mu), _ptr(ib), _ptr(ub), C.c_double(min_rating),
        C.c_double(max_rating), _ptr(errs), _ptr(stats)), ctx.handle)
    return stats, errs


def topn(predictor, u, v, users, n_candidates, rated_indptr, rated_items, N, mu=0.0,
         items_bias=None, users_bias=None, min_rating=1.0, max_rating=5.0, ctx=None):
    """Returns (items int32[n_users, N] (-1 padded), scores float64[n_users, N], counts)."""
    ctx = ctx or default_context()
    u, v = _as(u, np.float64), _as(v, np.float64)
    users = _as(users, np.int32).reshape(-1)
    indptr = _as(rated_indptr, np.int64)
    rated = _as(rated_items, np.int32)
    ib, ub = _as(items_bias, np.float64), _as(users_bias, np.float64)
    items = np.full((users.shape[0], N), -1, dtype=np.int32)
    scores = np.zeros((users.shape[0], N), dtype=np.float64)
    counts = np.zeros(users.shape[0], dtype=np.int32)
    _check(lib().mfrec_topn(
        ctx.handle, C.c_int(PREDICTORS[predictor]), C.c_int(u.shape[0]), _ptr(u), _ptr(v),
        C.c_int32(u.shape[1]), C.c_int32(v.shape[1]), _ptr(users), C.c_int32(users.shape[0]),
        C.c_int32(n_candidates), _ptr(indptr), _ptr(rated), C.c_double(mu), _ptr(ib), _ptr(ub),
        C.c_double(min_rating), C.c_double(max_rating), C.c_int32(N), _ptr(items), _ptr(scores),
        _ptr(counts)), ctx.handle)
    return items, scores, counts


def topn_sweep(predictor, u, v, users, n_candidates, rated_indptr, rated_items, N, mu=0.0,
               items_bias=None, users_bias=None, min_rating=1.0, max_rating=5.0, ctx=None, out=None):
    """Top-N for many users on the tensor cores (``users`` = None: all users).  Same results as
    ``topn``; returns (items, scores, counts, stats[8]).  ``out`` = preallocated (items int32
    [n, N], scores float64 [n, N], counts int32 [n]) arrays, e.g. in pinned memory."""
    ctx = ctx or default_context()
    u, v = _as(u, np.float64), _as(v, np.float64)
    n_users = v.shape[1] if users is None else None
    if users is not None:
        users = _as(users, np.int32).reshape(-1)
        n_users = users.shape[0]
    indptr = _as(rated_indptr, np.int64)
    rated = _as(rated_items, np.int32)
    ib, ub = _as(items_bias, np.float64), _as(users_bias, np.float64)
    if out is None:
        items = np.full((n_users, N), -1, dtype=np.int32)
        scores = np.zeros((n_users, N), dtype=np.float64)
        counts = np.zeros(n_users, dtype=np.int32)
    else:
        items, scores, counts = out
        assert items.shape == (n_users, N) and items.dtype == np.int32 and items.flags.c_contiguous
        assert scores.shape == (n_users, N) and scores.dtype == np.float64 and scores.flags.c_contiguous
        assert counts.shape == (n_users,) and counts.dtype == np.int32
    stats = np.zeros(8, dtype=np.float64)
    _check(lib().mfrec_topn_sweep(
        ctx.handle, C.c_int(PREDICTORS[predictor]), C.c_int(u.shape[0]), _ptr(u), _ptr(v),
        C.c_int32(u.shape[1]), C.c_int32(v.shape[1]), _ptr(users), C.c_int32(n_users),
        C.c_int32(n_candidates), _ptr(indptr), _ptr(rated), C.c_double(mu), _ptr(ib), _ptr(ub),
        C.c_double(min_rating), C.c_double(max_rating), C.c_int32(N), _ptr(items), _ptr(scores),
        _ptr(counts), _ptr(stats)), ctx.handle)
    return items, scores, counts, stats


def bias_stats(ratings_index, ratings, ni, nu, K2=0.01, K3=0.01, ctx=None):
    ctx = ctx or default_context()
    idx = _as(ratings_index, np.int32).reshape(-1, 2)
    r = _as(ratings, np.float64)
    ib = np.zeros(ni, dtype=np.float64)
    ub = np.zeros(nu, dtype=np.float64)
    mu = C.c_double(0.0)
    _check(lib().mfrec_bias_stats(
        ctx.handle, _ptr(idx), _ptr(r), C.c_int64(r.shape[0]), C.c_int32(ni), C.c_int32(nu),
        C.c_double(K2), C.c_double(K3), C.byref(mu), _ptr(ib), _ptr(ub)), ctx.handle)
    return float(mu.value), ib, ub


# ---------------------------------------------------------------------------------------
# resident objects
# ---------------------------------------------------------------------------------------
class Ratings(object):
    """Ratings packed into HBM in the stratified block layout (``mfrec_ratings``)."""

    def __init__(self, ratings_index, ratings, ni, nu, ctx=None, item_degree=None,
                 device_ptrs=None, nnz=None, ratings_are_f32=False, **opts):
        """Host arrays (int32 [nnz,2], float64/float32 [nnz]) or, with ``device_ptrs=(idx_ptr,
        r_ptr)`` and ``nnz``, raw device pointers."""
        self.ctx = ctx or default_context()
        self._h = C.c_void_p()
        self.ni, self.nu = int(ni), int(nu)
        o = _opts(**opts)
        deg = _as(item_degree, np.int64)
        if device_ptrs is not None:
            pidx, pr = C.c_void_p(int(device_ptrs[0])), C.c_void_p(int(device_ptrs[1]))
            n, is_dev, f32 = int(nnz), 1, int(bool(ratings_are_f32))
        else:
            idx = _as(ratings_index, np.int32).reshape(-1, 2)
            if ratings.dtype == np.float32:
                r, f32 = _as(ratings, np.float32), 1
            else:
                r, f32 = _as(ratings, np.float64), 0
            self._keep = (idx, r)
            pidx, pr, n, is_dev = _ptr(idx), _ptr(r), idx.shape[0], 0
        _check(lib().mfrec_ratings_pack(
            self.ctx.handle, pidx, pr, C.c_int(f32), C.c_int(is_dev), C.c_int64(n),
            C.c_int32(self.ni), C.c_int32(self.nu), _ptr(deg), C.byref(o), C.byref(self._h)),
            self.ctx.handle)
        self._keep = None
        info = (C.c_int64 * 8)()
        _check(lib().mfrec_ratings_info(self._h, info))
        (self.B, self.W, self.G, self.max_cb_items, self.nnz, self.launches_per_epoch,
         self.max_bucket, self.packed_len) = [int(x) for x in info]
        self.n_buckets = self.G * self.B * self.B * self.W * self.W

    def close(self):
        if getattr(self, "_h", None):
            lib().mfrec_ratings_destroy(self._h)
            self._h = None

    __del__ = close

    @property
    def handle(self):
        return self._h

    def perms(self):
        up = np.zeros(self.nu, dtype=np.int32)
        ip = np.zeros(self.ni, dtype=np.int32)
        _check(lib().mfrec_ratings_perm(self.ctx.handle, self._h, _ptr(up), _ptr(ip)), self.ctx.handle)
        return up, ip

    def order(self):
        out = np.zeros(self.packed_len, dtype=np.int64)
        _check(lib().mfrec_ratings_order(self.ctx.handle, self._h, _ptr(out)), self.ctx.handle)
        return out

    def offsets(self):
        off = np.zeros(self.n_buckets + 1, dtype=np.int64)
        cnt = np.zeros(self.n_buckets, dtype=np.int32)
        _check(lib().mfrec_ratings_offsets(self.ctx.handle, self._h, _ptr(off), _ptr(cnt)),
               self.ctx.handle)
        return off, cnt

    def packed(self):
        """(packed user ids, packed item ids, float32 ratings), each [packed_len]."""
        raw = np.zeros((self.packed_len, 3), dtype=np.int32)
        _check(lib().mfrec_ratings_packed(self.ctx.handle, self._h, _ptr(raw)), self.ctx.handle)
        return raw[:, 0].copy(), raw[:, 1].copy(), raw[:, 2].copy().view(np.float32)

    def quad_types(self):
        """{generic, chain, clean} quad counts of the layout (SGD kernel fast paths)."""
        out = (C.c_int64 * 4)()
        _check(lib().mfrec_ratings_quad_types(self._h, out))
        return dict(generic=int(out[0]), chain=int(out[1]), clean=int(out[2]), independent=int(out[3]))

    def copies(self):
        """(vbase int32 [ni + 1], item rows in HBM, items trained as more than one copy): item i is
        trained as vbase[i+1] - vbase[i] copies (hot-item splitting, include/mfrec_b200.h)."""
        vb = np.zeros(self.ni + 1, dtype=np.int32)
        cnt = (C.c_int64 * 2)()
        _check(lib().mfrec_ratings_copies(self._h, _ptr(vb), cnt))
        return vb, int(cnt[0]), int(cnt[1])

    def slab_items(self, slab):
        a, b = C.c_int32(), C.c_int32()
        _check(lib().mfrec_ratings_slab_items(self._h, C.c_int32(slab), C.byref(a), C.byref(b)))
        return a.value, b.value

    def replay_order(self, by_slab=False):
        """Input indices in one sequential order equivalent to the stratified schedule:
        slab, sub-epoch, row block, phase, worker, bucket order (sgd.cu header).  by_slab: a list
        with one such array per slab (a DSGD rank visits the slabs in its own ring order)."""
        order = self.order()
        off, cnt = self.offsets()
        B, W, G = self.B, self.W, self.G
        off = off[:-1].reshape(G, B, B, W * W)
        cnt = cnt.reshape(G, B, B, W * W)
        slabs = []
        for g in range(G):
            out = []
            for s in range(B):
                for rb in range(B):
                    cb = (rb + s) % B
                    for ph in range(W):
                        for w in range(W):   # buckets are stored worker-major: index w * W + phase
                            a, n = off[g, rb, cb, w * W + ph], cnt[g, rb, cb, w * W + ph]
                            if n:
                                out.append(order[a:a + n])
            slabs.append(np.concatenate(out) if out else np.zeros(0, dtype=np.int64))
        if by_slab:
            return slabs
        return np.concatenate(slabs) if slabs else np.zeros(0, dtype=np.int64)


class Model(object):
    """Factors + biases resident in HBM (``mfrec_model``), rows in the layout's packed order."""

    def __init__(self, k, ni, nu, u=None, v=None, items_bias=None, users_bias=None, layout=None,
                 ctx=None):
        self.ctx = ctx or (layout.ctx if layout is not None else default_context())
        self._h = C.c_void_p()
        self.k, self.ni, self.nu = int(k), int(ni), int(nu)
        u, v = _as(u, np.float64), _as(v, np.float64)
        ib, ub = _as(items_bias, np.float64), _as(users_bias, np.float64)
        _check(lib().mfrec_model_create(
            self.ctx.handle, layout.handle if layout is not None else None, C.c_int(self.k),
            C.c_int32(self.ni), C.c_int32(self.nu), _ptr(u), _ptr(v), _ptr(ib), _ptr(ub),
            C.byref(self._h)), self.ctx.handle)

    def close(self):
        if getattr(self, "_h", None):
            lib().mfrec_model_destroy(self._h)
            self._h = None

    __del__ = close

    @property
    def handle(self):
        return self._h

    def read(self):
        u = np.zeros((self.k, self.ni), dtype=np.float64)
        v = np.zeros((self.k, self.nu), dtype=np.float64)
        ib = np.zeros(self.ni, dtype=np.float64)
        ub = np.zeros(self.nu, dtype=np.float64)
        _check(lib().mfrec_model_read(self.ctx.handle, self._h, _ptr(u), _ptr(v), _ptr(ib), _ptr(ub)),
               self.ctx.handle)
        return u, v, ib, ub

    def device_ptrs(self):
        """((Q, item_bias, P, user_bias) raw device pointers, (ni, nu, kpad))."""
        ptrs = (C.c_void_p * 4)()
        dims = (C.c_int64 * 3)()
        _check(lib().mfrec_model_device_ptrs(self._h, ptrs, dims))
        return tuple(int(p or 0) for p in ptrs), tuple(int(d) for d in dims)

    def sgd_epoch(self, ratings, kernel, lr, K_users, K_items, K_bias, update_users=1,
                  update_items=1, slab=-1, sq_err_ptr=0):
        """Asynchronous: one epoch (or one slab's sub-epochs) on the context stream."""
        _check(lib().mfrec_sgd_epoch(
            self.ctx.handle, ratings.handle, self._h, C.c_int(kernel), C.c_double(lr),
            C.c_double(K_users), C.c_double(K_items), C.c_double(K_bias), C.c_int(update_users),
            C.c_int(update_items), C.c_int32(slab), C.c_void_p(int(sq_err_ptr) or None)),
            self.ctx.handle)

    def predict(self, predictor, pairs, real=None, mu=0.0, min_rating=1.0, max_rating=5.0,
                want_out=True, want_stats=False, device_ptrs=None, n=None, real_is_f32=False):
        """Host arrays, or ``device_ptrs=(pairs_ptr, real_ptr or 0, out_ptr or 0)`` with ``n``.
        Returns (out or None, raw stats [sum e^2, sum |e|, n_valid, 0] or None)."""
        stats = np.zeros(4, dtype=np.float64) if want_stats else None
        if device_ptrs is not None:
            pp, pr, po = [C.c_void_p(int(x) or None) for x in device_ptrs]
            _check(lib().mfrec_model_predict(
                self.ctx.handle, self._h, C.c_int(PREDICTORS[predictor]), pp, pr,
                C.c_int(int(real_is_f32)), C.c_int64(int(n)), C.c_int(1), C.c_double(mu),
                C.c_double(min_rating), C.c_double(max_rating), po, _ptr(stats)), self.ctx.handle)
            return None, stats
        pairs = _as(pairs, np.int32).reshape(-1, 2)
        real = _as(real, np.float64)
        out = np.zeros(pairs.shape[0], dtype=np.float64) if want_out else None
        _check(lib().mfrec_model_predict(
            self.ctx.handle, self._h, C.c_int(PREDICTORS[predictor]), _ptr(pairs), _ptr(real),
            C.c_int(0), C.c_int64(pairs.shape[0]), C.c_int(0), C.c_double(mu),
            C.c_double(min_rating), C.c_double(max_rating), _ptr(out), _ptr(stats)), self.ctx.handle)
        return out, stats


def _model_topn(self, predictor, users, n_candidates, rated_indptr, rated_items, N, mu=0.0, min_rating=1.0,
                max_rating=5.0, sweep=False, out=None):
    """Top-N on this RESIDENT model (identity layout): nothing but the user list, the rated-item
    CSR and the results cross PCIe.  sweep=True: the tensor-core path for many users.  Returns
    (items, scores, counts[, stats])."""
    if users is None:
        users = np.arange(self.nu, dtype=np.int32)
    users = _as(users, np.int32).reshape(-1)
    indptr = _as(rated_indptr, np.int64)
    rated = _as(rated_items, np.int32)
    n_users = users.shape[0]
    if out is None:
        items = np.full((n_users, N), -1, dtype=np.int32)
        scores = np.zeros((n_users, N), dtype=np.float64)
        counts = np.zeros(n_users, dtype=np.int32)
    else:
        items, scores, counts = out
    if sweep:
        stats = np.zeros(8, dtype=np.float64)
        _check(lib().mfrec_model_topn_sweep(
            self.ctx.handle, self._h, C.c_int(PREDICTORS[predictor]), _ptr(users), C.c_int32(n_users),
            C.c_int32(n_candidates), _ptr(indptr), _ptr(rated), C.c_double(mu), C.c_double(min_rating),
            C.c_double(max_rating), C.c_int32(N), _ptr(items), _ptr(scores), _ptr(counts), _ptr(stats)),
            self.ctx.handle)
        return items, scores, counts, stats
    _check(lib().mfrec_model_topn(
        self.ctx.handle, self._h, C.c_int(PREDICTORS[predictor]), _ptr(users), C.c_int32(n_users),
        C.c_int32(n_candidates), _ptr(indptr), _ptr(rated), C.c_double(mu), C.c_double(min_rating),
        C.c_double(max_rating), C.c_int32(N), _ptr(items), _ptr(scores), _ptr(counts)), self.ctx.handle)
    return items, scores, counts


Model.topn = _model_topn


_shard_ctx = {}


@atexit.register
def _close_shard_contexts():
    """Close the cached shard contexts while the module is still whole (a model that outlives them
    keeps its device context alive until it is destroyed)."""
    with _ctx_lock:
        for ctxs in _shard_ctx.values():
            for c in ctxs:
                c.close()
        _shard_ctx.clear()


def shard_contexts(devices):
    """One Context per entry of ``devices`` (a new one for every entry, also when ids repeat: a
    context runs one call at a time), kept per device tuple so that a ModelSet rebuilt for new
    factors reuses its streams and memory pools."""
    key = tuple(int(d) for d in devices)
    with _ctx_lock:
        if key not in _shard_ctx:
            _shard_ctx[key] = tuple(Context(d) for d in key)
        return _shard_ctx[key]


def _handles(objs):
    return (C.c_void_p * len(objs))(*[o.handle for o in objs])


class ModelSet(object):
    """The same factors resident on several shards, one ``Model`` per entry of ``devices``, each on its
    own Context.  Batched top-N (``topn(..., sweep=True)``) and host-array ``predict`` split their work
    over the shards (``mfrec_model_topn_sweep_multi`` / ``mfrec_model_predict_multi``) and return what
    one Model returns, bit for bit; everything else runs on the first shard."""

    def __init__(self, devices, k, ni, nu, u=None, v=None, items_bias=None, users_bias=None):
        ctxs = shard_contexts(devices)
        if not ctxs:
            raise ValueError("ModelSet needs at least one device")
        self.k, self.ni, self.nu = int(k), int(ni), int(nu)
        u, v = _as(u, np.float64), _as(v, np.float64)
        ib, ub = _as(items_bias, np.float64), _as(users_bias, np.float64)
        models, errors = [None] * len(ctxs), [None] * len(ctxs)

        def build(s):   # the uploads of the shards overlap (ctypes drops the GIL during the call)
            try:
                models[s] = Model(k, ni, nu, u, v, ib, ub, ctx=ctxs[s])
            except Exception as e:   # re-raised on the calling thread
                errors[s] = e

        threads = [threading.Thread(target=build, args=(s,)) for s in range(1, len(ctxs))]
        for t in threads:
            t.start()
        build(0)
        for t in threads:
            t.join()
        for e in errors:
            if e is not None:
                raise e
        self.models = tuple(models)
        self.devices = tuple(int(d) for d in devices)
        self.ctx = ctxs[0]

    def read(self):
        return self.models[0].read()

    def topn(self, predictor, users, n_candidates, rated_indptr, rated_items, N, mu=0.0, min_rating=1.0,
             max_rating=5.0, sweep=False, out=None):
        """``Model.topn``; with sweep=True the user list is split over the shards."""
        if not sweep:
            return self.models[0].topn(predictor, users, n_candidates, rated_indptr, rated_items, N, mu, min_rating,
                                       max_rating, sweep=False, out=out)
        users = None if users is None else _as(users, np.int32).reshape(-1)   # None: all users
        n_users = self.nu if users is None else users.shape[0]
        indptr = _as(rated_indptr, np.int64)
        rated = _as(rated_items, np.int32)
        if out is None:
            items = np.full((n_users, N), -1, dtype=np.int32)
            scores = np.zeros((n_users, N), dtype=np.float64)
            counts = np.zeros(n_users, dtype=np.int32)
        else:
            items, scores, counts = out
            assert items.shape == (n_users, N) and items.dtype == np.int32 and items.flags.c_contiguous
            assert scores.shape == (n_users, N) and scores.dtype == np.float64 and scores.flags.c_contiguous
            assert counts.shape == (n_users,) and counts.dtype == np.int32
        stats = np.zeros(8, dtype=np.float64)
        _check(lib().mfrec_model_topn_sweep_multi(
            _handles([m.ctx for m in self.models]), _handles(self.models), C.c_int(len(self.models)),
            C.c_int(PREDICTORS[predictor]), _ptr(users), C.c_int32(n_users), C.c_int32(n_candidates), _ptr(indptr),
            _ptr(rated), C.c_double(mu), C.c_double(min_rating), C.c_double(max_rating), C.c_int32(N), _ptr(items),
            _ptr(scores), _ptr(counts), _ptr(stats)), self.ctx.handle)
        return items, scores, counts, stats

    def predict(self, predictor, pairs, real=None, mu=0.0, min_rating=1.0, max_rating=5.0,
                want_out=True, want_stats=False, device_ptrs=None, n=None, real_is_f32=False):
        """``Model.predict``: host arrays are split over the shards; device pointers (which live on one
        device) go to the first shard."""
        if device_ptrs is not None:
            return self.models[0].predict(predictor, pairs, real, mu, min_rating, max_rating, want_out, want_stats,
                                          device_ptrs, n, real_is_f32)
        stats = np.zeros(4, dtype=np.float64) if want_stats else None
        pairs = _as(pairs, np.int32).reshape(-1, 2)
        real = _as(real, np.float64)
        out = np.zeros(pairs.shape[0], dtype=np.float64) if want_out else None
        _check(lib().mfrec_model_predict_multi(
            _handles([m.ctx for m in self.models]), _handles(self.models), C.c_int(len(self.models)),
            C.c_int(PREDICTORS[predictor]), _ptr(pairs), _ptr(real), C.c_int(0), C.c_int64(pairs.shape[0]),
            C.c_double(mu), C.c_double(min_rating), C.c_double(max_rating), _ptr(out), _ptr(stats)), self.ctx.handle)
        return out, stats


def copy_of_user(users, copies):
    """Which copy of a split item a user's rating trains: pack.cu's copy_of_user, restated for the
    tests (uint32 arithmetic)."""
    x = (np.asarray(users).astype(np.uint64) * np.uint64(0x9e3779b1)) & np.uint64(0xffffffff)
    x ^= x >> np.uint64(15)
    x = (x * np.uint64(0x85ebca77)) & np.uint64(0xffffffff)
    x ^= x >> np.uint64(13)
    return (x % np.asarray(copies).astype(np.uint64)).astype(np.int64)


def array_fingerprint(a):
    """Cheap identity of a numpy array's CONTENTS for cache invalidation: address, shape and a
    hash of ~4k strided samples (a full checksum of a 0.5 GB factor matrix would cost more than
    the call it guards).  In-place edits of single elements between the samples go unnoticed:
    code that pokes the arrays directly calls ``invalidate_model()``."""
    if a is None:
        return None
    flat = a.reshape(-1)
    step = max(1, flat.shape[0] // 4096)
    return (a.ctypes.data, a.shape, a.dtype.str, hash(flat[::step].tobytes()))


class PeerRing(object):
    """One rank of the DSGD ring (``mfrec_ring``): persistent launches that hand finished column
    blocks to the next rank through peer memory."""

    def __init__(self, ratings, model, rank, world, ctx=None):
        self.ctx = ctx or ratings.ctx
        self.ratings, self.model = ratings, model     # keep them alive: the ring borrows both
        self.rank, self.world = int(rank), int(world)
        self._h = C.c_void_p()
        _check(lib().mfrec_ring_create(self.ctx.handle, ratings.handle, model.handle, C.c_int(self.rank),
                                       C.c_int(self.world), C.byref(self._h)), self.ctx.handle)

    def close(self):
        if getattr(self, "_h", None):
            lib().mfrec_ring_destroy(self._h)
            self._h = None

    __del__ = close

    @property
    def handle(self):
        return self._h

    def export_handle(self):
        """64 bytes naming this rank's item-side block (a cudaIpcMemHandle_t)."""
        buf = (C.c_ubyte * 64)()
        _check(lib().mfrec_ring_handle(self._h, buf), self.ctx.handle)
        return bytes(buf)

    def connect(self, handles):
        """handles: list of ``world`` 64-byte strings, entry i exported by rank i."""
        blob = b"".join(handles)
        assert len(blob) == 64 * self.world
        _check(lib().mfrec_ring_connect(self._h, C.c_char_p(blob)), self.ctx.handle)

    def connect_local(self, next_ring):
        _check(lib().mfrec_ring_connect_local(self._h, next_ring.handle), self.ctx.handle)

    def epochs(self, kernel, lr, K_users, K_items, K_bias, n_epochs=1, sq_err_ptr=0):
        """Asynchronous; sq_err_ptr: device pointer to n_epochs doubles (or 0)."""
        _check(lib().mfrec_ring_epochs(
            self._h, C.c_int(kernel), C.c_double(lr), C.c_double(K_users), C.c_double(K_items),
            C.c_double(K_bias), C.c_int(int(n_epochs)), C.c_void_p(int(sq_err_ptr) or None)), self.ctx.handle)

    def wait(self):
        _check(lib().mfrec_ring_wait(self._h), self.ctx.handle)

    def sync_model(self):
        _check(lib().mfrec_ring_sync_model(self._h), self.ctx.handle)


def ring_epochs_one_device(rings, kernel, lr, K_users, K_items, K_bias, n_epochs=1, sq_err_ptr=0):
    """All ranks of a ring that live on ONE device, as a single cooperative launch (tests)."""
    arr = (C.c_void_p * len(rings))(*[r.handle for r in rings])
    ctx = rings[0].ctx
    _check(lib().mfrec_ring_epochs_one_device(
        arr, C.c_int(len(rings)), C.c_int(kernel), C.c_double(lr), C.c_double(K_users), C.c_double(K_items),
        C.c_double(K_bias), C.c_int(int(n_epochs)), C.c_void_p(int(sq_err_ptr) or None)), ctx.handle)
