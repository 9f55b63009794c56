"""Argument checking that mirrors what Cython's typed-buffer arguments do in the reference
(``np.ndarray[np.float64_t, ndim=2, mode="c"]`` etc., kmf_train.pyx:113-118): the same
exception types and messages, raised before any work is done.  Two deliberate tightenings:
``None`` is rejected (the reference segfaults) and out-of-range indices raise IndexError
(the reference disables bounds checks and corrupts memory)."""
import os

import numpy as np

_CNAME = {np.dtype(np.float64): "float64_t", np.dtype(np.int32): "int32_t"}
_GOT = {"f": {4: "float", 8: "double", 2: "short float", 16: "long double"},
        "i": {1: "signed char", 2: "short", 4: "int", 8: "long"},
        "u": {1: "unsigned char", 2: "unsigned short", 4: "unsigned int", 8: "unsigned long"},
        "b": {1: "bool"}, "c": {8: "float complex", 16: "double complex"}}


def buffer_arg(a, name, dtype, ndim, writable=True):
    if not isinstance(a, np.ndarray):
        raise TypeError("Argument '%s' has incorrect type (expected numpy.ndarray, got %s)"
                        % (name, type(a).__name__))
    dtype = np.dtype(dtype)
    if a.dtype != dtype:
        got = _GOT.get(a.dtype.kind, {}).get(a.dtype.itemsize, str(a.dtype))
        raise ValueError("Buffer dtype mismatch, expected '%s' but got '%s'" % (_CNAME[dtype], got))
    if a.ndim != ndim:
        raise ValueError("Buffer has wrong number of dimensions (expected %d, got %d)" % (ndim, a.ndim))
    if not a.flags.c_contiguous:
        raise ValueError("ndarray is not C-contiguous")
    if writable and not a.flags.writeable:
        raise ValueError("buffer source array is read-only")
    return a


def check_rating_arrays(u, v, ratings_index, ratings, items_bias=None, users_bias=None):
    """Shape consistency the native side relies on (it takes nnz from ``ratings``, ni / nu from the
    widths of ``u`` / ``v`` and copies nnz * 8, ni * 8, nu * 8 bytes from these host pointers): a
    short index or bias array must raise here, not be read out of bounds there."""
    if ratings_index.shape[0] and ratings_index.shape[1] != 2:
        raise ValueError("ratings_index must have shape [nnz, 2]")
    if ratings_index.shape[0] < ratings.shape[0]:
        raise ValueError("ratings_index has fewer rows than ratings")
    if items_bias is not None and items_bias.shape[0] < u.shape[1]:
        raise ValueError("items_bias is shorter than the item factor array")
    if users_bias is not None and users_bias.shape[0] < v.shape[1]:
        raise ValueError("users_bias is shorter than the user factor array")


# Process-wide knobs of the CUDA implementation (not part of the reference signature).
# schedule: "stratified" (default, fp32, all SMs) | "sequential" (fp64, reference order).
options = {
    "schedule": os.environ.get("MFREC_B200_SCHEDULE", "stratified"),
    "row_blocks": int(os.environ.get("MFREC_B200_ROW_BLOCKS", "0")),
    "workers": int(os.environ.get("MFREC_B200_WORKERS", "0")),
    "seed": int(os.environ.get("MFREC_B200_SEED", "0")),
    "device": int(os.environ.get("MFREC_B200_DEVICE", "-1")),
    # several CUDA devices, e.g. [0, 1, 2, 3] (MFREC_B200_DEVICES=0,1,2,3): train_linear_kernel /
    # train_logistic_kernel calls that train both sides run as a DSGD ring over them, and als_wrmf
    # (WRMFRecommender.train) splits each ALS half-pass's rows over them (bit-identical to one device);
    # the recommenders' resident models are then kept on every listed device (ids may repeat), so that
    # find_recommended_items_batch / precision_recall split their users and test_predict_rating its pairs
    # over them, and similar_items_batch its queries (bit-identical to one device); single-user calls
    # run on the first listed device
    "devices": [int(x) for x in os.environ.get("MFREC_B200_DEVICES", "").split(",") if x.strip()],
    # how the user-factor rows are kept in HBM while training: "f32" | "f16" | "bf16"
    # (mfrec_opts.storage in include/mfrec_b200.h: arithmetic stays float32; single device, both
    # sides trained, dim > 32)
    "storage": os.environ.get("MFREC_B200_STORAGE", "f32"),
}

STORAGE = {"f32": 0, "f16": 1, "bf16": 2}


def native_opts():
    sched = {"stratified": 0, "sequential": 1}[options["schedule"]]
    if options["storage"] not in STORAGE:
        raise ValueError("options['storage'] must be one of %s" % sorted(STORAGE))
    return dict(schedule=sched, row_blocks=options["row_blocks"], workers=options["workers"],
                seed=options["seed"], storage=STORAGE[options["storage"]])
