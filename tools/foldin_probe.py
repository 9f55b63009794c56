"""Batched fold-in (KMFRecommender.add_users, one mfrec_fold_in_kmf call) against the add_user loop
(one mfrec_train_kmf call per user) at Netflix shape: 480k users x 17.7k items, k = 128, random
factors, nbr_epochs = 200, new users with 20-200 ratings each drawn by item popularity
(mfrec_b200.synth).  For both kernels and each batch size it prints the host wall time of the loop
(timed on the first SAMPLE users and scaled), of one add_users call, the kernel launches of each,
and the number of levels (linear kernel: rows that share an item run one after the other), then
all of it as one JSON line.  Every timed span ends in a device synchronise.  Environment: USERS
(default 1000,10000), SAMPLE (20), EPOCHS (200), KERNELS (logistic,linear)."""
import json
import os
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np

from mfrec_b200 import _native, synth
from mfrec_b200.recommendation import KMFRecommender

SIZES = [int(x) for x in os.environ.get("USERS", "1000,10000").split(",")]
SAMPLE = int(os.environ.get("SAMPLE", "20"))
EPOCHS = int(os.environ.get("EPOCHS", "200"))
KERNELS = ["train_%s_kernel" % x for x in os.environ.get("KERNELS", "logistic,linear").split(",")]


def gpu_info():
    try:
        return subprocess.check_output(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                                       text=True).strip().splitlines()[0]
    except (OSError, subprocess.CalledProcessError):
        return "unknown GPU"


def new_users(n, ni, seed=7):
    _wu, wi = synth.marginals(480_000, ni)
    rng = np.random.default_rng(seed)
    items = [rng.choice(ni, int(rng.integers(20, 201)), replace=False, p=wi) for _ in range(n)]
    ratings = [rng.integers(1, 6, it.shape[0]).astype(np.float64) for it in items]
    return items, ratings


def levels(items, ni, kernel):
    """The batch's level count by the rule of mfrec_fold_in_kmf (include/mfrec_b200.h)."""
    if kernel == "train_logistic_kernel":
        return 1
    last, top = np.zeros(ni, dtype=np.int64), 0
    for it in items:
        lv = int(last[it].max()) + 1
        last[it] = lv
        top = max(top, lv)
    return top


def add_user(rec, label, items, ratings, kernel):
    """add_user (kmf.py:149-172); its own steps with retrain_user's kernel argument for the linear kernel."""
    if kernel == "train_logistic_kernel":
        return rec.add_user(label, items, ratings)
    new_id = rec._get_new_user_id()
    rec.users_index[label] = new_id
    rec.users_label[new_id] = label
    rec.svd_v = np.ascontiguousarray(np.c_[rec.svd_v, np.zeros(rec.dimensionality)])
    rec.users_bias = np.r_[rec.users_bias, 0.0]
    idx = np.zeros([ratings.shape[0], 2], dtype=np.int32)
    idx[:, 0] = new_id
    idx[:, 1] = items
    rec.retrain_user(new_id, idx, ratings, kernel=kernel)
    return new_id


def main():
    nu, ni, _nnz, k = synth.SHAPES["netflix"]
    gpu = gpu_info()
    print("GPU: %s" % gpu, flush=True)
    out = {"gpu": gpu, "shape": [nu, ni, k], "epochs": EPOCHS, "sample": SAMPLE}
    rec = KMFRecommender(nu, ni, {"nbr_epochs": EPOCHS, "nbr_features": k})
    rng = np.random.default_rng(0)
    rec.svd_u = rng.normal(0.0, 0.1, (k, ni))
    rec.svd_v = rng.normal(0.0, 0.1, (k, nu))
    rec.items_bias = rng.normal(0.0, 0.1, ni)
    rec.users_bias = rng.normal(0.0, 0.1, nu)
    saved = rec.svd_u.copy(), rec.svd_v, rec.items_bias.copy(), rec.users_bias

    def reset():
        rec.svd_u[...], rec.svd_v, rec.items_bias[...], rec.users_bias = saved
        for label in rec.users_label[nu:]:
            rec.users_index.pop(label, None)
        del rec.users_label[nu:]

    ctx = _native.default_context()
    items, ratings = new_users(max(SIZES), ni)
    print("model %d x %d, k = %d, %d epochs; new users: %d-%d ratings, mean %.0f"
          % (nu, ni, k, EPOCHS, min(len(i) for i in items), max(len(i) for i in items),
             np.mean([len(i) for i in items])), flush=True)
    # warm-up: module load, first launches, the host gather path
    rec.add_users(["w0", "w1"], items[:2], ratings[:2])
    add_user(rec, "w2", items[2], ratings[2], "train_logistic_kernel")
    ctx.sync()
    reset()
    for kernel in KERNELS:
        np.random.seed(0)
        n0 = ctx.launch_count
        t0 = time.perf_counter()
        for j in range(SAMPLE):
            add_user(rec, "s%d" % j, items[j], ratings[j], kernel)
        ctx.sync()
        per_user = (time.perf_counter() - t0) / SAMPLE
        loop_launches = (ctx.launch_count - n0) / SAMPLE
        reset()
        for n in SIZES:
            np.random.seed(0)
            labels = ["n%d" % j for j in range(n)]
            n0 = ctx.launch_count
            t0 = time.perf_counter()
            rec.add_users(labels, items[:n], ratings[:n], kernel=kernel)
            ctx.sync()
            dt = time.perf_counter() - t0
            launches = ctx.launch_count - n0
            reset()
            out.setdefault(kernel.split("_")[1], {})["n%d" % n] = dict(
                loop_s=round(per_user * n, 3), loop_ms_per_user=round(per_user * 1e3, 2), batch_s=round(dt, 4),
                speedup=round(per_user * n / dt, 1), launches=launches, levels=levels(items[:n], ni, kernel))
            print("%-21s %6d users: add_user loop %9.2f s (%.1f ms/user on %d users, %.0f launches) | "
                  "add_users %8.3f s (%d launches, %d levels) | speed-up %.1fx"
                  % (kernel, n, per_user * n, per_user * 1e3, SAMPLE, loop_launches * n, dt, launches,
                     levels(items[:n], ni, kernel), per_user * n / dt), flush=True)
    print(json.dumps(out), flush=True)


if __name__ == "__main__":
    main()
