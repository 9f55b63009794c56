"""Batched Funk-SVD fold-in (GDRecommender.retrain_users / retrain_items, one mfrec_fold_in_funk
call) against the retrain_user loop (one mfrec_train_funk call per user) at Netflix shape (480k users
x 17.7k items) or another of synth.SHAPES, with GDRecommender's defaults (k = 40, min_epochs 275,
min_improvement 1e-4, lr 0.001, K 0.05, feature_init 0.1), random factors and biases, and users with
20-200 ratings each drawn by item popularity (mfrec_b200.synth).

It prints the host wall time of the retrain_user loop on the first SAMPLE users under the default
(stratified) schedule and under the sequential one, scaled to each batch size; of one
retrain_users call per batch size; of one retrain_items call over ITEMS items of those ratings, the
most popular item (the longest chain) among them; the kernel launches of each; whether the batch
equals the sequential loop on the sampled users bit for bit, and how far the stratified loop is from
it (or the error with which the stratified loop fails); then all of it, with the GPU's name and
power limit, as one JSON line.  Every timed span ends in a device synchronise.  Environment: SHAPE
(netflix), USERS (1000,10000), SAMPLE (10), ITEMS (1000)."""
import json
import os
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np

from mfrec_b200 import _native, synth
from mfrec_b200.lib import gd_estimator
from mfrec_b200.recommendation import GDRecommender

SIZES = [int(x) for x in os.environ.get("USERS", "1000,10000").split(",")]
SAMPLE = int(os.environ.get("SAMPLE", "10"))
ITEMS = int(os.environ.get("ITEMS", "1000"))
SHAPE = os.environ.get("SHAPE", "netflix")


def gpu_info():
    try:
        return subprocess.check_output(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                                       text=True).strip().splitlines()[0]
    except (OSError, subprocess.CalledProcessError):
        return "unknown GPU"


def user_ratings(users, nu, ni, seed=7):
    """(ratings_index, ratings) of `users`, 20-200 items each drawn by popularity, shuffled."""
    _wu, wi = synth.marginals(nu, ni)
    rng = np.random.default_rng(seed)
    idx = []
    for u in users:
        it = rng.choice(ni, int(rng.integers(20, 201)), replace=False, p=wi)
        idx.append(np.stack([np.full(it.shape[0], u), it], axis=1))
    idx = np.concatenate(idx).astype(np.int32)
    idx = np.ascontiguousarray(idx[rng.permutation(idx.shape[0])])
    return idx, rng.integers(1, 6, idx.shape[0]).astype(np.float64)


def main():
    nu, ni, _nnz, _k = synth.SHAPES[SHAPE]
    gpu = gpu_info()
    print("GPU: %s" % gpu, flush=True)
    rec = GDRecommender(nu, ni)
    k = rec.dimensionality
    out = {"gpu": gpu, "shape": [nu, ni, k], "min_epochs": rec.min_epochs, "min_improvement": rec.min_improvement,
           "sample": SAMPLE}
    rng = np.random.default_rng(0)
    rec.svd_u = rng.normal(0.0, 0.1, (k, ni))
    rec.svd_v = rng.normal(0.0, 0.1, (k, nu))
    rec.items_bias = rng.normal(0.0, 0.1, ni)
    rec.users_bias = rng.normal(0.0, 0.1, nu)
    rec.overall_bias = 3.6
    saved = rec.svd_u.copy(), rec.svd_v.copy()

    def reset():
        rec.svd_u[...], rec.svd_v[...] = saved

    ctx = _native.default_context()
    users = np.random.default_rng(1).choice(nu, max(SIZES), replace=False)
    idx, r = user_ratings(users, nu, ni)
    cnt = np.bincount(idx[:, 0], minlength=nu)[users]
    print("model %d x %d, k = %d, min_epochs %d; users: %d-%d ratings, mean %.0f"
          % (nu, ni, k, rec.min_epochs, cnt.min(), cnt.max(), cnt.mean()), flush=True)
    sample = users[:SAMPLE]
    sidx = np.ascontiguousarray(idx[np.isin(idx[:, 0], sample)])
    sr = np.ascontiguousarray(r[np.isin(idx[:, 0], sample)])
    # warm-up: module load, first launches, the host gather path
    rec.retrain_users(users[:2], sidx, sr)
    ctx.sync()
    reset()

    loops, out["loop"] = {}, {}
    for sched in ("stratified", "sequential"):
        gd_estimator.options["schedule"] = sched
        try:
            rec.retrain_user(sample[0], sidx, sr)    # warm-up of this path
            ctx.sync()
        except _native.MfrecError as e:             # the stratified layout may not fit the shape
            out["loop"][sched] = dict(error=str(e))
            print("retrain_user loop, %-10s schedule: fails: %s" % (sched, e), flush=True)
            continue
        finally:
            reset()
        np.random.seed(0)
        n0 = ctx.launch_count
        t0 = time.perf_counter()
        for u in sample:
            rec.retrain_user(u, sidx, sr)
        ctx.sync()
        per_user = (time.perf_counter() - t0) / SAMPLE
        loops[sched] = (per_user, (ctx.launch_count - n0) / SAMPLE, rec.svd_v[:, sample].copy())
        reset()
        out["loop"][sched] = dict(ms_per_user=round(per_user * 1e3, 2), launches_per_user=loops[sched][1])
        print("retrain_user loop, %-10s schedule: %8.1f ms/user on %d users, %.0f launches/user"
              % (sched, per_user * 1e3, SAMPLE, loops[sched][1]), flush=True)
    gd_estimator.options["schedule"] = "stratified"

    np.random.seed(0)
    rec.retrain_users(sample, sidx, sr)
    batch_rows = rec.svd_v[:, sample].copy()
    reset()
    out["sample_equals_sequential_loop"] = bool(np.array_equal(batch_rows, loops["sequential"][2]))
    print("batch == sequential loop on the sampled users: %s" % out["sample_equals_sequential_loop"], flush=True)
    if "stratified" in loops:
        out["stratified_loop_max_abs_diff"] = float(np.abs(batch_rows - loops["stratified"][2]).max())
        print("stratified loop max |diff| from the batch: %.3g" % out["stratified_loop_max_abs_diff"], flush=True)

    for n in SIZES:
        m = np.isin(idx[:, 0], users[:n])
        bidx, br = np.ascontiguousarray(idx[m]), np.ascontiguousarray(r[m])
        np.random.seed(0)
        n0 = ctx.launch_count
        t0 = time.perf_counter()
        rec.retrain_users(users[:n], bidx, br)
        ctx.sync()
        dt = time.perf_counter() - t0
        launches = ctx.launch_count - n0
        reset()
        row = dict(batch_s=round(dt, 4), launches=launches, ratings=int(m.sum()), longest_row=int(cnt[:n].max()))
        text = ""
        for s, v in loops.items():
            row["loop_%s_s" % s] = round(v[0] * n, 2)
            row["speedup_vs_%s" % s] = round(v[0] * n / dt, 1)
            text += " | %s loop %.1f s, speed-up %.0fx" % (s, v[0] * n, v[0] * n / dt)
        out["users_n%d" % n] = row
        print("%6d users (%d ratings, longest row %d): retrain_users %8.3f s, %d launches%s"
              % (n, row["ratings"], row["longest_row"], dt, launches, text), flush=True)

    icnt = np.bincount(idx[:, 1], minlength=ni)
    top = int(np.argmax(icnt))
    rated = np.nonzero(icnt)[0]
    items = np.r_[top, np.random.default_rng(2).choice(rated[rated != top], min(ITEMS, rated.shape[0]) - 1,
                                                        replace=False)]
    np.random.seed(0)
    n0 = ctx.launch_count
    t0 = time.perf_counter()
    rec.retrain_items(items, idx, r)
    ctx.sync()
    dt = time.perf_counter() - t0
    launches = ctx.launch_count - n0
    reset()
    out["items"] = dict(n=int(items.shape[0]), batch_s=round(dt, 4), launches=launches,
                        longest_row=int(icnt[top]), ratings=int(icnt[items].sum()))
    print("retrain_items over %d items (%d ratings; the most popular item has %d): %8.3f s, %d launches"
          % (items.shape[0], out["items"]["ratings"], icnt[top], dt, launches), flush=True)
    print(json.dumps(out), flush=True)


if __name__ == "__main__":
    main()
