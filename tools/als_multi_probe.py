"""ALS-WRMF split over N GPUs of one process (mfrec_train_als_wrmf_multi): seconds per epoch and per
half-pass, per shard and overall, at ML-20M shape, for several k and N.

The problem and the timing are those of tools/als_large_k_probe.py: bench.py's secondary_als problem
(synth.SHAPES["ml20m"], gpu_synth seed 3, the reference's [0, counts...] arrays), the drop-in
`als_wrmf` timed with host arrays in and out, and an epoch's time taken as the difference of a 3-epoch
and a 1-epoch call (best of REPS each), so the transfers cancel.  N = 1 is the one-device call, i.e.
that probe's number.  For N > 1 `options["devices"]` = [0 .. N-1].

Beside the wall-clock epoch, for every run:
  - each shard's milliseconds per user / item half-pass (Gram + solve, CUDA events the library records
    when MFREC_ALS_SHARD_TIMES names a file; mean over the epochs of the 3-epoch call), and its row
    ranges;
  - the estimated cost of the slowest shard, sum(deg * k^2 + k^3 / 3) over its rows of both sides,
    against the total / N;
  - whether u and v after the 3-epoch call EQUAL those of the N = 1 call from the same start.
Once per k: the time of the longest single row (the item with the most neighbours, one CTA or
cluster's serial work, a floor no split removes), as the per-epoch time of a call whose only active
row is that item minus that of a call without active rows.
Prints one JSON document; KS=64,165 / NS=1,2 / REPS=n override the defaults.  N above the visible GPU
count is skipped and listed."""
import json
import os
import subprocess
import sys
import tempfile
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

import numpy as np  # noqa: E402
import torch  # noqa: E402

import bench  # noqa: E402
from mfrec_b200 import _native, synth  # noqa: E402
from mfrec_b200.lib import als_implicit  # noqa: E402


def gpu_info():
    out = subprocess.run(["nvidia-smi", "--query-gpu=index,name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()
    return {"nvidia_smi": out, "torch_name": torch.cuda.get_device_name(0), "device_count": torch.cuda.device_count()}


def main():
    ks = [int(x) for x in os.environ.get("KS", "64,165,166,256").split(",")]
    ns_all = [int(x) for x in os.environ.get("NS", "1,2,4,8").split(",")]
    reps = int(os.environ.get("REPS", "2"))
    ngpu = torch.cuda.device_count()
    ns = [n for n in ns_all if n <= ngpu]
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(0)
    _native.default_context(0)
    nu, ni, nnz, _ = synth.SHAPES["ml20m"]
    idx_d, _r = bench.gpu_synth(torch, dev, nu, ni, nnz, seed=3)
    idx = idx_d.cpu().numpy()
    del idx_d, _r
    users, items = idx[:, 0].astype(np.int64), idx[:, 1].astype(np.int64)
    ou, oi = np.lexsort((items, users)), np.lexsort((users, items))
    ur = np.r_[0, np.bincount(users, minlength=nu)].astype(np.int32)
    ir = np.r_[0, np.bincount(items, minlength=ni)].astype(np.int32)
    uc = np.ascontiguousarray(items[ou], np.int32)
    ic = np.ascontiguousarray(users[oi], np.int32)
    deg_u, deg_i = ur[1:].astype(np.int64), ir[1:].astype(np.int64)
    hot = int(np.argmax(deg_i))
    hot_cols = np.ascontiguousarray(ic[int(deg_i[:hot].sum()):int(deg_i[:hot + 1].sum())])
    times_file = tempfile.NamedTemporaryFile(prefix="als_multi_times_", suffix=".jsonl", delete=False).name
    res = {"gpu": gpu_info(), "shape": "ml20m-shaped implicit feedback %dx%d nnz=%d" % (nu, ni, nnz),
           "max_user_span": int(deg_u.max()), "max_item_span": int(deg_i.max()), "reps": reps,
           "n_skipped": [n for n in ns_all if n > ngpu], "runs": [], "longest_row": []}

    def als(devices, epochs, u, v, row_u=ur, col_u=uc, row_i=ir, col_i=ic):
        als_implicit.options["devices"] = list(devices)
        try:
            t0 = time.perf_counter()
            als_implicit.als_wrmf(epochs, u.shape[0], u, v, None, None, row_u, col_u, row_i, col_i, nu, ni,
                                  c_pos=1, k=0.015)
            return time.perf_counter() - t0
        finally:
            als_implicit.options["devices"] = []

    def per_epoch(devices, k, **kw):
        rng = np.random.default_rng(5)

        def call(epochs):
            u, v = rng.normal(0, 0.1, (k, ni)), rng.normal(0, 0.1, (k, nu))
            return als(devices, epochs, u, v, **kw)
        call(1)
        lo = min(call(1) for _ in range(reps))
        hi = min(call(3) for _ in range(reps))
        return (hi - lo) / 2.0, lo, hi

    for k in ks:
        kk, kkk = float(k) * k, float(k) ** 3 / 3.0
        cost_u, cost_i = deg_u * kk + kkk, deg_i * kk + kkk
        total = float(cost_u.sum() + cost_i.sum())
        # the floor: one row with the hottest item's neighbours (solved as item 0), against no row at
        # all (the same Grams and transfers)
        empty = np.zeros(1, np.int32)
        t_hot, _, _ = per_epoch([], k, row_u=empty, col_u=empty, row_i=np.r_[0, deg_i[hot]].astype(np.int32),
                                col_i=hot_cols)
        t_none, _, _ = per_epoch([], k, row_u=empty, col_u=empty, row_i=empty, col_i=empty)
        floor = {"k": k, "item": hot, "neighbours": int(deg_i[hot]), "s_per_epoch_hot_row_only": t_hot,
                 "s_per_epoch_no_rows": t_none, "s_longest_row": t_hot - t_none}
        print(json.dumps(floor), flush=True)
        res["longest_row"].append(floor)
        rng = np.random.default_rng(k)
        u_start, v_start = rng.normal(0, 0.1, (k, ni)), rng.normal(0, 0.1, (k, nu))
        ref = None
        for n in ns:
            devices = list(range(n)) if n > 1 else []
            s_epoch, lo, hi = per_epoch(devices, k)
            # one more 3-epoch call from the common start: equality with N = 1 and the shard times
            u, v = u_start.copy(), v_start.copy()
            open(times_file, "w").close()
            os.environ["MFREC_ALS_SHARD_TIMES"] = times_file
            try:
                als(devices, 3, u, v)
                if n == 1:   # the one-shard split path: its shard times, and the same factors again
                    u1, v1 = u_start.copy(), v_start.copy()
                    _native.train_als_wrmf_multi([0], 3, k, u1, v1, ur, uc, ir, ic, nu, ni, 1, 0.015)
                    one_shard_equal = bool(np.array_equal(u1, u) and np.array_equal(v1, v))
            finally:
                del os.environ["MFREC_ALS_SHARD_TIMES"]
            with open(times_file) as f:
                lines = [json.loads(x) for x in f if x.strip()]
            if n == 1:
                ref = (u, v)
            equal = bool(np.array_equal(u, ref[0]) and np.array_equal(v, ref[1]))
            shards = []
            for s in lines[-1]["shards"] if lines else []:
                hp = np.array(s["half_pass_ms"]).reshape(-1, 2)
                cost = float(cost_u[s["users"][0]:s["users"][1]].sum() + cost_i[s["items"][0]:s["items"][1]].sum())
                shards.append({"device": s["device"], "users": s["users"], "items": s["items"],
                               "ms_user_pass": float(hp[:, 0].mean()), "ms_item_pass": float(hp[:, 1].mean()),
                               "ms_epoch": float(hp.sum(axis=1).mean()), "est_cost": cost})
            run = {"k": k, "n_gpus": n, "solver": "one CTA per row" if lines and lines[-1]["csize"] == 1 else "cluster per row",
                   "s_per_epoch": s_epoch, "call_1_epoch_s": lo, "call_3_epochs_s": hi,
                   "s_user_pass_slowest_shard": max(s["ms_user_pass"] for s in shards) / 1e3 if shards else None,
                   "s_item_pass_slowest_shard": max(s["ms_item_pass"] for s in shards) / 1e3 if shards else None,
                   "est_cost_slowest_shard_over_even_share": (max(s["est_cost"] for s in shards) / (total / n)) if shards else None,
                   "identical_to_n1": equal, "shards": shards}
            if n == 1:
                run["one_shard_split_path_identical"] = one_shard_equal
            print(json.dumps(run), flush=True)
            res["runs"].append(run)
    os.unlink(times_file)
    res["gpu_after"] = gpu_info()
    print(json.dumps(res))   # the last line: the whole run


if __name__ == "__main__":
    main()
    sys.stdout.flush()
    os._exit(0)
