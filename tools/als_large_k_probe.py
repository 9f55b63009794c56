"""ALS-WRMF seconds per epoch (one user sweep + one item sweep) across k at ML-20M shape: the
one-CTA row solver (k <= 165 on a 227 KB device) and the cluster row solver above it.

The problem is bench.py's secondary_als one (synth.SHAPES["ml20m"], gpu_synth seed 3, the
reference's [0, counts...] arrays); the drop-in `als_wrmf` is timed with host arrays in and out, and
the per-epoch time is the difference of a 3-epoch and a 1-epoch call (best of REPS each), so the
transfers cancel.  Beside it: row solves per second and the float64 operation count from shapes,
sum_rows(span * k^2) + rows * k^3 / 3 per pass (Gram assembly + Cholesky), over the epoch time.
Prints one JSON document; KS=64,128,... and REPS=n override the defaults."""
import json
import os
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

import numpy as np  # noqa: E402
import torch  # noqa: E402

import bench  # noqa: E402
from mfrec_b200 import _native, synth  # noqa: E402
from mfrec_b200.lib import als_implicit  # noqa: E402


def gpu_info():
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                         capture_output=True, text=True).stdout.strip()
    return {"nvidia_smi": out, "torch_name": torch.cuda.get_device_name(0)}


def main():
    ks = [int(x) for x in os.environ.get("KS", "64,128,160,192,256").split(",")]
    reps = int(os.environ.get("REPS", "2"))
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
    rng = np.random.default_rng(5)
    res = {"gpu": gpu_info(), "shape": "ml20m-shaped implicit feedback %dx%d nnz=%d" % (nu, ni, nnz),
           "max_user_span": int(ur.max()), "max_item_span": int(ir.max()), "reps": reps, "runs": []}
    for k in ks:
        def call(epochs):
            u, v = rng.normal(0, 0.1, (k, ni)), rng.normal(0, 0.1, (k, nu))
            t0 = time.perf_counter()
            als_implicit.als_wrmf(epochs, k, u, v, None, None, ur, uc, ir, ic, nu, ni, c_pos=1, k=0.015)
            dt = time.perf_counter() - t0
            assert np.isfinite(u).all() and np.isfinite(v).all()
            return dt
        call(1)
        lo = min(call(1) for _ in range(reps))
        hi = min(call(3) for _ in range(reps))
        per_epoch = (hi - lo) / 2.0
        ops = 2 * (nnz * k * k) + (nu + ni) * k ** 3 / 3.0
        run = {"k": k, "solver": "one CTA per row" if k <= 165 else "cluster per row",
               "s_per_epoch": per_epoch, "row_solves_per_s": (nu + ni) / per_epoch,
               "fp64_ops_per_epoch": ops, "fp64_gflop_per_s": ops / per_epoch / 1e9,
               "call_1_epoch_s": lo, "call_3_epochs_s": hi}
        print(json.dumps(run), flush=True)
        res["runs"].append(run)
    res["gpu_after"] = gpu_info()
    print(json.dumps(res, indent=1))


if __name__ == "__main__":
    main()
    sys.stdout.flush()
    os._exit(0)
