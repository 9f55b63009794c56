"""All-users top-N served from N GPUs of one process (mfrec_model_topn_sweep_multi, _native.ModelSet)
against one GPU (mfrec_model_topn_sweep): model build time, whole-call time, each shard's sweep and
finish time, merged stats, and whether every output equals the N = 1 call.

Problem: bench.py's run_topn (synth.init_factors seed 2, k = 128, N = 100, predict_rating, all users,
all items, no rated lists) at Netflix shape (480,000 x 17,700) and at Yahoo shape (1,800,000 x 136,000).
Outputs go to pinned host arrays; models are resident (built once per N, timed separately).  N = 1 is one
Model on device 0; N > 1 is a ModelSet over devices 0 .. N-1.  With SHARE=1 the same N also runs as N
shards on device 0 (the split path without a second GPU).  Per-shard times come from the library's
MFREC_TOPN_SHARD_TIMES lines (CUDA events per shard, last timed call).
Prints one JSON line; SHAPES=netflix,yahoo / NS=1,2,4,8 / CALLS=n (>= 5) / SHARE=0|1 override the
defaults.  N above the visible GPU count is skipped and listed."""
import json
import os
import subprocess
import sys
import tempfile
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

import numpy as np  # noqa: E402
import torch  # noqa: E402

from mfrec_b200 import _native, synth  # noqa: E402

N_TOP = 100


def gpu_info():
    out = subprocess.run(["nvidia-smi", "--query-gpu=index,name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()
    return {"nvidia_smi": out, "torch_name": torch.cuda.get_device_name(0), "device_count": torch.cuda.device_count()}


def pinned_out(nu):
    items = torch.empty((nu, N_TOP), dtype=torch.int32).pin_memory()
    scores = torch.empty((nu, N_TOP), dtype=torch.float64).pin_memory()
    counts = torch.empty(nu, dtype=torch.int32).pin_memory()
    return items, scores, counts


def run(devices, u, v, calls, ref, times_file):
    nu, ni = v.shape[1], u.shape[1]
    k = u.shape[0]
    for d in set(devices):
        torch.cuda.synchronize(d)
    t0 = time.perf_counter()
    if len(devices) == 1:
        model = _native.Model(k, ni, nu, u, v, None, None, ctx=_native.default_context(devices[0]))
    else:
        model = _native.ModelSet(devices, k, ni, nu, u, v, None, None)
    build_ms = (time.perf_counter() - t0) * 1e3
    tens = pinned_out(nu)
    out = tuple(t.numpy() for t in tens)

    def call():
        # users = None: all users (the one-device Model.topn passes 0 .. nu-1, the set passes NULL)
        return model.topn("predict_rating", None, ni, None, None, N_TOP, sweep=True, out=out)[3]

    call()                                                    # warm-up (module load, pools)
    open(times_file, "w").close()
    ms, stats = [], None
    for _ in range(calls):
        t0 = time.perf_counter()
        stats = call()                                        # returns after the results are in host memory
        ms.append((time.perf_counter() - t0) * 1e3)
    if len(devices) == 1:
        shards = [{"device": devices[0], "users": [0, nu], "sweep_ms": float(stats[2]), "finish_ms": float(stats[7]),
                   "redone": float(stats[0])}]
    else:
        with open(times_file) as f:
            shards = json.loads(f.read().strip().splitlines()[-1])["shards"]
    res = {"devices": list(devices), "model_build_ms": build_ms, "call_ms_median": float(np.median(ms)),
           "call_ms": ms, "shards": shards,
           "stats": {"users_redone": float(stats[0]), "candidates_per_user": float(stats[1]),
                     "sweep_ms_max": float(stats[2]), "useful_flops": float(stats[3]), "overflows": float(stats[4]),
                     "padded_k": float(stats[5]), "z": float(stats[6]), "finish_ms_max": float(stats[7])}}
    if ref is None:
        ref = tuple(np.array(a) for a in out)
    else:
        res["equal_to_n1"] = bool(all(np.array_equal(a, b) for a, b in zip(out, ref)))
    del model
    return res, ref


def main():
    shapes = os.environ.get("SHAPES", "netflix,yahoo").split(",")
    ns_all = [int(x) for x in os.environ.get("NS", "1,2,4,8").split(",")]
    calls = max(5, int(os.environ.get("CALLS", "5")))
    share = os.environ.get("SHARE", "0") == "1"
    ngpu = torch.cuda.device_count()
    torch.cuda.set_device(0)
    times_file = os.path.join(tempfile.mkdtemp(), "shard_times.jsonl")
    os.environ["MFREC_TOPN_SHARD_TIMES"] = times_file        # read by the library at every multi call
    doc = {"gpus": gpu_info(), "problem": "bench.py run_topn: predict_rating, N = 100, all users x all items",
           "calls": calls, "skipped_n": [n for n in ns_all if n > ngpu], "runs": {}}
    for shape in shapes:
        nu, ni, _nnz, k = synth.SHAPES[shape]
        u, v = synth.init_factors(nu, ni, k, seed=2)
        runs, ref = [], None
        for n in [1] + [n for n in ns_all if 1 < n <= ngpu]:
            r, ref = run(list(range(n)), u, v, calls, ref, times_file)
            runs.append(r)
            print(json.dumps({"shape": shape, "n": n, "call_ms_median": r["call_ms_median"],
                              "equal_to_n1": r.get("equal_to_n1")}), file=sys.stderr, flush=True)
        if share:
            for n in [n for n in ns_all if n > 1]:
                r, _ = run([0] * n, u, v, calls, ref, times_file)
                r["one_device"] = True
                runs.append(r)
        doc["runs"][shape] = {"nu": nu, "ni": ni, "k": k, "results": runs}
        del u, v, ref
    doc["gpus_after"] = gpu_info()["nvidia_smi"]
    print(json.dumps(doc))


if __name__ == "__main__":
    main()
