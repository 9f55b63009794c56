"""bench.py --dump-outputs on the GPU: the files hold what the last timed step returned, two runs with
the same arguments write identical arrays, and --steps counts timed epochs (3 warm-up + 2 timed epochs
leave the same model as 4 + 1)."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
MODEL = ["item_bias", "item_factors", "item_ids", "sq_err", "user_bias", "user_factors", "user_ids"]
TOPN = ["topn_counts", "topn_items", "topn_scores", "topn_user_ids"]


def run_bench(out, names, warmup, steps, *extra):
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--warmup", str(warmup), "--steps", str(steps),
                        "--dump-outputs", str(out)] + list(extra),
                       stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, timeout=600, cwd=ROOT)
    assert p.returncode == 0, p.stderr[-2000:]
    line = json.loads([ln for ln in p.stdout.splitlines() if ln.startswith("{")][-1])
    assert line["steps"] == steps and line["warmup"] == warmup
    assert sorted(f[:-4] for f in os.listdir(out)) == names
    assert sum(os.path.getsize(os.path.join(out, f)) for f in os.listdir(out)) < 64e6
    dump = {n: np.load(os.path.join(out, n + ".npy")) for n in names}
    assert all(x.dtype == np.float64 and np.isfinite(x).all() for x in dump.values())
    return line, dump


def test_dump_outputs_are_reproducible_and_follow_steps(tmp_path):
    flags = ("--workload", "ml100k", "--no-e2e", "--no-secondary", "--no-cpu")
    line, a = run_bench(tmp_path / "a", MODEL, 3, 2, *flags)
    _, b = run_bench(tmp_path / "b", MODEL, 3, 2, *flags)
    _, c = run_bench(tmp_path / "c", MODEL, 4, 1, *flags)
    nu, ni, nnz, k = 943, 1682, 100_000, 20
    assert a["item_factors"].shape == (k, ni) and a["user_factors"].shape == (k, nu)
    assert np.array_equal(a["item_ids"], np.arange(ni)) and np.array_equal(a["user_ids"], np.arange(nu))
    assert np.abs(a["user_bias"]).max() > 0
    # the squared-error sum is the last epoch's: the same epoch the line's RMSE curve ends with
    assert len(line["rmse_per_epoch"]) == 5
    np.testing.assert_allclose(a["sq_err"][0], line["rmse_per_epoch"][-1] ** 2 * nnz, rtol=1e-12)
    for n in MODEL:
        assert np.array_equal(a[n], b[n]), "same arguments, different %s" % n
        assert np.array_equal(a[n], c[n]), "3 + 2 epochs and 4 + 1 epochs differ in %s" % n


def test_topn_dump_is_reproducible_and_matches_float64_scores(tmp_path):
    sys.path.insert(0, ROOT)
    import bench
    from mfrec_b200 import synth
    _, a = run_bench(tmp_path / "a", TOPN, 3, 1, "--workload", "topn")
    _, b = run_bench(tmp_path / "b", TOPN, 3, 1, "--workload", "topn")
    for n in TOPN:
        assert np.array_equal(a[n], b[n]), "same arguments, different %s" % n
    nu, ni, _nnz, k = synth.SHAPES["netflix"]
    users = a["topn_user_ids"].astype(np.int64)
    assert 0 < users.shape[0] < nu and np.all(np.diff(users) > 0) and users[-1] < nu
    assert a["topn_items"].shape == (users.shape[0], 100) and np.all(a["topn_counts"] == 100)
    # the dumped rows are the sampled users' rows: re-score a few of them in float64
    u0, v0 = synth.init_factors(nu, ni, k, seed=2)
    rows = np.arange(0, users.shape[0], users.shape[0] // 16)
    want_items, want_scores = bench.topn_float64(u0, v0, users[rows], 100)
    np.testing.assert_allclose(a["topn_scores"][rows], want_scores, rtol=1e-5, atol=1e-6)
    assert np.mean(a["topn_items"][rows] == want_items) > 0.95     # fp32 vs fp64 may swap near-ties
