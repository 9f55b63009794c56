"""bench.py's reference arm (`--impl reference`) runs on host cores only: check, without a GPU, that
it prints one JSON line with the keys of the contract (tiny sample so that it takes seconds)."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_the_contract_line():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1",
                          "--warmup", "1", "--cpu-sample", "20000"], stdout=subprocess.PIPE, stderr=subprocess.PIPE,
                         text=True, timeout=300, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [ln for ln in out.stdout.splitlines() if ln.startswith("{")]
    assert len(lines) == 1, out.stdout
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "rating_updates_per_s" and d["unit"] == "updates/s"
    assert d["value"] > 0 and d["higher_is_better"] is True and d["steps"] == 1
    assert d["cpu_baseline"]["kind"] in ("reference", "port") and d["cpu_baseline"]["cores"] == 1
    assert d["e2e"] == {"value": d["value"], "unit": "updates/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert "workload" in d["config"] and "model" not in d["config"]


@pytest.mark.parametrize("extra", [["--steps", "0"], ["--impl", "reference", "--dump-outputs", "DIR"],
                                   ["--gpus", "2", "--dump-outputs", "DIR"]])
def test_arguments_the_bench_cannot_honour_are_refused(extra, tmp_path):
    extra = [str(tmp_path / "dump") if a == "DIR" else a for a in extra]
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + extra, stdout=subprocess.PIPE,
                         stderr=subprocess.PIPE, text=True, timeout=300, cwd=ROOT)
    assert out.returncode == 2 and "error:" in out.stderr and out.stdout == "", out.stderr[-500:]
    assert not (tmp_path / "dump").exists()


def test_reference_arm_other_ranks_exit_quietly():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2",
                          "--steps", "1", "--warmup", "1", "--cpu-sample", "20000"], stdout=subprocess.PIPE,
                         stderr=subprocess.PIPE, text=True, timeout=300, cwd=ROOT, env=env)
    assert out.returncode == 0 and out.stdout.strip() == "", (out.stdout, out.stderr[-500:])
