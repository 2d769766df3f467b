"""CPU test (-m "not gpu"): the reference arm of bench.py (`--impl reference`, the CPU oracle timed on the host cores)
prints ONE JSON line with the keys the measurement contract names."""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_contract_line():
    env = dict(os.environ, OMP_NUM_THREADS=str(min(8, os.cpu_count() or 1)))
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "1"],
                       capture_output=True, text=True, timeout=600, cwd=ROOT, env=env)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1, r.stdout[-2000:]
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["unit"] == "patches/s" and d["higher_is_better"] is True
    assert d["n_gpus"] == 1 and d["value"] > 0 and d["ms_per_step"] > 0 and d["vs_baseline"] is None
    assert "workload" in d["config"] and d["data"] == "synthetic"
    cb = d["cpu_baseline"]
    assert cb["kind"] in ("port", "reference") and cb["cores"] >= 1 and cb["value"] == d["value"] and cb["sample"]
    e2e = d["e2e"]
    assert e2e["value"] == d["value"] and e2e["h2d_bytes_per_step"] == 0 and e2e["d2h_bytes_per_step"] == 0


def test_steps_below_one_is_rejected():
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "0"],
                       capture_output=True, text=True, timeout=300, cwd=ROOT)
    assert r.returncode == 2 and "--steps must be at least 1" in r.stderr


def test_reference_arm_non_zero_ranks_exit_quietly():
    """Under torchrun (N > 1) only rank 0 runs the CPU arm; the other ranks exit 0 without output."""
    env = dict(os.environ, RANK="1", LOCAL_RANK="1", WORLD_SIZE="2", MASTER_ADDR="127.0.0.1", MASTER_PORT="29599")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2", "--steps", "1", "--warmup", "1"],
                       capture_output=True, text=True, timeout=300, cwd=ROOT, env=env)
    assert r.returncode == 0, r.stderr[-2000:]
    assert not [l for l in r.stdout.splitlines() if l.startswith("{")]
