"""GPU test: `bench.py --dump-outputs DIR` writes what the last device-timed step computed, and two runs with the same
arguments see the same inputs."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
DUMPED = {"sample": ("std",)}
TRAINING = ("gammas", "loss_terms", "params_sample")


def _bench(out_dir, workload):
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--workload", workload, "--steps", "2",
                        "--warmup", "3", "--no-cpu-baseline", "--no-gpu-reference", "--no-profile",
                        "--dump-outputs", str(out_dir)], capture_output=True, text=True, timeout=900, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1, r.stdout[-2000:]
    return json.loads(lines[0])


def _load(out_dir, names):
    assert sorted(os.listdir(out_dir)) == sorted(n + ".npy" for n in names)
    return {n: np.load(os.path.join(out_dir, n + ".npy")) for n in names}


@pytest.mark.gpu
@pytest.mark.parametrize("workload", ["cond_grid", "vae", "sample"])
def test_dump_outputs_are_the_last_timed_step(tmp_path, workload):
    d = _bench(tmp_path, workload)
    names = DUMPED.get(workload, TRAINING)
    arrs = _load(tmp_path, names)
    assert all(a.dtype in (np.float32, np.float64) and a.size and np.isfinite(a).all() for a in arrs.values())
    assert sum(a.nbytes for a in arrs.values()) <= 64 << 20
    ret = arrs[names[0] if workload == "sample" else "loss_terms"]
    # bench.py reports the last element of the timed region's final output (of its first five) as last_loss
    assert float(ret.reshape(-1)[:5][-1]) == d["config"]["last_loss"]
    if workload != "sample":
        assert arrs["loss_terms"].shape == (5,)


@pytest.mark.gpu
def test_dump_outputs_repeat_with_the_same_arguments(tmp_path):
    runs = []
    for tag in ("a", "b"):
        _bench(tmp_path / tag, "cond_grid")
        runs.append(_load(tmp_path / tag, TRAINING))
    a, b = runs
    # Atomics make the sums order-dependent, so runs agree to rounding, not bit for bit: on a B200 the loss terms of two
    # runs differed by up to 1.2e-4 (relative).  Adam moves a weight by about lr = 1e-4 per step, and the five steps
    # before the dump can move a zero-gradient bias in opposite directions in two runs: at most 1e-3 apart.
    np.testing.assert_allclose(a["loss_terms"], b["loss_terms"], rtol=1e-3)
    np.testing.assert_allclose(a["gammas"], b["gammas"], rtol=1e-6)
    np.testing.assert_allclose(a["params_sample"], b["params_sample"], rtol=0, atol=2e-3)
