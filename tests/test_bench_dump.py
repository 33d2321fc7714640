"""bench.py --dump-outputs: what the timed path computed is written after the timed steps, within 64 MB, and two runs
with the same arguments write the same arrays (two builds can then be compared output for output)."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
STEPS, WARMUP = 7, 3


def run_bench(out_dir):
    cmd = [sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--steps", str(STEPS), "--warmup", str(WARMUP),
           "--no-cpu-baseline", "--no-prioritized", "--no-other-configs", "--dump-outputs", str(out_dir)]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
    return json.loads(r.stdout.strip().splitlines()[-1])


@pytest.mark.gpu
def test_dump_outputs_are_reproducible(tmp_path):
    a, b = tmp_path / "a", tmp_path / "b"
    assert run_bench(a)["steps"] == STEPS
    run_bench(b)
    names = sorted(os.listdir(a))
    assert names == sorted(os.listdir(b))
    assert {"cumulated_losses.npy", "td_abs.npy", "optimizer_state.count.npy", "params.Dense_0.kernel.npy",
            "target_params.Dense_0.kernel.npy", "optimizer_state.mu.Dense_0.kernel.npy",
            "optimizer_state.nu.Dense_0.kernel.npy"} <= set(names)
    assert sum(os.path.getsize(a / n) for n in names) <= 64 << 20
    for n in names:
        x, y = np.load(a / n), np.load(b / n)
        assert x.dtype in (np.float32, np.float64), n
        assert np.isfinite(x).all(), n
        np.testing.assert_array_equal(x, y, err_msg=n)
    # every head took one Adam step per warm-up and timed step, and no more
    np.testing.assert_array_equal(np.load(a / "optimizer_state.count.npy"), WARMUP + STEPS)
