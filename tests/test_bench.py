"""bench.py's command line: the number of timed steps and the dump of the last timed step."""
import json
import subprocess
import sys
from pathlib import Path

import numpy as np
import pytest

BENCH = Path(__file__).resolve().parent.parent / "bench.py"
NAMES = ("loss", "grads", "params")


def test_bench_rejects_zero_steps():
    out = subprocess.run([sys.executable, str(BENCH), "--steps", "0"], capture_output=True, text=True)
    assert out.returncode == 2 and "--steps" in out.stderr


def _run_bench(out_dir, steps):
    cmd = [sys.executable, str(BENCH), "--gpus", "1", "--model", "resnet18", "--batch", "32", "--steps", str(steps),
           "--warmup", "3", "--no-e2e", "--no-nccl-arm", "--dump-outputs", str(out_dir)]
    out = subprocess.run(cmd, capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stderr[-4000:]
    return json.loads(out.stdout.strip().splitlines()[-1]), {n: np.load(out_dir / f"{n}.npy") for n in NAMES}


@pytest.mark.gpu
def test_bench_dumps_the_last_timed_step(tmp_path):
    steps = 2
    res, d = _run_bench(tmp_path / "a", steps)
    assert res["steps"] == steps
    assert res["gpu_launches"] > 0 and res["gpu_launches"] % steps == 0  # the same launches in every timed step
    loss, grads, params = (d[n] for n in NAMES)
    assert loss.dtype == np.float64 and loss.shape == (1,) and abs(loss[0] - res["final_loss"]) < 1e-3
    # resnet18 has 11.7M parameters: both arrays are the same 4M-element sample
    assert grads.dtype == params.dtype == np.float32 and grads.shape == params.shape == (1 << 22,)
    assert np.isfinite(grads).all() and np.isfinite(params).all() and np.abs(grads).max() > 0
    assert sum(f.stat().st_size for f in (tmp_path / "a").iterdir()) <= 64 << 20
    # a second process with the same arguments computes exactly the same thing
    _, d2 = _run_bench(tmp_path / "b", steps)
    for n in NAMES:
        assert np.array_equal(d[n], d2[n]), n
