"""GPU: bench.py's b200 arm -- `--steps` sets the number of timed steps and `--dump-outputs` writes what the last of
them computed."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_bench_dump_outputs(cuda_dev, tmp_path):
    out = tmp_path / "dump"
    cmd = [sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "4", "--warmup", "3", "--no-parity",
           "--no-torch-eager", "--no-cpu-baseline", "--no-varlen", "--dump-outputs", str(out)]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-3000:]
    line = json.loads([ln for ln in r.stdout.splitlines() if ln.startswith("{")][-1])
    assert line["steps"] == 4 and line["gpu_launches"] == 4 * line["gpu_launches_per_step"]
    arrays = {p.stem: np.load(p) for p in out.glob("*.npy")}
    assert set(arrays) == {"loss", "logits", "grads", "weights"}
    assert sum(a.nbytes for a in arrays.values()) <= 64 << 20
    for name, a in arrays.items():
        assert a.dtype == np.float32 and np.isfinite(a).all(), name
    assert arrays["loss"].shape == (1,) and abs(float(arrays["loss"][0]) - line["loss"]["final"]) < 1e-4
    assert arrays["logits"].shape == (32, 6)
    assert arrays["grads"].shape == arrays["weights"].shape == (1 << 22,)
    assert np.abs(arrays["grads"]).max() > 0 and np.abs(arrays["weights"]).max() > 0
