"""bench.py --dump-outputs at a tiny size: the outputs of the last timed step of every leg land in DIR as float32 .npy
files, and the result line reports exactly the requested number of timed steps."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_bench_dumps_the_outputs_of_every_timed_leg(tmp_path):
    out = tmp_path / "outputs"
    cmd = [sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--steps", "3", "--warmup", "1", "--batch", "2",
           "--sustain-seconds", "0", "--no-cpu-baseline", "--no-eager-baseline", "--dump-outputs", str(out)]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=900, cwd=tmp_path)
    assert r.returncode == 0, r.stderr[-3000:]
    line = json.loads(r.stdout.strip().splitlines()[-1])
    assert line["steps"] == 3 and line["gpu_launches"] == 3 * line["launches_per_step"]
    got = {f[:-4]: np.load(out / f) for f in os.listdir(out)}
    assert sorted(got) == ["logits", "mask", "train_loss", "train_params"]
    assert all(a.dtype == np.float32 for a in got.values())
    assert sum(a.nbytes for a in got.values()) <= 64 << 20
    assert got["logits"].shape == (2, 10, 256, 512) and np.isfinite(got["logits"]).all()
    m = got["mask"]
    assert m.shape == (2, 256, 512) and np.array_equal(m, np.round(m)) and m.min() >= 0 and m.max() <= 9
    assert got["train_loss"].shape == () and np.isfinite(got["train_loss"])
    assert got["train_params"].shape == (1 << 22,) and np.isfinite(got["train_params"]).all()
