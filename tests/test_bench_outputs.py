"""`bench.py --dump-outputs DIR` (`-m gpu`): the logits of the last timed decode step land in DIR/logits.npy as float32, and
the inputs are seeded, so the same number of decode steps gives the same logits from run to run.  Two runs that split the
same five steps differently between `--warmup` and `--steps` end on the same step: each timed step is one decode step."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _bench(out_dir, steps, warmup):
    # two layers (one dense, one sparse) over a short context: this test is about what is written, not about speed
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", str(steps), "--warmup", str(warmup), "--layers", "2",
                        "--P", "4000", "--M", "8192", "--no-cpu-baseline", "--dump-outputs", str(out_dir)],
                       capture_output=True, text=True, cwd=ROOT, timeout=900)
    assert r.returncode == 0, r.stderr[-3000:]
    line = [json.loads(ln) for ln in r.stdout.splitlines() if ln.startswith("{")][-1]
    assert line["steps"] == steps and line["warmup"] == warmup
    return np.load(os.path.join(out_dir, "logits.npy"))


def test_dump_outputs_last_timed_step(cuda_lib, tmp_path):
    a = _bench(tmp_path / "a", steps=3, warmup=2)
    b = _bench(tmp_path / "b", steps=2, warmup=3)
    assert a.dtype == np.float32 and a.shape == (1, 128256) and np.isfinite(a).all() and float(np.abs(a).max()) > 0
    # the sparse layer's CTA merge may sum in a different order from run to run: fp32 noise, not a different sample
    assert float(np.abs(a - b).max()) <= 1e-2 * float(np.abs(a).max())
