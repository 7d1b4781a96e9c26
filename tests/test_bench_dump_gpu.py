"""-m gpu: bench.py --dump-outputs writes the logits of the last timed step, the same for every run with the same inputs."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _bench(steps, out):
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--arch", "resnet18", "--scheme", "uniform4", "--batch", "8",
                        "--steps", str(steps), "--warmup", "1", "--no-cpu-baseline", "--no-roofline", "--no-batch8",
                        "--dump-outputs", str(out)], capture_output=True, text=True, timeout=900, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-3000:]
    lines = [ln for ln in r.stdout.splitlines() if ln.startswith("{")]
    assert len(lines) == 1
    return json.loads(lines[0]), np.load(os.path.join(out, "logits.npy"))


def test_dump_is_the_last_timed_step(tmp_path):
    """bench.py rotates 4 seeded input batches: steps 1 and 5 both end on batch 0, steps 2 on batch 1."""
    d1, l1 = _bench(1, tmp_path / "s1")
    d5, l5 = _bench(5, tmp_path / "s5")
    d2, l2 = _bench(2, tmp_path / "s2")
    assert (d1["steps"], d5["steps"], d2["steps"]) == (1, 5, 2)
    assert sorted(os.listdir(tmp_path / "s1")) == ["logits.npy"]
    assert l1.dtype == np.float32 and l1.shape == (8, 1000) and np.isfinite(l1).all()
    assert not d1["config"]["overflow_flag_seen"] and d1["parity"]["bit_equal"]
    assert np.array_equal(l1, l5)
    assert not np.array_equal(l1, l2)
