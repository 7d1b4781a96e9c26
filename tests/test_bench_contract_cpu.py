"""bench.py contract pieces that run without a GPU: the reference arm (`--impl reference`) prints one JSON line with the
keys the driver reads, and non-zero ranks of a torchrun launch stay silent."""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _run(extra_env=None):
    env = dict(os.environ)
    env.update(extra_env or {})
    return subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--arch", "resnet18", "--scheme", "uniform8",
                           "--steps", "1", "--warmup", "1", "--cpu-batch", "1"], capture_output=True, text=True, timeout=600, env=env, cwd=ROOT)


def test_reference_arm_json_line():
    r = _run()
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [ln for ln in r.stdout.splitlines() if ln.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["higher_is_better"] is True and d["unit"] == "images/s" and d["value"] > 0
    for key in ("metric", "n_gpus", "steps", "warmup", "ms_per_step", "scaling", "vs_baseline", "dtype", "data", "config", "cpu_baseline", "e2e"):
        assert key in d, key
    assert d["config"]["workload"].startswith("resnet18_uniform8")
    assert d["cpu_baseline"]["kind"] in ("port", "reference") and d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["value"] == d["value"]
    assert d["e2e"] == {"value": d["value"], "unit": "images/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}


def test_reference_arm_other_ranks_are_silent():
    r = _run({"RANK": "1", "WORLD_SIZE": "2", "LOCAL_RANK": "1"})
    assert r.returncode == 0 and r.stdout.strip() == ""


def test_bad_arguments_are_refused(tmp_path):
    """No timed step to divide by, and an output dump of the CPU arm (it runs other inputs than the GPU path): usage errors."""
    for args in (["--steps", "0"], ["--impl", "reference", "--dump-outputs", str(tmp_path)]):
        r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + args, capture_output=True, text=True, timeout=300, cwd=ROOT)
        assert r.returncode == 2 and "error" in r.stderr and r.stdout == "", (args, r.stderr[-500:])
    assert not os.listdir(tmp_path)
