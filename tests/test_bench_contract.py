"""bench.py's reference arm runs on the host cores (no GPU needed): one bounded step at a reduced size must print ONE
JSON line with the contract's keys (the same line shape the GPU arm prints)."""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_the_contract_line():
    # as torchrun launches it: OMP_NUM_THREADS=1 in the environment must not throttle the CPU arm to one thread
    env = dict(os.environ, OMP_NUM_THREADS="1", JG_CPU_THREADS="2")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1",
                        "--warmup", "0", "--size", "64", "--batch", "1"], capture_output=True, text=True, timeout=600,
                       cwd=ROOT, env=env)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1, r.stdout
    d = json.loads(lines[0])
    for key in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
                "vs_baseline", "dtype", "data", "config", "e2e", "cpu_baseline", "impl"):
        assert key in d, key
    assert d["impl"] == "reference" and d["unit"] == "images/s" and d["higher_is_better"] is True
    assert d["value"] > 0 and d["cpu_baseline"]["kind"] in ("port", "reference") and d["cpu_baseline"]["cores"] >= 1
    assert d["e2e"]["h2d_bytes_per_step"] == 0 and d["e2e"]["d2h_bytes_per_step"] == 0
    assert "workload" in d["config"]
    assert d["cpu_baseline"]["cores"] == 2                       # the explicit thread count, not torchrun's 1
    assert d["steps"] == d["cpu_baseline"]["steps_timed"] == 1   # the line reports what was really timed
    if os.path.exists(os.path.join(ROOT, "oracle", "_ref", "models", "base_model.py")):
        assert d["cpu_baseline"]["kind"] == "reference"
