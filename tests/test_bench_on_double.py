"""bench.py's GPU arm on the kernel test double (tests/bench_on_double.py), tiny sizes: every configuration builds its
workload, runs its timed loops and the instrumented pass, and prints ONE JSON line with the contract's keys.  (Host
logic only: the values are a CPU emulation's.)"""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
KEYS = ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
        "vs_baseline", "dtype", "data", "config", "e2e", "gpu_launches", "clocks", "roofline")


# (configs 4 and 5 run the same way — `python tests/bench_on_double.py --config 4 --size 32 --batch 2` — and are left
# out of the suite for time: they share PaletteTrainer's path with config 2)
@pytest.mark.parametrize("args", [["--config", "2", "--size", "32", "--batch", "2"],
                                  ["--config", "3", "--size", "64", "--batch", "2"],
                                  ["--config", "6", "--size", "32"]], ids=lambda a: "cfg" + a[1])
def test_bench_gpu_arm_runs_end_to_end_on_the_double(args):
    r = subprocess.run([sys.executable, os.path.join(ROOT, "tests", "bench_on_double.py"), "--steps", "1", "--warmup", "1"]
                       + args, capture_output=True, text=True, timeout=900, cwd=ROOT,
                       env=dict(os.environ, OMP_NUM_THREADS="4"))
    assert r.returncode == 0, r.stderr[-3000:]
    lines = [l for l in r.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1, r.stdout[-2000:]
    d = json.loads(lines[0])
    for k in KEYS:
        assert k in d, k
    assert d["n_gpus"] == 1 and d["steps"] == 1 and d["scaling"] == "weak" and d["dtype"] == "bf16"
    assert d["value"] > 0 and d["e2e"]["value"] > 0 and d["e2e"]["h2d_bytes_per_step"] > 0
    assert d["roofline"]["bound"] == "tensor" and "workload" in d["config"]


def test_graft_entry_smoke_runs_on_the_double():
    """__graft_entry__.smoke() (what the driver runs on the B200 before the bench): its host side — build the net, the
    trainer, one explicit-draw step, the oracle comparison at 2e-2 — executes on the double."""
    code = "\n".join([
        "import sys; sys.path[:0] = [%r, %r]" % (ROOT, os.path.join(ROOT, "tests")),
        "import double_plugin; double_plugin.pytest_configure(None)",
        "from joligen_b200 import lib as L; L.load().jg_check_device = lambda: 0",
        "import __graft_entry__ as g; g.smoke()"])
    r = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert r.returncode == 0 and "smoke ok" in r.stdout, (r.stdout[-500:], r.stderr[-2000:])


def test_bench_dump_outputs_is_reproducible(tmp_path):
    """--dump-outputs DIR: the last timed step's loss, updated weights and EMA copy as float32 / float64 .npy files,
    64 MB at most in all, the same arrays from two runs with the same arguments, and other weights after one more timed
    step (the dump is taken after the timed loop, whose length --steps sets)."""
    import numpy as np
    dumps = []
    for run, steps in (("a", 2), ("b", 2), ("c", 3)):
        out = tmp_path / run
        r = subprocess.run([sys.executable, os.path.join(ROOT, "tests", "bench_on_double.py"), "--config", "2", "--size",
                            "32", "--batch", "2", "--steps", str(steps), "--warmup", "1", "--dump-outputs", str(out)],
                           capture_output=True, text=True, timeout=900, cwd=ROOT, env=dict(os.environ, OMP_NUM_THREADS="4"))
        assert r.returncode == 0, r.stderr[-3000:]
        assert json.loads([l for l in r.stdout.splitlines() if l.startswith("{")][0])["steps"] == steps
        dumps.append({p.name: np.load(p) for p in sorted(out.iterdir())})
    a, b, c = dumps
    assert {"loss.npy", "params_netG_A.npy", "ema.npy"} <= set(a) and set(a) == set(b)
    assert sum(v.nbytes for v in a.values()) <= 64 << 20
    for name, v in a.items():
        assert v.dtype in (np.float32, np.float64) and np.isfinite(v).all(), name
        assert np.array_equal(v, b[name]), name
        assert not np.array_equal(v, c[name]), name
