"""bench.py contract, the part that runs without a GPU: the reference arm prints ONE JSON line with the
keys the driver reads (metric / unit / value / e2e / cpu_baseline / impl), on the same workload
description as the GPU arm."""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_one_json_line():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1",
                          "--warmup", "1"], capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.strip().splitlines() if l.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "svi_steps_per_sec" and d["unit"] == "steps/s"
    assert d["higher_is_better"] is True and d["value"] > 0 and d["n_gpus"] == 1
    assert d["config"]["workload"].startswith("bayesian_logistic_regression_svi N=1e6 D=32")
    # unmodified Pyro when oracle/_ref is vendored, else the oracle port
    assert d["cpu_baseline"]["kind"] == "reference" or d["cpu_baseline"]["kind"].startswith("port")
    assert d["cpu_baseline"]["cores"] >= 1
    if os.path.isdir(os.path.join(ROOT, "oracle", "_ref", "pyro")):
        assert d["cpu_baseline"]["kind"] == "reference" and "unmodified Pyro" in d["cpu_baseline"]["sample"]
    assert d["e2e"] == {"value": d["value"], "unit": "steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}


def test_reference_arm_other_ranks_exit_quietly():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2"],
                         capture_output=True, text=True, timeout=120, cwd=ROOT, env=env)
    assert out.returncode == 0 and out.stdout.strip() == ""
