"""``bench.py --impl reference`` (the CPU arm: the oracle port on the host cores) runs without a GPU: its JSON line carries the keys of
the bench contract (metric / unit / value / e2e / cpu_baseline / config.workload ...) and sane values."""
import json
import os
import subprocess
import sys

import numpy as np

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_json_line():
    env = dict(os.environ)
    env.pop("RANK", None); env.pop("WORLD_SIZE", None)
    r = subprocess.run([sys.executable, os.path.join(REPO, "bench.py"), "--impl", "reference", "--steps", "2", "--warmup", "1",
                        "--cpu-min-seconds", "0.5"], cwd=REPO, env=env, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    line = [ln for ln in r.stdout.splitlines() if ln.startswith("{")][-1]
    d = json.loads(line)
    assert d["impl"] == "reference" and d["unit"] == "env.step()/s" and d["higher_is_better"] is True
    assert d["n_gpus"] == 1 and d["gpu_launches"] == 0 and d["dtype"] == "f64"
    assert d["value"] > 1e3 and d["ms_per_step"] > 0
    assert d["e2e"]["value"] == d["value"] and d["e2e"]["h2d_bytes_per_step"] == 0 and d["e2e"]["d2h_bytes_per_step"] == 0
    cb = d["cpu_baseline"]
    assert cb["kind"] == "port" and cb["cores"] >= 1 and cb["value"] == d["value"] and "sample" in cb
    assert "workload" in d["config"] and "model" not in d["config"]
    assert d["spread"]["min"] <= d["spread"]["median"] <= d["spread"]["max"]


def test_reference_arm_steps_and_dumped_outputs(tmp_path):
    """--steps sets the number of timed steps; --dump-outputs writes the last step's results, identical from run to run"""
    env = dict(os.environ)
    env.pop("RANK", None); env.pop("WORLD_SIZE", None)
    dumps = []
    for run in range(2):
        dump = tmp_path / f"run{run}"
        r = subprocess.run([sys.executable, os.path.join(REPO, "bench.py"), "--impl", "reference", "--steps", "3", "--warmup", "1",
                            "--batch", "64", "--dump-outputs", str(dump)], cwd=REPO, env=env, capture_output=True, text=True, timeout=600)
        assert r.returncode == 0, r.stderr[-2000:]
        d = json.loads([ln for ln in r.stdout.splitlines() if ln.startswith("{")][-1])
        assert d["steps"] == 3 and d["spread"]["n"] == 3
        dumps.append({f[:-4]: np.load(dump / f) for f in sorted(os.listdir(dump))})
    a, b = dumps
    assert {"rho", "status", "iterations", "p_or", "a_or", "load_v"} <= set(a)
    for name, x in a.items():
        assert x.dtype == np.float32 and x.shape[0] == 64 and x.size > 0, name
        assert np.array_equal(x, b[name], equal_nan=True), name
    assert (a["status"] == 0).all() and np.isfinite(a["rho"]).all()
