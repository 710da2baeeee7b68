"""The native arm of bench.py on one GPU: `--steps` is the number of timed steps in the JSON line, and `--dump-outputs`
writes the fit of the last timed step (winner b_best, objective opt, raw weights alpha_raw) -- the fit the line reports."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.mark.gpu
def test_native_arm_dumps_the_last_timed_fit(tmp_path):
    dump = tmp_path / "outputs"
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--steps", "2", "--warmup", "1",
                          "--no-extras", "--no-cpu-baseline", "--dump-outputs", str(dump)],
                         capture_output=True, text=True, timeout=900, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1
    j = json.loads(lines[0])
    assert j["steps"] == 2 and j["n_gpus"] == 1
    assert sorted(os.listdir(dump)) == ["alpha_raw.npy", "b_best.npy", "opt.npy"]
    b, opt, alpha = (np.load(dump / f) for f in ("b_best.npy", "opt.npy", "alpha_raw.npy"))
    assert b.dtype == opt.dtype == alpha.dtype == np.float64
    assert int(b) == j["result"]["b_best"] and float(opt) == j["result"]["opt"]
    assert alpha.shape == (j["config"]["M"] + 1,) and np.all(alpha >= 0) and np.any(alpha > 0)
