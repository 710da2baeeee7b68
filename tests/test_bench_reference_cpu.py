"""The reference arm of bench.py (`--impl reference`): the C restatement of the reference's own loop
(src/PartitionedLSOpt.jl:85-94) timed on the host cores, on the default workload's metric / unit / config, without
touching the product library.  Runs here without a GPU (one bounded step)."""
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_the_contract_line(tmp_path):
    dump = tmp_path / "outputs"
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0",
                          "--dump-outputs", str(dump)],
                         capture_output=True, text=True, timeout=600, cwd=ROOT, env=dict(os.environ, LD_DEBUG="libs"))        # the dynamic loader lists every library it maps on stderr
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1
    j = json.loads(lines[0])
    assert j["impl"] == "reference" and j["metric"] == "opt_fit_orthant_nnls_solves_per_sec" and j["unit"] == "nnls_problems/s"
    assert j["higher_is_better"] is True and j["n_gpus"] == 1 and j["steps"] == 1 and j["dtype"] == "f64"
    assert j["config"]["workload"].startswith("k20_m200") and j["config"]["K"] == 20 and j["config"]["M"] == 200
    assert j["value"] > 0 and abs(j["reference_orthants_per_sec"] - 2 * j["value"]) <= 1e-9 * j["value"]
    cb = j["cpu_baseline"]
    assert cb["kind"] == "port" and cb["cores"] >= 1 and cb["value"] == j["value"] and "orthants" in cb["sample"]
    assert j["e2e"] == {"value": j["value"], "unit": j["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert j["gpu_launches"] == 0
    # the arm is the oracle only: the product library is never mapped into that process
    assert "libpls_oracle" in out.stderr and "libpls_cuda" not in out.stderr
    # --dump-outputs: the last timed step's sampled orthants and their objectives, float64
    bl, objs = np.load(dump / "b_list.npy"), np.load(dump / "objs.npy")
    assert sorted(os.listdir(dump)) == ["b_list.npy", "objs.npy"]
    assert bl.dtype == objs.dtype == np.float64 and bl.shape == objs.shape == (cb["cores"],)
    assert np.all(bl == np.round(bl)) and np.all((0 <= bl) & (bl < 2 ** 21)) and np.all(objs > 0)
