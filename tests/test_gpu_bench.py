"""bench.py's GPU arm end to end on a small workload: --steps sets the number of timed steps of both timed loops, and
--dump-outputs writes what the last timed step returned."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_steps_and_dump_outputs(tmp_path):
    out = tmp_path / "outputs"
    env = dict(os.environ, DESC_BENCH_TRACE="1")          # one stderr line per timed step
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--workload", "small", "--steps", "4",
                        "--warmup", "1", "--no-cpu", "--no-side", "--dump-outputs", str(out)],
                       capture_output=True, text=True, timeout=600, env=env, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    j = json.loads(r.stdout.strip().splitlines()[-1])
    assert j["steps"] == 4
    assert r.stderr.count("step step_resident:") == 4 and r.stderr.count("step step_e2e:") == 4
    assert sorted(os.listdir(out)) == ["R_est.npy", "S_vec.npy"]
    S, R = np.load(out / "S_vec.npy"), np.load(out / "R_est.npy")
    n, m = j["config"]["n"], j["config"]["m"]
    assert S.dtype == np.float64 and S.shape == (m,)
    assert R.dtype == np.float64 and R.shape == (3, 3, n)
    assert np.all(np.isfinite(S)) and S.min() >= 0.0 and S.max() <= 1.0 + 1e-12   # convex combinations of d_ijk
    Rt = R.transpose(2, 0, 1)
    np.testing.assert_allclose(Rt @ Rt.transpose(0, 2, 1), np.broadcast_to(np.eye(3), (n, 3, 3)), atol=1e-9)
