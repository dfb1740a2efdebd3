"""bench.py on the device at a small size: --steps sets the number of timed steps, and --dump-outputs writes what the timed path
returned in its last step, the same from run to run since the inputs are seeded."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
pytestmark = pytest.mark.gpu


def _bench(steps, out_dir, n, m):
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--kkt-n", str(n), "--kkt-m", str(m), "--steps", str(steps), "--warmup", "1",
                        "--no-e2e", "--no-cpu", "--dump-outputs", str(out_dir)], capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert p.returncode == 0, p.stderr[-2000:]
    lines = [ln for ln in p.stdout.splitlines() if ln.startswith("{")]
    assert len(lines) == 1
    return json.loads(lines[0]), {k: np.load(os.path.join(out_dir, k + ".npy")) for k in ("dx", "dyc", "dyd")}


def test_steps_and_dumped_outputs(tmp_path):
    n, m = 20000, 40
    d2, out2 = _bench(2, tmp_path / "a", n, m)
    d4, out4 = _bench(4, tmp_path / "b", n, m)
    assert d2["steps"] == 2 and d4["steps"] == 4
    assert d4["gpu_launches"] == 2 * d2["gpu_launches"] > 0                   # every step is one KKT system's launches
    for out in (out2, out4):
        assert out["dx"].shape == (n,) and out["dyc"].shape == (m - m // 2,) and out["dyd"].shape == (m // 2,)
        assert all(a.dtype == np.float64 and np.isfinite(a).all() and np.abs(a).max() > 0 for a in out.values())
    for k in out2:
        assert np.abs(out2[k] - out4[k]).max() <= 1e-10 * np.abs(out4[k]).max(), k
