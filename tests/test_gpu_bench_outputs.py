"""GPU: bench.py --dump-outputs writes what the timed path computed in its last step, the same arrays from run to run
with the same seeded inputs, and --steps sets the number of timed steps."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _bench(out_dir, steps):
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", str(steps), "--warmup", "1",
                        "--groups", "24", "--nodes", "1500", "--parity-groups", "6", "--no-alt", "--no-cpu",
                        "--soak", "0", "--dump-outputs", str(out_dir)],
                       cwd=ROOT, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-3000:]
    lines = [ln for ln in r.stdout.splitlines() if ln.startswith("{")]
    assert len(lines) == 1
    return json.loads(lines[0])


def test_dump_outputs_and_steps(tmp_path):
    one, three = _bench(tmp_path / "one", 1), _bench(tmp_path / "three", 3)
    assert one["steps"] == 1 and three["steps"] == 3 and one["parity"]["ok"] and three["parity"]["ok"]
    assert three["gpu_launches"] == 3 * one["gpu_launches"] > 0
    names = sorted(os.listdir(tmp_path / "one"))
    assert names == sorted(os.listdir(tmp_path / "three"))
    assert names == ["assign.npy", "domain.npy", "scores.npy", "scores_cols.npy", "scores_feasible.npy",
                     "scores_rows.npy", "status.npy"]
    assert sum(os.path.getsize(tmp_path / "one" / n) for n in names) <= 64_000_000
    got = {n[:-4]: np.load(tmp_path / "one" / n) for n in names}
    for n, a in got.items():
        assert a.dtype in (np.float32, np.float64) and np.isfinite(a).all(), n
        b = np.load(tmp_path / "three" / f"{n}.npy")
        assert a.dtype == b.dtype and np.array_equal(a.view(np.uint8), b.view(np.uint8)), n
    total_r, groups = one["config"]["replicas_per_step"], one["config"]["groups"]
    assert got["assign"].shape == (total_r,) and got["status"].shape == got["domain"].shape == (groups,)
    assert (got["assign"] >= 0).any()
    # this size fits whole: every row of the dense matrix over every node
    assert got["scores"].shape == got["scores_feasible"].shape == (total_r, one["config"]["nodes"])
    assert np.isin(got["scores_feasible"], (0.0, 1.0)).all() and (got["scores"][got["scores_feasible"] == 0] == 0).all()
    assert np.array_equal(got["scores_rows"], np.arange(total_r)) and np.array_equal(got["scores_cols"], np.arange(one["config"]["nodes"]))
