"""GPU: bench.py's timed path - --steps sets the number of timed steps, and --dump-outputs writes the last step's
outputs (a fixed, seeded sample of the frame's rays, at most 64 MB) identically from run to run."""
import json
import subprocess
import sys
from pathlib import Path

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
ROOT = Path(__file__).resolve().parent.parent


def _bench(*args):
    p = subprocess.run([sys.executable, "bench.py", "--gpus", "1", "--no-cpu-baseline", "--no-extra", "--no-fast-mode",
                        *args], cwd=ROOT, capture_output=True, text=True, timeout=600)
    assert p.returncode == 0, p.stderr[-3000:]
    lines = [l for l in p.stdout.splitlines() if l.strip()]
    assert len(lines) == 1, p.stdout[:500]
    return json.loads(lines[0])


def test_steps_and_dumped_outputs(tmp_path):
    runs = []
    for i, steps in enumerate((2, 3)):
        d = _bench("--steps", str(steps), "--warmup", "1", "--dump-outputs", str(tmp_path / str(i)))
        assert d["steps"] == steps and len(d["config"]["step_ms"]) == steps
        runs.append({p.name: np.load(p) for p in sorted((tmp_path / str(i)).glob("*.npy"))})
    assert sum(p.stat().st_size for p in (tmp_path / "0").iterdir()) <= 64 << 20
    assert {"rgb_map.npy", "depth_map.npy", "acc_map.npy", "weights.npy", "z_vals.npy"} <= set(runs[0])
    assert runs[0].keys() == runs[1].keys()
    rows = runs[0]["rgb_map.npy"].shape[0]
    assert 0 < rows < 376 * 1408            # the cfg2 frame's outputs exceed 64 MB: a sample of its rays
    for name, a in runs[0].items():
        assert a.dtype in (np.float32, np.float64) and a.shape[0] == rows, name
        assert np.array_equal(a, runs[1][name], equal_nan=True), name
    assert np.isfinite(runs[0]["rgb_map.npy"]).all()
