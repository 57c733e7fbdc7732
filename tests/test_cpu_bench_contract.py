"""CPU tier: the driver-facing contract of bench.py that can be exercised without a GPU - the reference arm
(`--impl reference`, the in-repo oracle on the host cores): exactly one JSON line on stdout with the agreed keys,
alone and under torchrun (rank 0 prints, the other ranks exit 0 silently)."""
import json
import subprocess
import sys
from pathlib import Path

ROOT = Path(__file__).resolve().parent.parent
KEYS = {"impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
        "vs_baseline", "dtype", "data", "config", "cpu_baseline", "e2e"}


def _run(cmd):
    p = subprocess.run(cmd, cwd=ROOT, capture_output=True, text=True, timeout=900)
    assert p.returncode == 0, p.stderr[-2000:]
    lines = [l for l in p.stdout.splitlines() if l.strip()]
    assert len(lines) == 1, f"stdout must be one JSON line, got {len(lines)}: {p.stdout[:500]}"
    return json.loads(lines[0])


def _check(d, n_gpus):
    assert KEYS <= set(d), KEYS - set(d)
    assert d["impl"] == "reference" and d["n_gpus"] == n_gpus and d["unit"] == "rays/s"
    assert d["value"] > 0 and d["higher_is_better"] is True and d["vs_baseline"] is None
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["value"] == d["value"]
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert "workload" in d["config"]


def test_reference_arm_prints_one_json_line():
    _check(_run([sys.executable, "bench.py", "--impl", "reference", "--steps", "1", "--warmup", "1", "--ref-rows", "1"]), 1)


def _free_port() -> int:
    import socket
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def test_reference_arm_under_torchrun_only_rank0_reports():
    d = _run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2",
              "--master-addr", "127.0.0.1", "--master-port", str(_free_port()), "bench.py", "--impl", "reference",
              "--gpus", "2", "--steps", "1", "--warmup", "1", "--ref-rows", "1"])
    _check(d, 2)


def test_reference_arm_dumps_the_same_outputs_every_run(tmp_path):
    """--dump-outputs DIR: the last step's outputs as float32 / float64 .npy files, identical from run to run."""
    import numpy as np
    runs = []
    for i in range(2):
        d = tmp_path / str(i)
        _check(_run([sys.executable, "bench.py", "--impl", "reference", "--steps", "1", "--warmup", "1", "--ref-rows", "1",
                     "--dump-outputs", str(d)]), 1)
        runs.append({p.name: np.load(p) for p in sorted(d.glob("*.npy"))})
    assert {"rgb_map.npy", "depth_map.npy", "acc_map.npy", "weights.npy"} <= set(runs[0]) and runs[0].keys() == runs[1].keys()
    for name, a in runs[0].items():
        assert a.dtype in (np.float32, np.float64), name
        assert np.array_equal(a, runs[1][name], equal_nan=True), name
