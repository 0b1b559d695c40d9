"""bench.py's result contract.  CPU: the reference arm (`--impl reference`: the unmodified reference from
baseline/_ref, else the oracle port, timed on the host cores) prints exactly one JSON line with the keys every result
line carries.  GPU: the device arm times exactly --steps steps and writes the last one's result with --dump-outputs."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_one_contract_line():
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup",
                        "0", "--ref-seqs", "1"], capture_output=True, text=True, timeout=900, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.splitlines() if l.strip()]
    assert len(lines) == 1, lines
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["higher_is_better"] is True and d["unit"] == "sequences/s"
    for k in ("metric", "value", "n_gpus", "steps", "warmup", "ms_per_step", "scaling", "vs_baseline", "dtype", "data",
              "config", "cpu_baseline", "e2e"):
        assert k in d, k
    assert d["value"] > 0 and d["steps"] == 1
    has_ref = os.path.isdir(os.path.join(ROOT, "baseline", "_ref", "esm"))
    assert d["cpu_baseline"]["kind"] == ("reference" if has_ref else "port")
    assert d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["sample"]
    assert d["e2e"]["value"] == d["value"] and d["e2e"]["h2d_bytes_per_step"] == 0 and d["e2e"]["d2h_bytes_per_step"] == 0
    assert "workload" in d["config"]


@pytest.mark.gpu
def test_device_arm_dumps_the_last_timed_step(tmp_path):
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "3", "--warmup", "1", "--batch", "4",
                        "--no-extra", "--no-cpu-baseline", "--dump-outputs", str(tmp_path)],
                       capture_output=True, text=True, timeout=900, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.splitlines() if l.strip()]
    assert len(lines) == 1, lines
    d = json.loads(lines[0])
    assert d["steps"] == 3 and d["gpu_launches"] % 3 == 0 and d["value"] > 0
    assert sorted(os.listdir(tmp_path)) == ["mean_representations.npy"]
    mean = np.load(tmp_path / "mean_representations.npy")
    assert mean.dtype == np.float32 and mean.shape == (4, 1280) and np.isfinite(mean).all()
