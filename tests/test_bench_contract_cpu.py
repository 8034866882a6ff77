"""CPU: bench.py's reference arm (the only bench leg that runs without a GPU) prints the contracted JSON line."""
import json
import subprocess
import sys
from pathlib import Path

import pytest

ROOT = Path(__file__).resolve().parent.parent


def test_reference_arm_json_contract():
    res = subprocess.run([sys.executable, str(ROOT / "bench.py"), "--impl", "reference", "--steps", "2", "--warmup", "1",
                          "--ref-max-batch", "2"],
                         capture_output=True, text=True, timeout=900, cwd=str(ROOT))
    assert res.returncode == 0, res.stderr[-2000:]
    line = [l for l in res.stdout.splitlines() if l.startswith("{")][-1]
    d = json.loads(line)
    assert d["impl"] == "reference" and d["metric"] == "denoiser-steps/sec" and d["unit"] == "steps/s"
    assert d["higher_is_better"] is True and d["value"] > 0
    # oracle/_ref (the pip-installed reference) when present, else the oracle port
    from oracle import reference
    expect_kind = "reference" if reference.installed() else "port"
    assert d["cpu_baseline"]["kind"] == expect_kind
    assert d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["value"] == d["value"]
    assert d["steps"] == 2 and d["sample_batch"] == 2 and d["extrapolated"] is True
    assert d["e2e"] == {"value": d["value"], "unit": "steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert "configs[1]" in d["config"]["workload"]
    sys.path.insert(0, str(ROOT))
    import bench
    assert d["config"] == bench.build_config(1)   # both arms print the same config object


@pytest.mark.parametrize("argv", [["--steps", "0"], ["--impl", "reference", "--dump-outputs", "out"]])
def test_rejected_arguments(argv, tmp_path):
    res = subprocess.run([sys.executable, str(ROOT / "bench.py"), *argv], capture_output=True, text=True, timeout=120,
                         cwd=str(tmp_path))
    assert res.returncode == 2 and res.stdout == "" and "error" in res.stderr
    assert not (tmp_path / "out").exists()


def test_reference_arm_other_ranks_exit_quietly():
    import os
    env = dict(os.environ, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1")
    res = subprocess.run([sys.executable, str(ROOT / "bench.py"), "--impl", "reference", "--gpus", "2"],
                         capture_output=True, text=True, timeout=120, cwd=str(ROOT), env=env)
    assert res.returncode == 0 and res.stdout.strip() == ""
