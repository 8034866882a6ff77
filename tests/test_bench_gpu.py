"""GPU: `bench.py --dump-outputs` writes the outputs of the last timed step, consistent with the JSON line."""
import json
import subprocess
import sys
from pathlib import Path

import numpy as np
import pytest

ROOT = Path(__file__).resolve().parent.parent
pytestmark = pytest.mark.gpu


def test_dump_outputs(tmp_path):
    sys.path.insert(0, str(ROOT))
    import bench
    out = tmp_path / "dump"
    res = subprocess.run([sys.executable, str(ROOT / "bench.py"), "--steps", "3", "--warmup", "1", "--no-secondary",
                          "--no-cpu-baseline", "--dump-outputs", str(out)],
                         capture_output=True, text=True, timeout=900, cwd=str(tmp_path))
    assert res.returncode == 0, res.stderr[-3000:]
    d = json.loads(res.stdout.strip().splitlines()[-1])
    assert d["steps"] == 3
    paths = sorted(out.iterdir())
    assert [p.name for p in paths] == ["loss.npy", "loss_rows.npy", "pred.npy"]
    assert sum(p.stat().st_size for p in paths) <= 64e6
    loss, loss_rows, pred = (np.load(p) for p in paths)
    assert loss.dtype == loss_rows.dtype == pred.dtype == np.float32
    assert pred.shape == (bench.DUMP_ROWS, 512) and np.isfinite(pred).all() and pred.std() > 0
    assert loss.shape == () and loss_rows.shape == (bench.BATCH,)
    assert np.isclose(float(loss), float(loss_rows.mean()), rtol=1e-5)
    assert round(float(loss), 6) == d["loss"]
