"""bench.py --dump-outputs: the last timed step's results of the GPU arm as float .npy files, the same from run to run, so
that two builds of the project can be compared output for output."""
import json
import subprocess
import sys
from pathlib import Path

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
ROOT = Path(__file__).resolve().parent.parent


def _bench_dump(out_dir, steps):
    out = subprocess.run([sys.executable, str(ROOT / "bench.py"), "--gpus", "1", "--steps", str(steps), "--warmup", "1", "--headline-only",
                          "--no-cpu-baseline", "--batch", "2", "--events", "20000", "--dump-outputs", str(out_dir)],
                         capture_output=True, text=True, timeout=900)
    assert out.returncode == 0, out.stderr[-2000:]
    assert json.loads(out.stdout.splitlines()[-1])["steps"] == steps
    return {p.stem: np.load(p) for p in sorted(out_dir.glob("*.npy"))}


def test_dump_outputs_reproducible(tmp_path):
    a = _bench_dump(tmp_path / "a", 4)
    b = _bench_dump(tmp_path / "b", 4)
    assert set(a) == {"decoded", "detections", "num_detections"}
    assert sum(v.nbytes for v in a.values()) <= 64 << 20
    for k in a:
        assert a[k].dtype in (np.float32, np.float64), (k, a[k].dtype)
        assert np.array_equal(a[k], b[k]), f"{k} differs between two runs with the same arguments"
    dec, det, n = a["decoded"], a["detections"], a["num_detections"].astype(np.int64)
    assert dec.shape[0] == det.shape[0] == len(n) == 2 and det.shape[2] == 6 and np.isfinite(dec).all()
    for i in range(2):
        assert 0 <= n[i] <= det.shape[1] and not det[i, n[i]:].any()
