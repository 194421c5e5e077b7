"""GPU: `bench.py --dump-outputs DIR` writes what the last timed step computed (a small DeepFM configuration of the benchmark)."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.mark.gpu
def test_bench_dump_outputs(dev, tmp_path):
    out = tmp_path / "outputs"
    cmd = [sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "3", "--warmup", "1", "--batch", "1024", "--scale-vocab", "0.01",
           "--no-cpu-baseline", "--dump-outputs", str(out)]
    r = subprocess.run(cmd, capture_output=True, text=True, cwd=tmp_path, timeout=900)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-4000:]
    line = json.loads(r.stdout.strip().splitlines()[-1])
    assert line["steps"] == 3
    got = {f[: -len(".npy")]: np.load(out / f) for f in os.listdir(out)}
    assert {"loss", "prob", "fm_w", "fm_w0", "dnn_W0", "dnn_b0", "dnn_W3", "dnn_b3", "table_rows"} <= set(got)
    assert all(a.dtype in (np.float32, np.float64) for a in got.values())
    assert sum(a.nbytes for a in got.values()) <= 64 << 20
    assert got["prob"].shape == (1024,) and np.all((got["prob"] > 0) & (got["prob"] < 1))
    assert got["table_rows"].shape == (26, 1024, 16) and got["dnn_W0"].shape[0] == 13 + 26 * 16 and got["dnn_W3"].shape == (128, 1)
    assert got["loss"].shape == (1,) and 0 < got["loss"][0] < 5
