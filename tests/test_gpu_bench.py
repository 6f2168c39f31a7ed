"""bench.py at a tiny step count: --steps sets the number of timed steps, --dump-outputs writes the last step's outputs."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_bench_steps_and_dump_outputs(tmp_path):
    out = tmp_path / "dump"
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--steps", "3", "--warmup", "1",
                        "--no-cpu-baseline", "--no-sequence", "--dump-outputs", str(out)],
                       capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stdout[-4000:] + r.stderr[-4000:]
    res = json.loads(r.stdout.strip().splitlines()[-1])
    assert res["steps"] == res["timed_steps"] == 3
    assert res["with_status_err"]["steps"] == res["e2e"]["steps"] == res["e2e_rgb_frames"]["steps"] == 3
    files = sorted(os.listdir(out))
    assert sum(os.path.getsize(out / f) for f in files) <= 64 << 20
    arrs = {f[:-len(".npy")]: np.load(out / f) for f in files}
    assert all(a.dtype in (np.float32, np.float64) for a in arrs.values())
    assert arrs["p1"].shape == (20000, 2) and arrs["fb_dist"].shape == (20000,)
    assert (arrs["fb_dist"] < 1).mean() > 0.99                # the synthetic shift is tracked everywhere
    assert {"level%d" % l for l in range(5)} | {"scharr%d" % l for l in range(5)} <= set(arrs)
