"""bench.py --dump-outputs on the GPU: two runs with the same arguments write the same arrays (the inputs are seeded and the timed
region is exactly --steps steps), all float32 / float64 and within 64 MB."""
import glob
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
pytestmark = pytest.mark.gpu


def _bench(out_dir, steps):
    cmd = [sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--config", "askubuntu", "--steps", str(steps), "--warmup", "2",
           "--no-cpu-baseline", "--dump-outputs", str(out_dir)]
    r = subprocess.run(cmd, cwd=str(out_dir.parent), capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
    line = json.loads([l for l in r.stdout.splitlines() if l.startswith("{")][-1])
    assert line["steps"] == line["timing"]["timed_steps"] == steps
    return {os.path.basename(p)[:-4]: np.load(p) for p in sorted(glob.glob(os.path.join(str(out_dir), "*.npy")))}


def test_dump_outputs_repeat_across_runs(tmp_path):
    a = _bench(tmp_path / "a", 3)
    b = _bench(tmp_path / "b", 3)
    assert sorted(a) == sorted(b)
    assert {"loss_g_loss", "loss_d_loss", "gen_W_q0", "gen_W_p1", "disc_w1", "disc_b4"} <= set(a)
    assert sum(x.nbytes for x in a.values()) <= 64 << 20
    assert a["gen_W_q0"].shape == (1000, 600) and a["gen_W_p1"].shape == (600, 1000)   # a catalog below DUMP_ROWS is kept whole
    for k in a:
        assert a[k].dtype in (np.float32, np.float64) and np.isfinite(a[k]).all(), k
        assert np.allclose(a[k], b[k], rtol=1e-3, atol=1e-5), (k, float(np.abs(a[k] - b[k]).max()))
    assert float(a["loss_cnt"]) > 0
