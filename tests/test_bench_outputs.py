"""``bench.py`` times exactly ``--steps`` steps and ``--dump-outputs`` writes what that region computed, the same
arrays in every run with the same arguments (needs a B200).  Plain SGD: Adam's normalised step turns last-bit
differences of a near-zero gradient (atomic reductions) into learning-rate-sized ones, SGD keeps them last-bit."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _bench(out_dir, steps):
    env = dict(os.environ)
    for k in ("RANK", "WORLD_SIZE", "LOCAL_RANK"):
        env.pop(k, None)
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--steps", str(steps),
                        "--warmup", "3", "--optimizer", "sgd", "--skip-e2e", "--dump-outputs", str(out_dir)],
                       cwd=ROOT, env=env, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
    return json.loads([ln for ln in r.stdout.splitlines() if ln.startswith("{")][-1])


def test_bench_times_steps_and_dumps_reproducible_outputs(tmp_path):
    steps = 7
    recs = [_bench(tmp_path / f"run{i}", steps) for i in range(2)]
    for rec in recs:
        t = rec["timing"]
        assert rec["steps"] == steps and t["regions"] * t["steps_per_region"] == steps
    outs = []
    for i in range(2):
        d = tmp_path / f"run{i}"
        arrays = {n: np.load(d / f"{n}.npy") for n in ("center", "weights", "loss_accuracy")}
        assert sum(os.path.getsize(d / f"{n}.npy") for n in arrays) <= 64 * 2**20
        assert all(a.dtype == np.float32 and np.isfinite(a).all() for a in arrays.values())
        assert arrays["center"].shape == arrays["weights"].shape == (recs[i]["ps_gbs"]["bytes_each_way"] // 4,)
        assert arrays["loss_accuracy"].shape == (steps, 2) and (arrays["loss_accuracy"][:, 0] > 0).all()
        outs.append(arrays)
    for n in outs[0]:
        np.testing.assert_allclose(outs[0][n], outs[1][n], rtol=1e-4, atol=1e-5, err_msg=n)
