"""The same-box comparator: ``bench.py --impl reference`` drives the UNMODIFIED reference package (``baseline/_ref``)
through its own public API on stand-in Keras / Spark modules (``baseline/shims``).  Skipped when the offline install is
absent (``baseline/_ref`` is git-ignored)."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.mark.skipif(not os.path.isdir(os.path.join(ROOT, "baseline", "_ref", "distkeras")),
                    reason="reference package not installed under baseline/_ref")
def test_reference_arm_runs_the_unmodified_package():
    env = dict(os.environ, CUDA_VISIBLE_DEVICES="")
    for k in ("RANK", "WORLD_SIZE", "LOCAL_RANK"):
        env.pop(k, None)
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "5", "--warmup", "3"],
                       cwd=ROOT, env=env, capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stderr[-2000:]
    rec = json.loads([ln for ln in r.stdout.splitlines() if ln.startswith("{")][-1])
    assert rec["impl"] == "reference" and rec["value"] > 0 and rec["unit"] == "samples/s"
    assert rec["config"]["trainer"] == "ADAG" and rec["config"]["batch_per_worker"] == 64
    # nothing of this repository is on that path: the package under test is the reference's own
    import importlib.util

    spec = importlib.util.spec_from_file_location("ref_trainers", os.path.join(ROOT, "baseline", "_ref", "distkeras", "trainers.py"))
    assert spec is not None
    src = open(os.path.join(ROOT, "baseline", "_ref", "distkeras", "trainers.py")).read()
    assert "distkeras_b200" not in src


def test_adag_matches_recorded_reference_run():
    """``tests/golden/reference_arm_adag_mnist_mlp.json`` is what ``bench.py --impl reference --steps 5 --warmup 3``
    printed when the unmodified reference ran (CPU, one worker).  The same job through this package's ADAG must do
    the same bookkeeping: W + K steps recorded per worker and the reference's update counter (starts at 1, one
    increment per committed window)."""
    import torch

    import bench
    from distkeras_b200 import trainers
    from distkeras_b200.data import Dataset
    from distkeras_b200.models import ZOO

    rec = json.load(open(os.path.join(ROOT, "tests", "golden", "reference_arm_adag_mnist_mlp.json")))
    assert rec["impl"] == "reference" and rec["value"] > 0 and rec["unit"] == "samples/s"
    cfg = rec["config"]
    assert cfg["trainer"] == "ADAG" and cfg["batch_per_worker"] == bench.DEFAULT_BATCH[cfg["model"]] == 64
    assert cfg["communication_window"] == bench.DEFAULT_WINDOW["adag"]
    B, tau, steps = cfg["batch_per_worker"], cfg["communication_window"], rec["warmup"] + rec["steps"]
    g = torch.Generator().manual_seed(0)
    x = torch.rand(steps * B, *bench.IN_SHAPE[cfg["model"]], generator=g)
    y = torch.randint(0, 10, (steps * B,), generator=g).to(torch.int32)
    t = trainers.ADAG(ZOO[cfg["model"]](seed=0), cfg["worker_optimizer"], "categorical_crossentropy",
                      num_workers=cfg["num_workers"], batch_size=B, communication_window=tau)
    t.backend = "thread"
    t.train(Dataset({"features": x, "label": y}))
    per_worker = {}
    for h in t.get_history():
        per_worker[h["worker_id"]] = per_worker.get(h["worker_id"], 0) + 1
    assert sorted(per_worker.values()) == rec["steps_done_per_worker"]
    assert t.num_updates() == rec["num_updates"] == 1 + steps // tau


def test_shims_live_outside_the_reference_package():
    shims = os.path.join(ROOT, "baseline", "shims")
    assert {"keras", "pyspark", "tensorflow"} <= set(os.listdir(shims))
