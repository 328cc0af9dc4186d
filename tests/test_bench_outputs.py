"""bench.py --steps K --dump-outputs DIR: the predictions of the last timed step are written, are the same from run to
run with the same arguments, and are the oracle's predictions for that step's input set (step k reads set k % n_sets)."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from oracle import oracle as orc

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _bench(out_dir, steps, args):
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", str(steps), "--warmup", "2",
                        "--dump-outputs", str(out_dir)] + args, capture_output=True, text=True, timeout=600)
    assert p.returncode == 0, p.stderr[-3000:]
    line = json.loads(p.stdout.strip().splitlines()[-1])
    assert line["steps"] == steps
    return np.load(os.path.join(str(out_dir), "forest_predictions.npy"))


def _oracle_last_step(steps, n_sets):
    forest = orc.synth_xgb_forest(n_trees=1000, depth=6, n_features=32, seed=0)
    X = np.random.default_rng(1).standard_normal((n_sets, 64, 32)).astype(np.float32)
    return orc.forest_predict_xgb(forest, X[(steps - 1) % n_sets], 0.5)


def _check(tmp_path, steps, n_sets, args):
    a = _bench(tmp_path / "a", steps, args)
    b = _bench(tmp_path / "b", steps, args)
    assert a.dtype == np.float32 and a.shape == (64,)
    assert np.array_equal(a, b)
    assert np.array_equal(a, _oracle_last_step(steps, n_sets))


def test_reference_arm_dumps_last_step(tmp_path):
    _check(tmp_path, 70, 256, ["--impl", "reference"])


@pytest.mark.gpu
def test_b200_arm_dumps_last_step(gpu_native, tmp_path):
    _check(tmp_path, 70, 64, ["--no-plugin", "--no-ref-path", "--no-bert", "--no-resnet", "--no-llama", "--cpu-seconds", "1"])
