"""End-to-end drop-in topology on a GPU box: forked CPU actors + forked stager + CUDA learner in the main process."""
import os
import subprocess
import sys

import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_train_pipeline_runs_to_completion():
    cmd = [sys.executable, os.path.join(ROOT, "examples", "train.py"), "--synthetic-env", "--actors", "2", "--training-steps", "6",
           "--learning-starts", "400", "--buffer-capacity", "3200", "--batch-size", "8", "--log-interval", "2",
           "--save-interval", "1000000"]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=600, cwd=ROOT)
    tail = (r.stdout + r.stderr)[-3000:]
    assert r.returncode == 0, tail
    assert "done: 6 updates" in r.stdout, tail
    assert "number of training steps:" in r.stdout and "buffer size:" in r.stdout, tail


def test_train_pipeline_with_batched_gpu_actors():
    """same topology with all actors behind one batched GPU inference process (worker.VectorActor, --gpu-actors)"""
    cmd = [sys.executable, os.path.join(ROOT, "examples", "train.py"), "--synthetic-env", "--actors", "4", "--gpu-actors", "--training-steps", "6",
           "--learning-starts", "400", "--buffer-capacity", "3200", "--batch-size", "8", "--log-interval", "2",
           "--save-interval", "1000000"]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=600, cwd=ROOT)
    tail = (r.stdout + r.stderr)[-3000:]
    assert r.returncode == 0, tail
    assert "done: 6 updates" in r.stdout, tail
