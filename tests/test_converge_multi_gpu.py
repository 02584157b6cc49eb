"""Runs tests/converge_multi_gpu_check.py under torchrun when the box has >= 2 GPUs."""
import os
import subprocess
import sys

import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_two_rank_converge(tmp_path):
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs >= 2 GPUs")
    env = dict(os.environ, MMSBM_TMP=str(tmp_path))
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2",
           "--master-addr", "127.0.0.1", "--master-port", "29541",
           os.path.join(ROOT, "tests", "converge_multi_gpu_check.py")]
    res = subprocess.run(cmd, capture_output=True, text=True, timeout=600, env=env, cwd=ROOT)
    assert res.returncode == 0, res.stdout[-3000:] + res.stderr[-3000:]
    assert "converge multi-gpu ok" in res.stdout
