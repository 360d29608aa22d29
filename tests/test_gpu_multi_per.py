"""Multi-GPU check of sharded prioritized updates (tests/multi_gpu_per_check.py under torchrun, 2 ranks); needs >= 2 GPUs on
the box (skipped otherwise)."""
import os
import signal
import subprocess
import sys

import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_sharded_prioritized_updates_agree_across_ranks():
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs at least 2 GPUs")
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr", "127.0.0.1",
           "--master-port", "29553", os.path.join(ROOT, "tests", "multi_gpu_per_check.py")]
    # a session of its own, so that a timeout takes every rank with it
    proc = subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, start_new_session=True)
    try:
        out, err = proc.communicate(timeout=900)
    except subprocess.TimeoutExpired:
        os.killpg(proc.pid, signal.SIGKILL)
        out, err = proc.communicate()
        pytest.fail("timed out\n" + out[-3000:] + err[-3000:])
    assert proc.returncode == 0, out[-3000:] + err[-3000:]
    assert "PER SHARDED OK" in out
