"""Point evaluation and non-matching interpolation over two ranks (needs >= 2 GPUs; skipped on the single-GPU tier):
tests/multigpu_interp_check.py under torchrun."""
import os
import subprocess
import sys

import pytest


@pytest.mark.gpu
def test_two_gpu_eval_interpolate():
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2", "--master-addr", "127.0.0.1",
                        "--master-port", "29637", os.path.join(root, "tests", "multigpu_interp_check.py")], capture_output=True, text=True,
                       timeout=900)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
