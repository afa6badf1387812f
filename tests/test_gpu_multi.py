"""Multi-GPU parity: spawns tests/multi_gpu_check.py on 2 GPUs (NCCL) when the machine has them."""
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.mark.gpu
def test_two_gpu_slabs_equal_the_single_domain_oracle(tmp_path):
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs (the one-GPU two-slab emulation is in test_gpu_parity.py)")
    env = dict(os.environ, MASTER_ADDR="127.0.0.1")
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr", "127.0.0.1",
           "--master-port", "29917", os.path.join(ROOT, "tests", "multi_gpu_check.py")]
    r = subprocess.run(cmd, cwd=ROOT, env=env, capture_output=True, text=True, timeout=900)
    log = r.stdout + r.stderr
    (tmp_path / "multi_gpu_check.log").write_text(log)
    assert r.returncode == 0, log[-4000:]
    assert "MULTI_GPU_CHECK_OK" in log, log[-4000:]
