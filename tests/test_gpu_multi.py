"""Multi-GPU paths that need more than one device (skipped on a single-GPU box): launched as one rank per GPU over NCCL."""
import os
import subprocess
import sys
import pytest

pytestmark = pytest.mark.gpu


def test_sharded_proof_and_two_devices_in_one_process(tmp_path):
    import torch
    n = torch.cuda.device_count()
    if n < 2:
        pytest.skip("needs >= 2 GPUs")
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr", "127.0.0.1", "--master-port", "29731",
           os.path.join(root, "tests", "multi_gpu_worker.py")]
    out = subprocess.run(cmd, capture_output=True, text=True, timeout=900)
    (tmp_path / "multi_gpu_worker.log").write_text(out.stdout + "\n---- stderr ----\n" + out.stderr)
    assert out.returncode == 0 and "multi-gpu ok" in out.stdout, out.stdout[-2000:] + out.stderr[-4000:]
