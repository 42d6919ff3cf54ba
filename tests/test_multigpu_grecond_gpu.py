"""GPU, >= 2 devices: GreConD on rows sharded over 2 ranks (NCCL) gives every rank the world-1 factors, including a case
where rank 1 holds no rows (skipped on 1-GPU boxes)."""
import os
import socket
import subprocess
import sys

import pytest

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_sharded_grecond_two_gpus_nccl():
    if torch.cuda.device_count() < 2:
        pytest.skip("needs at least 2 GPUs")
    s = socket.socket(); s.bind(("127.0.0.1", 0)); port = s.getsockname()[1]; s.close()
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr", "127.0.0.1",
           "--master-port", str(port), os.path.join(ROOT, "tests", "multi_gpu_grecond_worker.py")]
    out = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, timeout=900, cwd=ROOT)
    assert out.returncode == 0, out.stdout[-4000:]
    assert "rank 0 of 2 ok" in out.stdout and "rank 1 of 2 ok" in out.stdout
