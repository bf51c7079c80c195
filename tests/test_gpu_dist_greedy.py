"""GPU: all_pairs_step(..., greedy=True) through the C ABI equals mc2_identity_greedy_clusters on every rank.  World size 1
always; world size 2 over NCCL when the box has two GPUs (tests/multi_gpu_greedy_check.py under torch.distributed.run)."""
import os
import socket
import subprocess
import sys

import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _run(cmd):
    p = subprocess.run(cmd, cwd=ROOT, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, timeout=900)
    assert p.returncode == 0 and " OK " in p.stdout, p.stdout[-3000:]


def test_greedy_step_world1(built_lib):
    _run([sys.executable, "tests/multi_gpu_greedy_check.py", "--n-seqs", "1500"])


def test_greedy_step_world2_nccl(built_lib):
    if built_lib.device_count() < 2:
        pytest.skip("one GPU on this box")
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port_no = s.getsockname()[1]
    s.close()
    _run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr", "127.0.0.1",
          "--master-port", str(port_no), "tests/multi_gpu_greedy_check.py", "--n-seqs", "1501"])
