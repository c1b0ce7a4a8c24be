"""The peer-memory all-reduce fused with the prototype update (csrc/peer.cu) at 65 and 128 tasks, against NCCL and the
stand-alone update, bit-exact: with two ranks where two GPUs exist, and with one rank on any GPU (the update kernel and
the reducer size of runs with more than 64 tasks)."""
import os
import subprocess
import sys

import pytest
import torch

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _run(nproc, port):
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", str(nproc),
           "--master-addr", "127.0.0.1", "--master-port", str(port),
           os.path.join(ROOT, "tests", "multigpu", "peer_allreduce_many_check.py")]
    out = subprocess.run(cmd, capture_output=True, text=True, timeout=300, cwd=ROOT)
    assert out.returncode == 0, out.stdout[-2000:] + out.stderr[-2000:]
    assert out.stdout.count("peer all-reduce many ok") == nproc, out.stdout[-2000:]


@pytest.mark.skipif(not torch.cuda.is_available() or torch.cuda.device_count() < 2, reason="needs >= 2 GPUs")
def test_peer_allreduce_128_tasks_matches_nccl():
    _run(2, 29551)


@pytest.mark.skipif(not torch.cuda.is_available(), reason="needs a GPU")
def test_peer_allreduce_128_tasks_single_rank():
    _run(1, 29552)
