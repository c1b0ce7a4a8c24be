"""Exact-mode prototypes across data-parallel ranks (tests/multigpu/proto_global_view_check.py): two ranks with half of a
B = 24 VOC-shaped batch each must end with bit-identical prototypes and counts equal to one process's exact-mode update
on the whole batch, over peer memory and over NCCL, eagerly and from a CUDA graph.  With one rank the same script
checks the count exchange of both transports against the all-gathered totals on any GPU."""
import os
import subprocess
import sys

import pytest
import torch

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _run(nproc, port, peer):
    env = dict(os.environ, BACS_PEER_ALLREDUCE="1" if peer else "0")
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", str(nproc),
           "--master-addr", "127.0.0.1", "--master-port", str(port),
           os.path.join(ROOT, "tests", "multigpu", "proto_global_view_check.py")]
    out = subprocess.run(cmd, capture_output=True, text=True, timeout=600, cwd=ROOT, env=env)
    assert out.returncode == 0, out.stdout[-2000:] + out.stderr[-3000:]
    assert out.stdout.count("proto global view ok") == nproc, out.stdout[-2000:]


@pytest.mark.skipif(not torch.cuda.is_available() or torch.cuda.device_count() < 2, reason="needs >= 2 GPUs")
@pytest.mark.parametrize("peer", [True, False], ids=["peer", "nccl"])
def test_two_ranks_equal_one_process(peer):
    _run(2, 29561 + int(peer), peer)


@pytest.mark.skipif(not torch.cuda.is_available(), reason="needs a GPU")
@pytest.mark.parametrize("peer", [True, False], ids=["peer", "nccl"])
def test_single_rank(peer):
    _run(1, 29563 + int(peer), peer)
