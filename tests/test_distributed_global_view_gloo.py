"""World-size-2 gloo test (CPU) of the host protocol of the global prototype view: every rank all-gathers its task totals
(distributed.gather_task_counts), forms its view from the [world, T] table, accumulates its half of the batch over
that view and adds its sums and counts into the others' with the packed all-reduce.  The merged state must equal the
exact-mode sums and counts of one process fed the concatenation in rank order.  The CUDA kernels are replaced by the
fp64 reference here; only the cross-rank protocol of bacs_b200.distributed is under test."""
import os
import socket
import sys

import numpy as np
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HERE = os.path.dirname(os.path.abspath(__file__))
T, D, B, H, W = 6, 16, 7, 16, 20
BOUNDS = (0, 3, 7)                    # unequal halves


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    return port


def _batch():
    g = torch.Generator().manual_seed(5)
    c = torch.randint(-1, T + 2, (B, H // 4, W // 4), generator=g)
    task = c.repeat_interleave(4, 1).repeat_interleave(4, 2).numpy()
    task = np.where(task >= T, -1, task)
    task[0][task[0] == 1] = -1
    return torch.randn(B, D, H, W, generator=g, dtype=torch.float64), task


def _worker(rank, world, port, out_dir):
    sys.path[:0] = [ROOT, HERE]
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    from proto_view_ref import exact_view_sums
    from bacs_b200.distributed import allreduce_packed, gather_task_counts
    feat, task = _batch()
    lo, hi = BOUNDS[rank], BOUNDS[rank + 1]
    totals = torch.from_numpy(np.stack([(task[lo:hi] == t).sum() for t in range(T)]).astype(np.int64))
    table = gather_task_counts(totals)
    assert table.shape == (world, T)
    view = (table[:rank].sum(0).numpy(), table.sum(0).numpy())
    s, _, n = exact_view_sums(feat[lo:hi], task[lo:hi], T, view)
    packed = torch.zeros(T * D + T, dtype=torch.float64)
    sums, counts = packed[:T * D].view(T, D), packed[T * D:]
    sums.copy_(s)
    counts.copy_(n.double())
    allreduce_packed(sums, counts)
    torch.save({"sums": sums.clone(), "counts": counts.clone(), "table": table}, os.path.join(out_dir, "rank%d.pt" % rank))
    dist.destroy_process_group()


def test_global_view_protocol_matches_single_process(tmp_path):
    world = 2
    mp.spawn(_worker, args=(world, _free_port(), str(tmp_path)), nprocs=world, join=True)
    sys.path[:0] = [ROOT, HERE]
    from proto_view_ref import exact_view_sums
    r = [torch.load(os.path.join(tmp_path, "rank%d.pt" % k)) for k in range(world)]
    assert torch.equal(r[0]["sums"], r[1]["sums"]) and torch.equal(r[0]["counts"], r[1]["counts"])
    assert torch.equal(r[0]["table"], r[1]["table"])
    feat, task = _batch()
    S, A, N = exact_view_sums(feat, task, T)
    assert torch.equal(r[0]["counts"].long(), N)
    assert torch.all((r[0]["sums"] - S).abs() <= 1e-12 * A)
    # the per-channel sums the default N > 1 path would merge are a different computation
    ch = sum(exact_view_sums(feat[b:b + 1], task[b:b + 1], T)[0] for b in range(B))
    assert not torch.allclose(ch, S, rtol=1e-6, atol=1e-6)
