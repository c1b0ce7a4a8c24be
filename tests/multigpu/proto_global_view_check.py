"""Check of the exact-mode prototype update across data-parallel ranks (Prototypes(exact_across_ranks=True)).  Run with
  python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 tests/multigpu/proto_global_view_check.py
with N >= 1 GPUs, with and without BACS_PEER_ALLREDUCE=0 (NCCL all-gather of the counts instead of peer memory).

Every rank holds B = 24 / N images of a VOC-shaped batch (512 x 512 labels, 32 x 32 bf16 features, D = 512).  After
each of three steps the prototypes and counts must be bit-identical across ranks and equal those of one process fed
the whole batch (rank 0's images first) in the exact mode: counts exact, prototypes within 1e-6 relative.  Three more
steps replayed from a CUDA graph must give the same state as three eager steps.  The count exchange on its own must
give view_pre = the totals of the lower ranks and view_n = the totals of all ranks.  Every rank prints
'proto global view ok'."""
import os
import sys

import torch
import torch.distributed as dist

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__)))))

B, D, H, W, h, w, T = 24, 512, 512, 512, 32, 32, 6
INITIAL, INCREMENT = 15, 1                     # VOC 15-1 at its sixth task: classes 1..20


def make_batch(step, dev):
    g = torch.Generator().manual_seed(1000 + step)
    c = torch.randint(0, 21, (B, H // 32, W // 32), generator=g)
    c = torch.where(torch.rand(c.shape, generator=g) > 0.95, torch.full_like(c, 255), c)
    labels = c.repeat_interleave(32, 1).repeat_interleave(32, 2)
    labels[1][labels[1] == 17] = 0             # an image without a pixel of task 2
    feat = torch.randn(B, D, h, w, generator=g).to(torch.bfloat16)
    return feat.to(dev), labels.to(dev)


def make_prototypes(dev, **kw):
    from bacs_b200.loss.prototypes import Prototypes
    P = Prototypes(exact=True, **kw)
    P.set_continual_task_size(INITIAL, INCREMENT)
    g = torch.Generator().manual_seed(7)
    P._prototypes_tensors = torch.randn(T, D, generator=g).to(dev)
    P._count_features = torch.randint(1, 100, (T,), generator=g).to(dev)
    P.refresh_ready()
    return P


def gathered(x, world):
    parts = [torch.empty_like(x) for _ in range(world)]
    dist.all_gather(parts, x)
    return parts


def main():
    rank, local, world = int(os.environ["RANK"]), int(os.environ["LOCAL_RANK"]), int(os.environ["WORLD_SIZE"])
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    dist.init_process_group("nccl", device_id=dev)
    from bacs_b200 import ops
    from bacs_b200.distributed import check_peer_errors, exchange_task_counts, peer_reducer
    peer = os.environ.get("BACS_PEER_ALLREDUCE", "1") != "0"
    lo, hi = rank * B // world, (rank + 1) * B // world

    # the count exchange on its own, against the all-gathered totals
    feat, labels = make_batch(0, dev)
    P = make_prototypes(dev, exact_across_ranks=True)
    lut = P._device_task_lut(dev, T)
    _, _, n_bt, _ = ops.label_downsample_task(labels[lo:hi].contiguous(), h, w, lut, T)
    red = peer_reducer(T * D + T, dev)
    assert (red is not None) == peer, "symmetric memory unavailable" if peer else "peer reducer not disabled"
    vp, vn = exchange_task_counts(n_bt, red)
    table = torch.stack(gathered(n_bt.long().sum(0), world))
    assert torch.equal(vp, table[:rank].sum(0)) and torch.equal(vn, table.sum(0)), (rank, vp, vn, table)

    # three eager steps against one process fed the whole batch
    R = make_prototypes(dev, sync_across_ranks=False)
    for step in range(3):
        feat, labels = make_batch(step, dev)
        P.update_feats_prototypes(feat[lo:hi].contiguous(), labels[lo:hi].contiguous())
        R.update_feats_prototypes(feat, labels)
        torch.cuda.synchronize()
        check_peer_errors()
        for x in (P._prototypes_tensors, P._count_features, P.ready_flag):
            assert all(torch.equal(x, y) for y in gathered(x, world)), (rank, step, "ranks differ")
        assert torch.equal(P._count_features, R._count_features), (rank, step)
        ref = R._prototypes_tensors
        err = float(((P._prototypes_tensors - ref).abs() / ref.abs().clamp_min(1e-30)).max())
        assert err <= 1e-6, (rank, step, err)
        assert int(P.ready_flag) == int(R.ready_flag)

    # three graph replays against three eager steps from the same state
    feat, labels = make_batch(3, dev)
    x, y = feat[lo:hi].contiguous(), labels[lo:hi].contiguous()
    E = make_prototypes(dev, exact_across_ranks=True)
    E._prototypes_tensors.copy_(P._prototypes_tensors)
    E._count_features.copy_(P._count_features)
    for _ in range(3):
        E.update_feats_prototypes(x, y)
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    p0, c0 = P._prototypes_tensors.clone(), P._count_features.clone()
    with torch.cuda.stream(side):
        P.update_feats_prototypes(x, y)                       # warm-up outside the capture
    torch.cuda.current_stream().wait_stream(side)
    torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        P.update_feats_prototypes(x, y)
    P._prototypes_tensors.copy_(p0)
    P._count_features.copy_(c0)
    for _ in range(3):
        graph.replay()
    torch.cuda.synchronize()
    check_peer_errors()
    assert torch.equal(P._prototypes_tensors, E._prototypes_tensors), rank
    assert torch.equal(P._count_features, E._count_features), rank
    print("rank %d: proto global view ok (world %d, %s)" % (rank, world, "peer memory" if peer else "NCCL"), flush=True)
    dist.barrier()
    os._exit(0)


if __name__ == "__main__":
    main()
