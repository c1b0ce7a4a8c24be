"""Check of the peer-memory all-reduce fused with the prototype update (csrc/peer.cu) for runs with more than 64 tasks,
against NCCL.  Run with
  python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 tests/multigpu/peer_allreduce_many_check.py
with N >= 1 GPUs.  The reducer is the one distributed.peer_reducer caches (sized for 128 tasks x 2048 channels); the
state is 128 x 2048 (the largest it takes) and 65 x 512 (the smallest count served by the 128-task update kernel).
Every rank prints 'peer all-reduce many ok'."""
import os
import sys

import torch
import torch.distributed as dist

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__)))))


def main():
    rank, local, world = int(os.environ["RANK"]), int(os.environ["LOCAL_RANK"]), int(os.environ["WORLD_SIZE"])
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    dist.init_process_group("nccl", device_id=dev)
    from bacs_b200 import ops
    from bacs_b200.distributed import peer_reducer
    for T, D in ((128, 2048), (65, 512)):
        n = T * D + T
        red = peer_reducer(n, dev)
        assert red is not None, "symmetric memory unavailable"
        assert red.n_max >= 128 * 2048 + 128
        g = torch.Generator(device=dev).manual_seed(200 + rank + T)
        proto = torch.randn(T, D, device=dev, generator=g)
        proto_ref = proto.clone()
        for count_dtype in (torch.int64, torch.float32):
            count = torch.full((T,), 1000, dtype=count_dtype, device=dev)
            empty = count_dtype == torch.float32                    # the last task: no count yet and no pixels
            if empty:
                count[T - 1] = 0
            count_ref = count.clone()
            for step in range(3):
                packed = torch.randn(n, dtype=torch.float64, device=dev, generator=g)
                packed[T * D:] = torch.randint(0, 50, (T,), device=dev, generator=g).double()
                if empty:
                    packed[T * D + T - 1] = 0
                if rank == 0:
                    packed[T * D + 1] = 0                           # a task without pixels on this rank
                want = packed.clone()
                dist.all_reduce(want)
                parts = [torch.empty_like(packed) for _ in range(world)]
                dist.all_gather(parts, packed)
                exact = parts[0].clone()                            # the sum in rank order, the same on every rank
                for p in parts[1:]:
                    exact += p
                ready = red.allreduce(packed, proto, count, T, D)
                torch.cuda.synchronize()
                assert int(red.error) == 0, "a peer timed out"
                assert torch.equal(packed, exact), (rank, T, step, float((packed - exact).abs().max()))
                assert torch.allclose(packed, want, rtol=1e-12, atol=1e-12)
                ready_ref = ops.proto_update(proto_ref, count_ref, exact[:T * D].view(T, D), exact[T * D:])
                assert torch.equal(proto, proto_ref), (rank, T, step)
                assert torch.equal(count, count_ref), (rank, T, step)
                assert int(ready) == int(ready_ref) == (0 if empty else 1), (int(ready), int(ready_ref))
    print("rank %d: peer all-reduce many ok (world %d)" % (rank, world), flush=True)
    torch.cuda.synchronize()
    dist.barrier()
    os._exit(0)


if __name__ == "__main__":
    main()
