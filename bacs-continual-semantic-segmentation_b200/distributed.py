"""Cross-rank state of the BACS loss path: ONE packed fp64 all-reduce per step.

The reference never synchronises prototypes (each DDP rank keeps its own copy,
loss/prototypes.py:157-163) and lets torchmetrics all_gather the confusion matrix.  Here
each rank's per-task feature sums [T,D], pixel counts [T] and (at evaluation) the K x K
confusion matrix travel in one contiguous fp64 buffer -- integer counts stay exact below
2^53 -- through a single NCCL all-reduce over NVLink / NVSwitch, after which every rank
applies the identical running-mean update.  The payload is a few tens of KB, i.e.
latency-bound; there is no data-path collective anywhere else on this path."""
from __future__ import annotations

from typing import Optional

import torch
import torch.distributed as dist


def world_size() -> int:
    return dist.get_world_size() if dist.is_available() and dist.is_initialized() else 1


def allreduce_packed(sums: torch.Tensor, counts: torch.Tensor, group=None) -> None:
    """``sums`` [T,D] and ``counts`` [T] must be views of one contiguous fp64 buffer laid
    out [T*D | T] (ops.proto_accumulate allocates them that way): one collective moves both."""
    if world_size() == 1:
        return
    base = sums.untyped_storage().data_ptr()
    contiguous = (sums.dtype == torch.float64 and counts.dtype == torch.float64
                  and counts.data_ptr() == sums.data_ptr() + sums.numel() * 8
                  and sums.untyped_storage().data_ptr() == counts.untyped_storage().data_ptr() == base)
    if contiguous:
        packed = torch.empty(0, dtype=torch.float64, device=sums.device).set_(
            sums.untyped_storage(), sums.storage_offset(), (sums.numel() + counts.numel(),))
        dist.all_reduce(packed, op=dist.ReduceOp.SUM, group=group)
    else:
        packed = torch.cat([sums.reshape(-1), counts.reshape(-1)])
        dist.all_reduce(packed, op=dist.ReduceOp.SUM, group=group)
        sums.copy_(packed[:sums.numel()].view_as(sums))
        counts.copy_(packed[sums.numel():])


class PeerReducer:
    """One-shot all-reduce over NVLink peer memory, fused with the prototype update (csrc/peer.cu).

    The symmetric buffer (two step-parity slots of ``n_max`` doubles, one flag row, and the count table of the
    global prototype view: two step-parity slots of ``world`` x 128 int64) is allocated with
    ``torch.distributed._symmetric_memory`` and exchanged once; afterwards a step is ONE kernel launch with no
    host synchronisation, capturable in a CUDA graph.  ``create`` returns None when symmetric memory is not
    available for the group (the caller then uses the packed NCCL all-reduce)."""

    FLAG_DOUBLES = 32                      # 64 uint32 flags: 0..15 the sums phase, 32..47 the count phase
    COUNT_FLAG_OFFSET = 32                 # first uint32 of the count phase's flags

    def __init__(self, n_max: int, device: torch.device, group=None):
        import ctypes as C
        import torch.distributed._symmetric_memory as symm
        group = group or dist.group.WORLD
        self.n_max, self.device = int(n_max), device
        self.rank, self.world = dist.get_rank(group), dist.get_world_size(group)
        count_table = 2 * self.world * 128
        self.buf = symm.empty(2 * self.n_max + self.FLAG_DOUBLES + count_table, dtype=torch.float64, device=device)
        self.buf.zero_()
        torch.cuda.synchronize(device)
        self.handle = symm.rendezvous(self.buf, group)
        ptrs = [int(p) for p in self.handle.buffer_ptrs]
        if len(ptrs) != self.world or self.world > 16:
            raise RuntimeError("unexpected symmetric-memory layout")
        self.peer_buf = (C.c_uint64 * self.world)(*ptrs)
        self.peer_flag = (C.c_uint64 * self.world)(*[p + 2 * self.n_max * 8 for p in ptrs])
        self.peer_count_flag = (C.c_uint64 * self.world)(*[p + 2 * self.n_max * 8 + self.COUNT_FLAG_OFFSET * 4
                                                            for p in ptrs])
        self.peer_count_table = (C.c_uint64 * self.world)(*[p + (2 * self.n_max + self.FLAG_DOUBLES) * 8 for p in ptrs])
        self.step = torch.zeros(1, dtype=torch.int32, device=device)
        self.count_step = torch.zeros(1, dtype=torch.int32, device=device)
        self.error = torch.zeros(1, dtype=torch.int32, device=device)
        dist.barrier(group)                # every rank has zeroed its flags before anybody publishes
        torch.cuda.synchronize(device)
        import os
        from . import _cabi
        ms = os.environ.get("BACS_PEER_TIMEOUT_MS")
        if ms:
            _cabi.check(_cabi.load().bacs_peer_set_timeout_ms(int(ms)), "bacs_peer_set_timeout_ms")

    @classmethod
    def create(cls, n_max: int, device: torch.device, group=None) -> "Optional[PeerReducer]":
        import os
        if os.environ.get("BACS_PEER_ALLREDUCE", "1") == "0":
            return None
        try:
            return cls(n_max, device, group)
        except Exception as exc:           # noqa: BLE001 -- transport choice only: NCCL does the same sum
            import warnings
            warnings.warn("bacs_b200: peer-memory all-reduce unavailable (%r); using the NCCL all-reduce" % (exc,))
            return None

    def check(self) -> None:
        """Host synchronisation point: raises when any exchange since the last check timed out (the kernel then left
        prototypes / counts untouched on THIS rank while the peers may have advanced, so the run cannot continue).
        Called by Prototypes at the end of an epoch / task and by bench.py's N > 1 verification step."""
        step = int(self.error.item())
        if step != 0:
            self.error.zero_()
            raise RuntimeError(
                "bacs_b200: NVLink peer all-reduce timed out on rank %d at exchange %d (a peer did not publish its "
                "state within the time-out, see bacs_peer_set_timeout_ms / BACS_PEER_TIMEOUT_MS); prototypes are no "
                "longer identical across ranks" % (self.rank, step))

    def allreduce(self, packed: torch.Tensor, proto: Optional[torch.Tensor] = None,
                  count: Optional[torch.Tensor] = None, T: int = 0, D: int = 0) -> Optional[torch.Tensor]:
        """In-place sum of ``packed`` (fp64, contiguous) over the ranks; with ``proto`` / ``count`` the running-mean
        prototype update runs in the same launch and the int32 ready flag is returned."""
        from . import _cabi, ops
        if packed.dtype != torch.float64 or not packed.is_contiguous() or packed.numel() > self.n_max:
            raise ValueError("PeerReducer.allreduce: packed must be contiguous fp64 with <= %d elements" % self.n_max)
        ready = None
        args_proto = (None, None, 0, 0, 0, None)
        if proto is not None:
            ready = torch.empty(1, dtype=torch.int32, device=packed.device)
            args_proto = (proto.data_ptr(), count.data_ptr(), int(count.dtype == torch.int64), int(T), int(D),
                          ready.data_ptr())
        lib = _cabi.load()
        _cabi.check(lib.bacs_peer_allreduce(packed.data_ptr(), packed.numel(), self.n_max, self.rank, self.world,
                                            self.peer_buf, self.peer_flag, self.step.data_ptr(), self.error.data_ptr(),
                                            *args_proto, ops._stream()),
                    "bacs_peer_allreduce")
        return ready


    def count_view(self, n_bt: torch.Tensor):
        """Count phase of the global prototype view (one launch): returns (view_pre, view_n) int64 [T] for
        ops.proto_accumulate_view.  On a time-out the view is marked invalid, the step then changes no prototype or
        count, and ``check`` raises."""
        from . import _cabi, ops
        n_bt = ops._cuda(n_bt, "PeerReducer.count_view", torch.int32)
        B, T = n_bt.shape
        view_pre = torch.empty(T, dtype=torch.int64, device=n_bt.device)
        view_n = torch.empty(T, dtype=torch.int64, device=n_bt.device)
        _cabi.check(_cabi.load().bacs_peer_count_exchange(n_bt.data_ptr(), B, T, self.rank, self.world,
                                                          self.peer_count_table, self.peer_count_flag,
                                                          self.count_step.data_ptr(), self.error.data_ptr(),
                                                          view_pre.data_ptr(), view_n.data_ptr(), ops._stream()),
                    "bacs_peer_count_exchange")
        return view_pre, view_n


_peer_reducers = {}


def peer_reducer(n: int, device: torch.device) -> "Optional[PeerReducer]":
    """Cached per device; sized for the largest prototype state the kernels take (128 tasks x 2048 channels)."""
    key = (device.index, world_size())
    if key not in _peer_reducers:
        _peer_reducers[key] = PeerReducer.create(max(int(n), 128 * 2048 + 128), device)
    red = _peer_reducers[key]
    return red if (red is not None and n <= red.n_max) else None


def check_peer_errors() -> None:
    """Raise if any peer exchange of this process timed out (no-op without a peer reducer)."""
    for red in _peer_reducers.values():
        if red is not None:
            red.check()


def gather_task_counts(totals: torch.Tensor, group=None) -> torch.Tensor:
    """[world, T] table of every rank's task totals, rank r in row r (one all-gather; the table is ``totals`` itself
    at world size 1)."""
    world = world_size()
    if world == 1:
        return totals.reshape(1, -1)
    table = torch.empty(world * totals.numel(), dtype=totals.dtype, device=totals.device)
    dist.all_gather_into_tensor(table, totals, group=group)
    return table.view(world, totals.numel())


def exchange_task_counts(n_bt: torch.Tensor, reducer: "Optional[PeerReducer]" = None):
    """Global view of the exact-mode prototype sums: (view_pre, view_n) int64 [T], task t's masked pixels in the images
    of the lower ranks / of all ranks.  Through peer memory when ``reducer`` is given, else one all-gather of the
    [T] task totals; no host synchronisation either way."""
    if reducer is not None:
        return reducer.count_view(n_bt)
    from . import ops
    table = gather_task_counts(ops.proto_task_totals(n_bt))
    return ops.proto_count_view(table, dist.get_rank() if world_size() > 1 else 0)


def allreduce_state(sums: Optional[torch.Tensor], counts: Optional[torch.Tensor],
                    confmat: Optional[torch.Tensor], group=None) -> None:
    """Prototype sums / counts and an int64 confusion matrix in one fp64 all-reduce
    (bacs_pack_state / bacs_unpack_state do the int64 <-> fp64 conversion on the device)."""
    if world_size() == 1:
        return
    from . import ops
    device = (confmat if confmat is not None else sums).device
    packed = ops.pack_state(sums, counts, confmat, device)
    dist.all_reduce(packed, op=dist.ReduceOp.SUM, group=group)
    ops.unpack_state(packed, sums, counts, confmat)
