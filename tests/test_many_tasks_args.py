"""CPU tests of the task-count limit (1 <= T <= 128, the int8 task map's range) of the task down-sample, the prototype
sums and update, the peer all-reduce's prototype update and bacs_seen_logits_many, answered before any CUDA call.
Placeholder pointers are only passed where the call is refused and are never dereferenced."""
import ctypes as C

import pytest
import torch

INVALID = -1
PTR = 0x1000
LIMIT_MSG = "not in [1,128]"


@pytest.fixture(scope="module")
def cabi():
    from bacs_b200 import _cabi
    return _cabi


def _downsample(lib, T):
    return lib.bacs_label_downsample_task(PTR, 2, 64, 64, 4, 4, PTR, T, None, PTR, PTR, PTR, None)


def _accumulate(lib, T):
    return lib.bacs_proto_accumulate(PTR, 1, 2, 64, 4, 4, PTR, PTR, PTR, T, 0, PTR, PTR, PTR, 1 << 30, None)


def _accumulate_update(lib, T):
    return lib.bacs_proto_accumulate_update(PTR, 1, 2, 64, 4, 4, PTR, PTR, PTR, T, 0, PTR, PTR, PTR, 1 << 30, PTR, PTR,
                                            1, PTR, None)


def _update(lib, T):
    return lib.bacs_proto_update(PTR, PTR, 1, PTR, PTR, T, 64, PTR, None)


def _peer(lib, T):
    n = 1 << 20
    bufs = (C.c_uint64 * 1)(PTR)
    return lib.bacs_peer_allreduce(PTR, n, n, 0, 1, bufs, bufs, PTR, PTR, PTR, PTR, 1, T, 64, PTR, None)


def _many_stacked(lib, T):
    return lib.bacs_seen_logits_many(PTR, 1, 2, 64, 4, 4, PTR, PTR, PTR, None, None, T, PTR, None, None)


def _many_heads(lib, T):
    return lib.bacs_seen_logits_many(PTR, 1, 2, 64, 4, 4, PTR, None, None, PTR, PTR, T, PTR, None, None)


ENTRY_POINTS = [("bacs_label_downsample_task", _downsample), ("bacs_proto_accumulate", _accumulate),
                ("bacs_proto_accumulate_update", _accumulate_update), ("bacs_proto_update", _update),
                ("bacs_peer_allreduce", _peer), ("bacs_seen_logits_many", _many_stacked),
                ("bacs_seen_logits_many", _many_heads)]


@pytest.mark.parametrize("name,call", ENTRY_POINTS, ids=[f.__name__.lstrip("_") for _, f in ENTRY_POINTS])
@pytest.mark.parametrize("T", [0, 129, 200])
def test_task_count_refused(cabi, name, call, T):
    assert call(cabi.load(), T) == INVALID
    msg = cabi.last_error()
    assert msg.startswith(name + ":"), msg
    assert ("T=%d %s" % (T, LIMIT_MSG)) in msg, msg


def test_seen_logits_keep_their_32_head_limit(cabi):
    lib = cabi.load()
    assert lib.bacs_seen_logits(PTR, 1, 2, 64, 4, 4, PTR, PTR, PTR, 33, PTR, None) == INVALID
    assert "T=33 not in [1,32]" in cabi.last_error()
    heads = (C.c_void_p * 33)(*([PTR] * 33))
    assert lib.bacs_seen_logits_heads(PTR, 1, 2, 64, 4, 4, PTR, heads, heads, 33, PTR, None, None) == INVALID
    assert "T=33 not in [1,32]" in cabi.last_error()


def test_seen_logits_many_needs_one_head_form(cabi):
    lib = cabi.load()
    # neither the stacked nor the per-head arrays
    assert lib.bacs_seen_logits_many(PTR, 1, 2, 64, 4, 4, PTR, None, None, None, None, 40, PTR, None, None) == INVALID
    assert "null pointer" in cabi.last_error()
    # a null head inside the per-head arrays
    w = (C.c_void_p * 40)(*([PTR] * 39 + [None]))
    assert lib.bacs_seen_logits_many(PTR, 1, 2, 64, 4, 4, PTR, None, None, w, w, 40, PTR, None, None) == INVALID
    assert "null head 39" in cabi.last_error()


@pytest.mark.parametrize("B,D", [(1, 1), (24, 512), (8, 2048)])
def test_proto_workspace_is_monotone_in_T(cabi, B, D):
    lib = cabi.load()
    sizes = [lib.bacs_proto_workspace_bytes(B, D, T) for T in range(1, 129)]
    assert all(b >= a for a, b in zip(sizes, sizes[1:]))
    assert sizes[-1] >= B * D * 128 * 2 * 4


def test_python_refuses_more_than_128_tasks():
    from bacs_b200 import _cabi, ops
    ops.check_task_count(128, "x")
    for T in (0, 129):
        with pytest.raises(_cabi.BacsError, match=r"\[1, 128\]"):
            ops.check_task_count(T, "x")
    # before any tensor reaches the device: CPU tensors would be refused later with a different error
    with pytest.raises(_cabi.BacsError, match="128"):
        ops.label_downsample_task(torch.zeros(1, 8, 8, dtype=torch.int64), 2, 2, torch.zeros(256, dtype=torch.int32),
                                  129)
    with pytest.raises(_cabi.BacsError, match="128"):
        ops.proto_accumulate(torch.zeros(1, 4, 2, 2), None, None, None, 129)
    with pytest.raises(_cabi.BacsError, match="128"):
        ops.proto_update(torch.zeros(129, 4), torch.zeros(129), None, None)
    with pytest.raises(_cabi.BacsError, match="128"):
        ops.seen_logits_many(torch.zeros(1, 4, 2, 2), torch.zeros(129, 4), torch.zeros(129, 4), torch.zeros(129))
    with pytest.raises(_cabi.BacsError, match="128"):
        ops.seen_logits_many(torch.zeros(1, 4, 2, 2), torch.zeros(129, 4), [torch.zeros(4)] * 129,
                             [torch.zeros(1)] * 129)
