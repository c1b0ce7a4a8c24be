"""CPU tests of the global prototype view: the new entry points' argument checks, answered before any CUDA call
(placeholder pointers are never dereferenced), and the property the view rests on -- summed over the shards of a
batch, the shards' global-view sums are the exact-mode sums of the whole batch, and their counts add up to its counts.
The sums come from an fp64 reference that is checked against the oracle's exact mode on the whole batch."""
import ctypes as C

import numpy as np
import pytest
import torch

from oracle import bacs_oracle as O
from proto_view_ref import exact_view_sums, shard_views

INVALID = -1
PTR = 0x1000           # placeholder: only passed where the call is refused


@pytest.fixture(scope="module")
def cabi():
    from bacs_b200 import _cabi
    return _cabi


def _view_call(cabi, T=6, mode=0, view_pre=PTR, view_n=PTR):
    return cabi.load().bacs_proto_accumulate_view(PTR, cabi.BF16, 2, 64, 8, 8, PTR, PTR, PTR, T, mode, view_pre, view_n,
                                                  PTR, PTR, PTR, 1 << 20, None)


@pytest.mark.parametrize("view_pre,view_n", [(PTR, None), (None, PTR)])
def test_view_needs_both_arrays(cabi, view_pre, view_n):
    assert _view_call(cabi, view_pre=view_pre, view_n=view_n) == INVALID
    assert "go together" in cabi.last_error()


@pytest.mark.parametrize("T", [0, -1, 129, 1000])
def test_view_task_count(cabi, T):
    assert _view_call(cabi, T=T) == INVALID
    assert cabi.last_error().startswith("bacs_proto_accumulate_view:")
    assert cabi.load().bacs_proto_task_totals(PTR, 2, T, PTR, None) == INVALID
    assert cabi.load().bacs_proto_count_view(PTR, 2, 0, T, PTR, PTR, None) == INVALID
    table = (C.c_uint64 * 2)(PTR, PTR)
    assert cabi.load().bacs_peer_count_exchange(PTR, 2, T, 0, 2, table, table, PTR, PTR, PTR, PTR, None) == INVALID


@pytest.mark.parametrize("mode", [1, 2, -1])
def test_view_needs_exact_mode(cabi, mode):
    assert _view_call(cabi, mode=mode) == INVALID
    assert cabi.last_error().startswith("bacs_proto_accumulate_view:")


def test_count_exchange_arguments(cabi):
    lib = cabi.load()
    assert lib.bacs_proto_count_view(None, 2, 0, 6, PTR, PTR, None) == INVALID
    assert lib.bacs_proto_count_view(PTR, 2, 2, 6, PTR, PTR, None) == INVALID          # rank >= world
    assert lib.bacs_proto_count_view(PTR, 0, 0, 6, PTR, PTR, None) == INVALID
    assert lib.bacs_proto_task_totals(PTR, 0, 6, PTR, None) == INVALID
    assert lib.bacs_proto_task_totals(None, 2, 6, PTR, None) == INVALID
    table = (C.c_uint64 * 17)(*([PTR] * 17))
    assert lib.bacs_peer_count_exchange(PTR, 2, 6, 0, 17, table, table, PTR, PTR, PTR, PTR, None) == INVALID
    assert lib.bacs_peer_count_exchange(PTR, 2, 6, 2, 2, table, table, PTR, PTR, PTR, PTR, None) == INVALID
    assert lib.bacs_peer_count_exchange(PTR, 2, 6, 0, 2, table, table, PTR, PTR, None, PTR, None) == INVALID


# --------------------------------------------------------------------------------------
# the property: shard sums add up to the exact sums of the concatenated batch
# --------------------------------------------------------------------------------------
INITIAL, INCREMENT = 2, 1        # class c >= 1 belongs to task c - 1


def _batch(B, D, H, W, T, seed):
    g = torch.Generator().manual_seed(seed)
    c = torch.randint(0, T + 3, (B, H // 4, W // 4), generator=g)
    c = torch.where(torch.rand(c.shape, generator=g) > 0.93, torch.full_like(c, 255), c)
    labels = c.repeat_interleave(4, 1).repeat_interleave(4, 2)
    labels[0][labels[0] == 2] = 0                        # image 0 has no pixel of task 1
    feat = torch.randn(B, D, H, W, generator=g, dtype=torch.float64)
    lut = O.class_task_lut(INITIAL, INCREMENT)
    lab = labels.numpy()
    task = np.where(lab < 256, lut[np.clip(lab, 0, 255)], -1)
    task = np.where(task >= T, -1, task)
    n_bt = np.stack([[(task[b] == t).sum() for t in range(T)] for b in range(B)])
    return feat, labels, task, n_bt


SPLITS = [(0, 6, 12), (0, 1, 5, 12), (0, 1, 2, 4, 5, 8, 9, 11, 12), (0, 11, 12)]


@pytest.mark.parametrize("bounds", SPLITS, ids=["2-even", "3-uneven", "8-shards", "2-last-single"])
@pytest.mark.parametrize("T", [3, 6])
def test_shard_sums_add_up_to_batch_sums(bounds, T):
    B, D = 12, 16
    feat, labels, task, n_bt = _batch(B, D, 16, 20, T, seed=T * 100 + len(bounds))
    assert n_bt[0, 1] == 0 and n_bt[:, 1].sum() > 0
    S, A, N = exact_view_sums(feat, task, T)
    # the fp64 reference agrees with the oracle's exact mode on the whole batch
    so, no = O.proto_accumulate(feat.float(), labels, INITIAL, INCREMENT, T, mode="exact")
    assert torch.equal(no, N)
    assert torch.all((so.double() - S).abs() <= 1e-5 * A + 1e-30)
    total, counts = torch.zeros_like(S), torch.zeros_like(N)
    for (lo, hi), view in zip(zip(bounds[:-1], bounds[1:]), shard_views(n_bt, bounds)):
        assert np.all(view[0] + n_bt[lo:hi].sum(0) <= view[1])
        s, _, n = exact_view_sums(feat[lo:hi], task[lo:hi], T, view)
        total += s
        counts += n
    assert torch.equal(counts, N)
    assert torch.all((total - S).abs() <= 1e-12 * A)
    # and the global view is not the local one: a shard on its own gives different rows
    s_local = sum(exact_view_sums(feat[lo:hi], task[lo:hi], T)[0] for lo, hi in zip(bounds[:-1], bounds[1:]))
    assert not torch.allclose(s_local, S, rtol=1e-6, atol=1e-6)
