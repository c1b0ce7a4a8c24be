"""The global view of the exact-mode prototype sums (bacs_proto_accumulate_view) in one process: a batch is cut into
W shards, each shard is accumulated with the view that its rank would receive from the count exchange, and the fp64
sums of the shards are added in shard order.  That must give the exact mode on the whole batch: counts exact, sums
within 1e-12 x (sum of the row's |addends|) of the whole-batch launch and within 1e-5 x the same of the fp64 oracle.

Every kernel path is covered: the one-hot mma.sync kernel (bf16, fp16), the 8-pixel table kernel with its gather
(fp32, h*w not a multiple of 32) and the ragged-row table kernel (h*w not a multiple of 8), each at T <= 32 and with
its 32-task windows (T > 32)."""
import numpy as np
import pytest
import torch

from oracle import bacs_oracle as O
from proto_view_ref import exact_view_sums, shard_views

pytestmark = pytest.mark.gpu

INITIAL, INCREMENT = 2, 1        # class c >= 1 belongs to task c - 1
DTYPES = {"f32": torch.float32, "bf16": torch.bfloat16, "f16": torch.float16}
# W = 2 (even), 3 (uneven, a 1-image shard holding no pixel of task 1), 8 (uneven, several 1-image shards)
SPLITS = {2: (0, 6, 12), 3: (0, 1, 5, 12), 8: (0, 1, 2, 4, 5, 8, 9, 11, 12)}
# (path, dtype, (D, h, w), task counts)
PATHS = [("mma", "bf16", (64, 32, 40), (6, 32, 33, 128)),
         ("mma", "f16", (64, 32, 40), (6, 32, 33, 128)),
         ("vec", "f32", (40, 24, 42), (6, 33, 128)),
         ("scalar", "f32", (40, 29, 41), (25, 32, 33)),
         ("scalar", "bf16", (40, 29, 41), (25, 32))]
CASES = [(p, d, g, T) for p, d, g, Ts in PATHS for T in Ts]
IDS = ["%s-%s-T%d" % (p, d, T) for p, d, _, T in CASES]


@pytest.fixture(scope="module")
def ops():
    from bacs_b200 import ops as _ops
    return _ops


def _batch(ops, dname, D, h, w, T, seed, B=12):
    g = torch.Generator().manual_seed(seed)
    c = torch.randint(1, T + 4, (B, (h + 3) // 4, (w + 3) // 4), generator=g)
    u = torch.rand(c.shape, generator=g)
    c = torch.where(u < 0.15, torch.zeros_like(c), c)
    c = torch.where(u > 0.95, torch.full_like(c, 255), c)
    labels = c.repeat_interleave(4, 1).repeat_interleave(4, 2)[:, :h, :w].contiguous()
    sp = torch.rand(B, h, w, generator=g) < 0.05
    labels = torch.where(sp, torch.randint(0, T + 2, (B, h, w), generator=g), labels)
    labels[0][labels[0] == 2] = 0                         # image 0 (a shard of its own) has no pixel of task 1
    feat = torch.randn(B, D, h, w, generator=g).to(DTYPES[dname]).cuda()
    lut = torch.from_numpy(O.class_task_lut(INITIAL, INCREMENT).astype(np.int32)).cuda()
    task, rank, n_bt, _ = ops.label_downsample_task(labels.cuda(), h, w, lut, T)
    return feat, task, rank, n_bt


def _path(monkeypatch, path):
    if path != "mma":
        monkeypatch.setenv("BACS_NO_PROTO_MMA", "1")


def _shard_sums(ops, feat, task, rank, n_bt, T, bounds):
    views = shard_views(n_bt.cpu().numpy(), bounds)
    total = torch.zeros(T, feat.shape[1], dtype=torch.float64, device=feat.device)
    counts = torch.zeros(T, dtype=torch.float64, device=feat.device)
    for (lo, hi), (vp, vn) in zip(zip(bounds[:-1], bounds[1:]), views):
        s, n = ops.proto_accumulate_view(feat[lo:hi], task[lo:hi], rank[lo:hi], n_bt[lo:hi].contiguous(), T,
                                         torch.from_numpy(vp).cuda(), torch.from_numpy(vn).cuda())
        total += s
        counts += n
    return total, counts


@pytest.mark.parametrize("W", sorted(SPLITS))
@pytest.mark.parametrize("path,dname,geom,T", CASES, ids=IDS)
def test_shards_equal_whole_batch(ops, monkeypatch, path, dname, geom, T, W):
    _path(monkeypatch, path)
    D, h, w = geom
    feat, task, rank, n_bt = _batch(ops, dname, D, h, w, T, seed=T * 7 + D)
    nb = n_bt.cpu().numpy()
    assert nb[0, 1] == 0 and nb[:, 1].sum() > 0
    total, counts = _shard_sums(ops, feat, task, rank, n_bt, T, SPLITS[W])
    whole, whole_n = ops.proto_accumulate(feat, task, rank, n_bt, T, 0)
    S, A, N = exact_view_sums(feat, task.cpu().numpy().astype(np.int64), T)
    torch.cuda.synchronize()
    assert torch.equal(counts.cpu().long(), N) and torch.equal(whole_n.cpu().long(), N)
    A = A.cuda()
    assert torch.all((total - whole).abs() <= 1e-12 * A), float(((total - whole).abs() / (A + 1e-300)).max())
    assert torch.all((total - S.cuda()).abs() <= 1e-5 * A + 1e-30)


@pytest.mark.parametrize("path,dname,geom,T", [c for c in CASES if c[3] in (6, 33, 128, 25)],
                         ids=[i for c, i in zip(CASES, IDS) if c[3] in (6, 33, 128, 25)])
def test_large_view_offsets(ops, monkeypatch, path, dname, geom, T):
    """A rank far into the global batch: D * (view_pre + pre_bt) passes 2^31, so the row arithmetic must be int64."""
    _path(monkeypatch, path)
    D, h, w = geom
    feat, task, rank, n_bt = _batch(ops, dname, D, h, w, T, seed=T * 11 + D, B=5)
    tot = n_bt.cpu().numpy().astype(np.int64).sum(0)
    g = np.random.default_rng(T)
    vp = (2 ** 31 // D + g.integers(0, 10 ** 6, T)).astype(np.int64)
    vn = vp + tot + g.integers(0, 10 ** 6, T)
    s, n = ops.proto_accumulate_view(feat, task, rank, n_bt, T, torch.from_numpy(vp).cuda(), torch.from_numpy(vn).cuda())
    S, A, N = exact_view_sums(feat, task.cpu().numpy().astype(np.int64), T, (vp, vn))
    torch.cuda.synchronize()
    assert torch.equal(n.cpu().long(), N)
    assert torch.all((s.cpu() - S).abs() <= 1e-5 * A + 1e-30)


@pytest.mark.parametrize("path,dname,geom,T", CASES, ids=IDS)
def test_local_view_is_bit_identical(ops, monkeypatch, path, dname, geom, T):
    _path(monkeypatch, path)
    D, h, w = geom
    feat, task, rank, n_bt = _batch(ops, dname, D, h, w, T, seed=T * 13 + D)
    tot = n_bt.long().sum(0)
    s, n = ops.proto_accumulate_view(feat, task, rank, n_bt, T, torch.zeros_like(tot), tot)
    s0, n0 = ops.proto_accumulate(feat, task, rank, n_bt, T, 0)
    torch.cuda.synchronize()
    assert torch.equal(s, s0) and torch.equal(n, n0)


@pytest.mark.parametrize("path,dname,geom,T", [c for c in CASES if c[3] in (6, 33)],
                         ids=[i for c, i in zip(CASES, IDS) if c[3] in (6, 33)])
def test_invalid_view_adds_nothing(ops, monkeypatch, path, dname, geom, T):
    """view_n < 0 (the mark of a count phase that timed out): no sums, -inf counts, and an update that changes nothing."""
    _path(monkeypatch, path)
    D, h, w = geom
    feat, task, rank, n_bt = _batch(ops, dname, D, h, w, T, seed=T * 17 + D)
    s, n = ops.proto_accumulate_view(feat, task, rank, n_bt, T, torch.zeros(T, dtype=torch.int64, device="cuda"),
                                     torch.full((T,), -1, dtype=torch.int64, device="cuda"))
    proto = torch.randn(T, D, device="cuda")
    count = torch.arange(T, dtype=torch.int64, device="cuda") + 5
    p0, c0 = proto.clone(), count.clone()
    ops.proto_update(proto, count, s, n)
    torch.cuda.synchronize()
    assert torch.all(s == 0) and torch.all(n == float("-inf"))
    assert torch.equal(proto, p0) and torch.equal(count, c0)


def test_count_exchange_world_size_one(ops):
    from bacs_b200.distributed import exchange_task_counts
    for T in (6, 128):
        _, _, _, n_bt = _batch(ops, "bf16", 16, 32, 40, T, seed=T)
        vp, vn = exchange_task_counts(n_bt)
        torch.cuda.synchronize()
        assert vp.dtype == vn.dtype == torch.int64
        assert torch.equal(vp.cpu(), torch.zeros(T, dtype=torch.int64))
        assert torch.equal(vn.cpu(), n_bt.cpu().long().sum(0))
        table = torch.tensor([[3] * T, [5] * T, [7] * T], dtype=torch.int64, device="cuda")
        vp, vn = ops.proto_count_view(table, 1)
        torch.cuda.synchronize()
        assert torch.all(vp == 3) and torch.all(vn == 15)


@pytest.mark.parametrize("T", [6, 128])
def test_step_path_graph_replay(ops, T):
    """count exchange -> view accumulate -> update, captured in a CUDA graph: replays match the eager run bit for bit."""
    from bacs_b200.distributed import exchange_task_counts
    D, h, w = 64, 32, 40
    feat, task, rank, n_bt = _batch(ops, "bf16", D, h, w, T, seed=T + 1)
    proto0 = torch.randn(T, D, device="cuda")
    count0 = torch.full((T,), 3, dtype=torch.int64, device="cuda")

    def step(proto, count):
        vp, vn = exchange_task_counts(n_bt)
        s, n = ops.proto_accumulate_view(feat, task, rank, n_bt, T, vp, vn)
        return ops.proto_update(proto, count, s, n)

    want_p, want_c = proto0.clone(), count0.clone()
    for _ in range(3):
        step(want_p, want_c)
    proto, count = proto0.clone(), count0.clone()
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        wp, wc = proto0.clone(), count0.clone()
        step(wp, wc)                                        # warm-up outside the capture
    torch.cuda.current_stream().wait_stream(side)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        ready = step(proto, count)
    proto.copy_(proto0)
    count.copy_(count0)
    for _ in range(3):
        graph.replay()
    torch.cuda.synchronize()
    assert torch.equal(proto, want_p) and torch.equal(count, want_c)
    assert int(ready) == 1
