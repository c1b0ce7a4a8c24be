"""Continual runs longer than 32 tasks (33 <= T <= 128): the task down-sample, the prototype sums and running-mean
update on every kernel path, bacs_seen_logits_many, and the whole BACS loss step, against float64 / oracle references.

Error model as in test_gpu_seen_heads.py: a value that is a sum of terms may differ from its float64 value by
1e-5 x (the sum of the terms' absolute values); counts, task ids and ranks are exact."""
import numpy as np
import pytest
import torch

from oracle import bacs_oracle as O

pytestmark = pytest.mark.gpu

RTOL = 1e-5
MANY = (33, 40, 64, 65, 127, 128)
DTYPES = {"f32": torch.float32, "bf16": torch.bfloat16, "f16": torch.float16}
INITIAL, INCREMENT = 2, 1        # class c >= 1 belongs to task c - 1: classes 1..T span all T tasks


@pytest.fixture(scope="module")
def ops():
    from bacs_b200 import ops as _ops
    return _ops


def _labels(B, H, W, T, seed, block=4):
    """[B,H,W] int64 in blocks: background, ignore 255, classes of every task and classes of tasks not created yet."""
    g = torch.Generator().manual_seed(seed)
    gh, gw = (H + block - 1) // block, (W + block - 1) // block
    c = torch.randint(0, min(T + 8, 254) + 1, (B, gh, gw), generator=g)
    u = torch.rand(B, gh, gw, generator=g)
    c = torch.where(u < 0.2, torch.zeros_like(c), c)
    c = torch.where(u > 0.95, torch.full_like(c, 255), c)
    lab = c.repeat_interleave(block, 1).repeat_interleave(block, 2)[:, :H, :W].contiguous()
    sp = torch.rand(B, H, W, generator=g) < 0.05          # per-pixel speckle of random classes
    return torch.where(sp, torch.randint(0, T + 2, (B, H, W), generator=g), lab)


def _task_ref(labels, h, w, T):
    """-> task [B,h,w] (int, -1 none), rank [B,h,w], n_bt [B,T] from the oracle's down-sample and np.rint class->task."""
    down = O.downsample_labels(labels, h, w).numpy()
    lut = O.class_task_lut(INITIAL, INCREMENT)
    task = np.where((down >= 0) & (down < 256), lut[np.clip(down, 0, 255)], -1)
    task = np.where(task >= T, -1, task)
    B = task.shape[0]
    flat = task.reshape(B, -1)
    rank = np.zeros_like(flat)
    n_bt = np.zeros((B, T), dtype=np.int64)
    for b in range(B):
        for t in range(T):
            m = flat[b] == t
            rank[b, m] = np.arange(int(m.sum()))
            n_bt[b, t] = int(m.sum())
    return task, rank.reshape(task.shape), n_bt


def _device_lut():
    return torch.from_numpy(O.class_task_lut(INITIAL, INCREMENT).astype(np.int32)).cuda()


# --------------------------------------------------------------------------------------
# task down-sample
# --------------------------------------------------------------------------------------
@pytest.mark.parametrize("T", MANY)
@pytest.mark.parametrize("B,H,W,h,w", [(3, 96, 80, 48, 40), (2, 512, 512, 32, 32), (1, 37, 53, 37, 53)])
def test_downsample_task_bit_exact(ops, T, B, H, W, h, w):
    labels = _labels(B, H, W, T, seed=T + H)
    task, rank, n_bt, down = ops.label_downsample_task(labels.cuda(), h, w, _device_lut(), T, want_labels_down=True)
    want_task, want_rank, want_n = _task_ref(labels, h, w, T)
    assert torch.equal(down.cpu(), O.downsample_labels(labels, h, w))
    assert np.array_equal(task.cpu().numpy().astype(np.int64), want_task)
    got_rank = rank.cpu().numpy()
    assert np.array_equal(np.where(want_task >= 0, got_rank, 0), want_rank)
    assert np.array_equal(n_bt.cpu().numpy(), want_n)
    assert int((want_n > 0).sum(1).max()) > 32, "labels must span more than 32 tasks"


# --------------------------------------------------------------------------------------
# prototype sums / running-mean update
# --------------------------------------------------------------------------------------
def _sums64(feat, task, n_bt, T, mode):
    """float64 sums [T,D] and sums of |terms| of the reference's masked view(D,-1) rows (mode 0) or channels (1)."""
    x = feat.detach().cpu().double()
    B, D = x.shape[:2]
    xf = x.reshape(B, D, -1)
    tf = torch.from_numpy(task.reshape(B, -1))
    S = torch.zeros(T, D, dtype=torch.float64)
    A = torch.zeros(T, D, dtype=torch.float64)
    for t in range(T):
        n = int(n_bt[:, t].sum())
        if n == 0:
            continue
        if mode == 1:
            m = (tf == t).unsqueeze(1).double()
            S[t] = (xf * m).sum((0, 2))
            A[t] = (xf.abs() * m).sum((0, 2))
        else:
            flat = torch.cat([xf[b][:, tf[b] == t].reshape(-1) for b in range(B)]).view(D, n)
            S[t], A[t] = flat.sum(-1), flat.abs().sum(-1)
    return S, A


# (path, dtype name, geometry): mma = one-hot GEMM (16-bit, hw % 32 == 0, D % 16 == 0); vec = 8-pixel table kernel;
# scalar = table kernel for ragged rows (hw % 8 != 0)
PROTO_PATHS = [("mma", "bf16", (3, 64, 48, 40)), ("mma", "f16", (3, 64, 48, 40)),
               ("vec", "bf16", (3, 64, 48, 40)), ("vec", "f32", (3, 48, 48, 40)),
               ("scalar", "f32", (2, 40, 45, 41)), ("scalar", "bf16", (2, 40, 45, 41))]


@pytest.mark.parametrize("mode", [0, 1], ids=["exact", "channel"])
@pytest.mark.parametrize("path,dname,geom", PROTO_PATHS, ids=["%s-%s" % (p, d) for p, d, _ in PROTO_PATHS])
@pytest.mark.parametrize("T", MANY)
def test_proto_sums_and_update(ops, monkeypatch, T, path, dname, geom, mode):
    if path != "mma":
        monkeypatch.setenv("BACS_NO_PROTO_MMA", "1")
    _check_proto(ops, T, dname, geom, mode)


@pytest.mark.parametrize("mode", [0, 1], ids=["exact", "channel"])
@pytest.mark.parametrize("dname", ["f32", "bf16"])
@pytest.mark.parametrize("T", [25, 28, 32])
def test_proto_ragged_rows_25_to_32_tasks(ops, T, dname, mode):
    """the table kernel for ragged rows at 25..32 tasks: its 2048 * T bytes of shared memory need the opt-in above
    the 48 KB default (without it the launch fails)"""
    _check_proto(ops, T, dname, (2, 40, 45, 41), mode)


def _check_proto(ops, T, dname, geom, mode):
    B, D, h, w = geom
    dtype = DTYPES[dname]
    g = torch.Generator().manual_seed(T * 7 + D)
    feat = (torch.randn(B, D, h, w, generator=g) * 2).to(dtype).cuda()
    labels = _labels(B, h, w, T, seed=T * 3 + h)
    task, rank, n_bt, _ = ops.label_downsample_task(labels.cuda(), h, w, _device_lut(), T)
    want_task, _, want_n = _task_ref(labels, h, w, T)
    sums, counts = ops.proto_accumulate(feat, task, rank, n_bt, T, mode)
    S, A = _sums64(feat, want_task, want_n, T, mode)
    err = (sums.cpu() - S).abs()
    assert bool((err <= RTOL * A).all()), "sums: worst %.3g of 1e-5 x sum|terms|" % float((err / (RTOL * A + 1e-300)).max())
    assert torch.equal(counts.cpu(), torch.from_numpy(want_n.sum(0)).double())
    # running mean, fused into the sums' launches and as its own launch, for both count types
    proto0 = torch.randn(T, D, generator=g).cuda()
    for cdt in (torch.int64, torch.float32):
        count0 = torch.randint(0, 3, (T,), generator=g).to(cdt).cuda()
        n = torch.from_numpy(want_n.sum(0)).cuda()
        num = sums.float() + count0.float().unsqueeze(1) * proto0
        want_p = torch.where((n > 0).unsqueeze(1), num / (count0 + n).float().unsqueeze(1), proto0)
        want_c = torch.where(n > 0, count0 + n.to(cdt), count0)
        want_ready = int(bool((want_c != 0).all()))
        p, c = proto0.clone(), count0.clone()
        s2, c2, ready = ops.proto_accumulate_update(feat, task, rank, n_bt, mode, p, c)
        assert torch.equal(c, want_c) and int(ready) == want_ready
        assert torch.allclose(p, want_p, rtol=RTOL, atol=RTOL * float(want_p.abs().max()))
        p, c = proto0.clone(), count0.clone()
        ready = ops.proto_update(p, c, sums, counts)
        assert torch.equal(c, want_c) and int(ready) == want_ready
        assert torch.allclose(p, want_p, rtol=RTOL, atol=RTOL * float(want_p.abs().max()))


# --------------------------------------------------------------------------------------
# bacs_seen_logits_many
# --------------------------------------------------------------------------------------
def seen_logits64(feat, proto, weight, bias):
    x = feat.detach().cpu().double()
    B, D, h, w = x.shape
    sx = torch.sigmoid(x).reshape(B, D, h * w)
    sp = torch.sigmoid(proto.detach().cpu().double())
    W = weight.detach().cpu().double().reshape(-1, D)
    bb = bias.detach().cpu().double().reshape(-1)
    T = W.shape[0]
    z = torch.empty(B, T, h * w, dtype=torch.float64)
    a = torch.empty_like(z)
    for t in range(T):
        d = (sx - sp[t].view(1, D, 1)).abs()
        z[:, t] = torch.einsum("c,bcq->bq", W[t], d) + bb[t]
        a[:, t] = torch.einsum("c,bcq->bq", W[t].abs(), d) + bb[t].abs()
    return z.view(B, T, h, w), a.view(B, T, h, w)


def _seen_inputs(T, D, B, h, w, dtype, seed):
    g = torch.Generator().manual_seed(seed)
    feat = (torch.randn(B, D, h, w, generator=g) * 2).to(dtype).cuda()
    proto = (torch.randn(T, D, generator=g) * 1.5).cuda()
    weight = (torch.randn(T, D, generator=g) * 0.2).cuda()
    bias = torch.randn(T, generator=g).cuda()
    return feat, proto, weight, bias


def _check64(z, feat, proto, weight, bias):
    z64, a64 = seen_logits64(feat, proto, weight, bias)
    err = (z.cpu().double() - z64).abs()
    bad = err > RTOL * a64
    assert not bool(bad.any()), "%d of %d entries beyond 1e-5 x sum|terms|" % (int(bad.sum()), bad.numel())


# (D, B, h, w): the VOC feature grid, a channel count that takes a cluster split, a ragged pixel count
SEEN_GEOMS = [(512, 2, 32, 32), (256, 1, 8, 8), (48, 2, 7, 9)]


@pytest.mark.parametrize("geom", SEEN_GEOMS, ids=["D%d-B%d-%dx%d" % g for g in SEEN_GEOMS])
@pytest.mark.parametrize("dname", list(DTYPES))
@pytest.mark.parametrize("T", MANY)
def test_seen_logits_many_against_fp64(ops, T, dname, geom):
    D, B, h, w = geom
    feat, proto, weight, bias = _seen_inputs(T, D, B, h, w, DTYPES[dname], seed=T * 1000 + D)
    z = ops.seen_logits_many(feat, proto, weight, bias)
    _check64(z, feat, proto, weight, bias)
    # the per-head form: same kernel, same bits; the focal accumulator (pre-filled with NaN) cleared everywhere
    ws = [weight[t].clone().reshape(1, D, 1, 1) for t in range(T)]
    bs = [bias[t].clone().reshape(1) for t in range(T)]
    zero = torch.full((B, h, w), float("nan"), device="cuda")
    zh = ops.seen_logits_many(feat, proto, ws, bs, zero_out=zero)
    assert torch.equal(zh, z)
    assert bool((zero == 0).all())


@pytest.mark.parametrize("dname", list(DTYPES))
@pytest.mark.parametrize("T", [1, 5, 12, 17, 32])
def test_seen_logits_many_agrees_with_seen_logits(ops, T, dname):
    """At T <= 32: within the fp64 bound at every shape.  Bit for bit where both launches split the channels over
    the same cluster size: the per-head sums then take the same order whatever TMAX and pixels per thread.  That holds
    at T > 16 (both launches use the TMAX = 32 plan, so the same cluster size) and, with today's cluster-size rule, at
    the small D = 48 grid, where both plans pick the same size.  The D = 48 equality rests on that rule: a change to
    it may change which plans agree."""
    for D, B, h, w in [(512, 2, 32, 32), (48, 2, 16, 16)]:
        feat, proto, weight, bias = _seen_inputs(T, D, B, h, w, DTYPES[dname], seed=T + D)
        z_many = ops.seen_logits_many(feat, proto, weight, bias)
        z_old = ops.seen_logits(feat, proto, weight, bias)
        _check64(z_many, feat, proto, weight, bias)
        if D < 64 or T > 16:
            assert torch.equal(z_many, z_old)


# --------------------------------------------------------------------------------------
# the whole BACS loss step
# --------------------------------------------------------------------------------------
def _many_cfg(T):
    from bacs_b200 import synth
    initial = 11 if T <= 40 else 24
    K = initial + (T - 1)
    return synth.StepConfig("many%d" % T, B=2, K=K, old_cl=K - 1, T=T, H=32, W=512, D=64, A=16,
                            initial_classes=initial, increment=1, Br=2)


def _many_inputs(cfg, seed):
    from bacs_b200 import synth
    inp = synth.make_step_inputs(cfg, seed=seed)
    gen = torch.Generator().manual_seed(seed + 1)
    inp.mask = synth.make_labels(cfg, gen, classes=list(range(1, cfg.K)), block=4)   # pixels of every task
    return inp


@pytest.mark.parametrize("T", [40, 128])
def test_step_matches_oracle(T):
    from bacs_b200 import synth
    cfg = _many_cfg(T)
    inp = _many_inputs(cfg, seed=T)
    loss_fn, net, batch, leaves = synth.build_bacs_step(cfg, inp, device="cuda")
    loss, preds = loss_fn.compute_loss(batch, net, train=True)
    loss.backward()
    torch.cuda.synchronize()

    leaf = lambda t: t.clone().requires_grad_(True)
    lg, na, hw, hb = leaf(inp.logits), leaf(inp.new_att), leaf(inp.head_w), leaf(inp.head_b)
    rp = inp.replay
    rlg, rsem = leaf(rp["logits"]), leaf(rp["sem_logits"])
    rp2 = dict(rp, logits=rlg, sem_logits=rsem, n_classes=rp["n_classes"].numpy())
    want = O.bacs_step(lg, inp.pen, inp.old_att, na, inp.mask, inp.protos, inp.counts, hw, hb,
                       initial_classes=cfg.initial_classes, increment=cfg.increment, old_cl=cfg.old_cl,
                       task_num=cfg.T - 1, epoch=3, max_epochs=30, replay=rp2, nb_current_classes=cfg.K)
    want["loss"].backward()
    got, ref = float(loss.detach()), float(want["loss"].detach())
    assert abs(got - ref) <= 1e-5 * abs(ref), (got, ref)
    assert torch.equal(preds.cpu(), want["preds"])
    P = loss_fn._prototypes
    wp = want["protos"]
    assert torch.allclose(P._prototypes_tensors.cpu(), wp, rtol=1e-5, atol=1e-5 * float(wp.abs().max()))
    assert torch.equal(P._count_features.cpu().double(), want["counts"].double())
    assert bool((want["counts"] > inp.counts)[32:].any()), "the step must update prototypes of tasks beyond 32"
    for key, w in (("logits", lg.grad), ("new_att", na.grad), ("replay_logits", rlg.grad), ("replay_sem", rsem.grad)):
        g = leaves[key].grad.cpu()
        tol = 3e-5 if key == "new_att" else 1e-5       # the bounds of test_gpu_fullstep.py
        assert float((g - w).abs().max()) <= tol * float(w.abs().max()), key
    t = cfg.T - 1
    gw = leaves["head_w"].grad.cpu().reshape(-1)
    assert float((gw - hw.grad[t]).abs().max()) <= 3e-5 * float(hw.grad[t].abs().max())


def test_step_is_free_of_host_sync_at_128_tasks():
    """the T = 128 step captures in a CUDA graph, replays bit for bit, and runs under set_sync_debug_mode("error")"""
    from bacs_b200 import synth
    cfg = _many_cfg(128)
    inp = _many_inputs(cfg, seed=5)
    loss_fn, net, batch, leaves = synth.build_bacs_step(cfg, inp, device="cuda")
    protos0 = loss_fn._prototypes._prototypes_tensors.clone()
    counts0 = loss_fn._prototypes._count_features.clone()

    def step():
        for v in leaves.values():
            v.grad = None
        loss, preds = loss_fn.compute_loss(batch, net, train=True)
        loss.backward()
        return loss, preds

    def reset():
        loss_fn._prototypes._prototypes_tensors.copy_(protos0)
        loss_fn._prototypes._count_features.copy_(counts0)

    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        step()
    torch.cuda.current_stream().wait_stream(s)
    torch.cuda.synchronize()
    reset()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        gl, gp = step()
    reset()
    g.replay()
    torch.cuda.synchronize()
    graph_loss, graph_preds = float(gl), gp.clone()
    graph_grad = leaves["logits"].grad.clone()
    graph_protos = loss_fn._prototypes._prototypes_tensors.clone()
    reset()
    eager_loss, eager_preds = step()
    assert graph_loss == float(eager_loss)
    assert torch.equal(graph_preds, eager_preds)
    assert torch.equal(graph_grad, leaves["logits"].grad)
    assert torch.equal(graph_protos, loss_fn._prototypes._prototypes_tensors)
    reset()
    torch.cuda.set_sync_debug_mode("error")
    try:
        step()
    finally:
        torch.cuda.set_sync_debug_mode(0)
