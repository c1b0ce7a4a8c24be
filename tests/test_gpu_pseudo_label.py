"""GPU tests of the pseudo-labelled background (bacs_loss.py:205-210): labels[labels == 0] = argmax_c teacher, in place.

* Full-resolution teacher: exactly torch.where(mask == 0, teacher.float().argmax(1), mask), ties included (teacher
  values drawn from a few integers), at every storage type, odd and unaligned sizes, and a misaligned teacher view.
* Low-res teacher: exactly the preds of the fused low-res loss kernel at the same sem_logits where the label is 0, and
  torch's F.interpolate + argmax except at fp32 near-ties.
* The whole BACSLoss step with pseudo_label=True in both data flows against the same step fed the pre-rewritten mask,
  and its capture in a CUDA graph (the torch form synchronised twice and could not be captured)."""
import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu

DTYPES = {"f32": torch.float32, "bf16": torch.bfloat16, "f16": torch.float16}


@pytest.fixture(scope="module")
def ops():
    from bacs_b200 import ops as _ops
    return _ops


@pytest.fixture(scope="module")
def cabi():
    from bacs_b200 import _cabi
    return _cabi


def _label_sets(B, H, W, K, seed):
    """mixed (0, classes, 255, negative and out-of-range values), all 0, and no 0 at all"""
    g = torch.Generator().manual_seed(seed)
    u = torch.rand(B, H, W, generator=g)
    lab = torch.randint(1, 300, (B, H, W), generator=g)
    lab = torch.where(u < 0.5, torch.zeros_like(lab), lab)
    lab = torch.where((u > 0.8) & (u < 0.9), torch.full_like(lab, 255), lab)
    lab = torch.where(u > 0.97, torch.full_like(lab, -7), lab)
    no0 = torch.where(lab == 0, torch.full_like(lab, 255), lab)
    return {"mixed": lab, "all0": torch.zeros_like(lab), "no0": no0}


def _teacher(B, K, H, W, dtype, seed, offset=False):
    """logits from five integers (ties are common); `offset`: a view one element into its storage"""
    g = torch.Generator().manual_seed(seed)
    t = torch.randint(-2, 3, (B, K, H, W), generator=g).to(dtype).cuda()
    if offset:
        buf = torch.empty(t.numel() + 1, dtype=dtype, device="cuda")
        buf[1:].copy_(t.reshape(-1))
        t = buf[1:].view(B, K, H, W)
        assert t.data_ptr() % 16 != 0
    return t


# name: (B, H, W, teacher view off its 16-byte alignment)
SHAPES = {
    "odd-hw": (3, 37, 41, False),      # H*W odd
    "hw-not-8": (2, 30, 35, False),    # H*W even, not a multiple of 8
    "b1": (1, 64, 96, False),
    "b24": (24, 16, 24, False),
    "offset": (2, 32, 48, True),       # 2-byte (16-bit) / 4-byte (fp32) storage offset
}
KTS = [1, 2, 7, 20, 21, 101, 150, 255, 300]


@pytest.mark.parametrize("shape", list(SHAPES))
@pytest.mark.parametrize("Kt", KTS)
@pytest.mark.parametrize("dtype", list(DTYPES))
def test_full_resolution_matches_torch(ops, dtype, Kt, shape):
    B, H, W, offset = SHAPES[shape]
    seed = Kt * 100 + sum(map(ord, shape + dtype))
    teacher = _teacher(B, Kt, H, W, DTYPES[dtype], seed, offset)
    am = teacher.float().argmax(1)
    for kind, lab in _label_sets(B, H, W, Kt, seed).items():
        lab = lab.cuda()
        want = torch.where(lab == 0, am, lab)
        got = ops.pseudo_label_inplace(lab, teacher)
        assert got is lab
        assert torch.equal(lab, want), kind


def test_full_resolution_voc_size(ops):
    """VOC 15-1 at B=24, 512x512, K_t = 20, bf16 teacher; synthetic labels with background areas"""
    from bacs_b200 import synth
    cfg = synth.CONFIGS["voc15-1_b24"]
    g = torch.Generator().manual_seed(15)
    teacher = (torch.randn(cfg.B, 20, cfg.H, cfg.W, generator=g) * 2).to(torch.bfloat16).cuda()
    lab = synth.make_labels(cfg, g).cuda()
    want = torch.where(lab == 0, teacher.float().argmax(1), lab)
    ops.pseudo_label_inplace(lab, teacher)
    assert torch.equal(lab, want)


def test_non_contiguous_labels(ops):
    """a non-contiguous mask is rewritten in place through a contiguous copy, as the torch form rewrote it"""
    teacher = _teacher(2, 9, 24, 40, torch.float32, 3)
    base = _label_sets(2, 40, 24, 9, 4)["mixed"].cuda()
    lab = base.transpose(1, 2)
    assert not lab.is_contiguous()
    want = torch.where(lab == 0, teacher.argmax(1), lab)
    assert ops.pseudo_label_inplace(lab, teacher) is lab
    assert torch.equal(lab, want)


# name: (B, H, W, lh, lw, K_t): the geometries of test_gpu_lowres_geometry.py, the two exact forms, and ADE20K's
# 151 classes at lw = 128 (staging at one image row per CTA)
LOWRES = {
    "500x375-s16": (2, 500, 375, 32, 24, 21),
    "375x500-s16": (2, 375, 500, 24, 32, 21),
    "513x513-s16": (2, 513, 513, 33, 33, 21),
    "500x375-s8": (2, 500, 375, 63, 47, 21),
    "512x500-s16": (2, 512, 500, 32, 32, 21),
    "500x512-s16": (2, 500, 512, 32, 32, 21),
    "17x17-s16": (3, 17, 17, 2, 2, 21),
    "9x9-s16": (3, 9, 9, 1, 1, 21),
    "16x40-s16": (3, 16, 40, 1, 3, 21),
    "512x512-s16-exact": (2, 512, 512, 32, 32, 20),
    "256x192-s8-exact": (2, 256, 192, 32, 24, 20),
    "37x2048-k151": (1, 37, 2048, 3, 128, 151),
}


def _near_tie_only(got_am, up, where):
    """pixels (inside `where`) whose arg-max differs from torch's: only where the fp32 top-2 gap is <= 1e-5 max|v|"""
    top2 = up.topk(2, dim=1)[0]
    gap = top2[:, 0] - top2[:, 1]
    tie = gap <= 1e-5 * up.abs().amax(1)
    diff = (got_am != up.argmax(1)) & where
    assert int((diff & ~tie).sum()) == 0, "arg-max differs from torch away from near-ties at %d pixels" % int(diff.sum())
    return int(diff.sum())


@pytest.mark.parametrize("dtype", list(DTYPES))
@pytest.mark.parametrize("geom", list(LOWRES))
def test_lowres_matches_loss_kernel_preds(ops, cabi, geom, dtype):
    B, H, W, lh, lw, Kt = LOWRES[geom]
    seed = sum(map(ord, geom + dtype))
    g = torch.Generator().manual_seed(seed)
    sem = (torch.randn(B, Kt, lh, lw, generator=g) * 3).to(DTYPES[dtype]).cuda()
    preds = ops.pixel_loss(sem, torch.zeros(B, H, W, dtype=torch.int64, device="cuda"), cabi.PIX_CE, want_grad=False,
                           lowres=True)["preds"]
    up = F.interpolate(sem.float(), size=(H, W), mode="bilinear", align_corners=False)
    for kind, lab in _label_sets(B, H, W, Kt, seed).items():
        lab = lab.cuda()
        want = torch.where(lab == 0, preds, lab)
        bg = lab == 0
        ops.pseudo_label_inplace(lab, sem, lowres=True)
        assert torch.equal(lab, want), kind
        n = _near_tie_only(torch.where(bg, lab, up.argmax(1)), up, bg)
        print("pseudo lowres %s %s %s: %d of %d background pixels differ from F.interpolate + argmax (near-ties)"
              % (geom, dtype, kind, n, int(bg.sum())))


@pytest.mark.parametrize("H,W,lh,lw,Kt", [(500, 375, 31, 24, 21), (513, 513, 32, 32, 21), (32, 32, 8, 8, 5),
                                          (512, 512, 32, 32, 256), (480, 480, 20, 20, 21)])
def test_lowres_unsupported_leaves_labels(ops, cabi, H, W, lh, lw, Kt):
    sem = torch.randn(1, Kt, lh, lw, device="cuda")
    lab = _label_sets(1, H, W, Kt, 7)["mixed"].cuda()
    before = lab.clone()
    with pytest.raises(cabi.BacsError):
        ops.pseudo_label_inplace(lab, sem, lowres=True)
    torch.cuda.synchronize()
    assert torch.equal(lab, before)


# ---- the whole step ------------------------------------------------------------------------------------------------
def _step(fused, teacher, seed=5, pseudo=True, mask=None):
    """BACSLoss(bg_weighted_ce=False) on the 'small' config with the teacher's logits (full-res [B,K_t,H,W], or
    sem_logits [B,K_t,h,w] when `fused`) registered on loss_fn.prev_model; `mask` replaces the batch's labels"""
    from bacs_b200 import synth
    cfg = synth.CONFIGS["small"]
    inp = synth.make_step_inputs(cfg, seed=seed)
    loss_fn, net, batch, leaves = synth.build_bacs_step(cfg, inp, bg_weighted_ce=False, pseudo_label=pseudo,
                                                        fused_logit_upsample=fused)
    img = batch["main"][0]
    if mask is not None:
        batch["main"][1].copy_(mask)
    prev = loss_fn.prev_model
    if fused:
        g = torch.Generator().manual_seed(seed + 1)
        sem = (torch.randn(cfg.B, cfg.K, cfg.h, cfg.w, generator=g) * 2).cuda().requires_grad_(True)
        rsem = (torch.randn(cfg.Br, cfg.K, cfg.h, cfg.w, generator=g) * 2).cuda().requires_grad_(True)
        net.register_sem(img, sem)
        net.register_sem(batch["buffer"][0], rsem)
        leaves.update(sem=sem, rsem=rsem)
        prev.register_sem(img, teacher)
    else:
        _, pen, atts = prev(img, return_penultimate=True, return_attentions=True)
        prev.register(img, teacher, pen, atts)
    return cfg, loss_fn, net, batch, leaves


def _teacher_for(fused, seed=9):
    from bacs_b200 import synth
    cfg = synth.CONFIGS["small"]
    g = torch.Generator().manual_seed(seed)
    h, w = (cfg.h, cfg.w) if fused else (cfg.H, cfg.W)
    return (torch.randn(cfg.B, cfg.old_cl, h, w, generator=g) * 2).cuda()    # K_t = old_cl != K


def _expected_mask(ops, cabi, mask, teacher, fused):
    if fused:
        am = ops.pixel_loss(teacher, torch.zeros_like(mask), cabi.PIX_CE, want_grad=False, lowres=True)["preds"]
    else:
        am = teacher.float().argmax(1)
    return torch.where(mask == 0, am, mask)


@pytest.mark.parametrize("fused", [False, True], ids=["reference-flow", "fused-flow"])
def test_step_matches_prerewritten_mask(ops, cabi, fused):
    teacher = _teacher_for(fused)
    cfg, loss_fn, net, batch, leaves = _step(fused, teacher)
    mask = batch["main"][1]
    want_mask = _expected_mask(ops, cabi, mask.clone(), teacher, fused)
    assert int((want_mask != mask).sum()) > 0
    loss, preds = loss_fn.compute_loss(batch, net, train=True)
    loss.backward()
    assert torch.equal(batch["main"][1], want_mask)

    cfg, loss_r, net_r, batch_r, leaves_r = _step(fused, teacher, pseudo=False, mask=want_mask)
    loss_w, preds_w = loss_r.compute_loss(batch_r, net_r, train=True)
    loss_w.backward()
    assert float(loss) == float(loss_w)
    assert torch.equal(preds, preds_w)
    # (prototype sums and some gradients are accumulated with atomics: equal up to the summation order)
    for got, want, what in [(loss_fn.prototypes, loss_r.prototypes, "prototypes"),
                            (loss_fn._prototypes._count_features, loss_r._prototypes._count_features, "counts")] + \
            [(leaves[k].grad, leaves_r[k].grad, "d" + k) for k in sorted(leaves)]:
        if want is None:
            assert got is None, what
            continue
        atol = 1e-6 * float(want.abs().max())
        assert torch.allclose(got, want, rtol=0, atol=atol), "%s %.3e" % (what, float((got - want).abs().max()))
    if not fused:
        assert torch.equal(leaves["logits"].grad, leaves_r["logits"].grad)


@pytest.mark.parametrize("fused", [False, True], ids=["reference-flow", "fused-flow"])
def test_step_is_free_of_host_sync(ops, cabi, fused):
    """with pseudo_label=True the step captures in a CUDA graph, and replay equals eager bit for bit (recipe of
    test_gpu_step.py::test_step_is_free_of_host_sync; the mask is restored before every run, the step rewrites it);
    an eager step also runs under torch.cuda.set_sync_debug_mode("error"), which the step without pseudo labels passes"""
    teacher = _teacher_for(fused)
    cfg, loss_fn, net, batch, leaves = _step(fused, teacher)
    mask = batch["main"][1]
    mask0 = mask.clone()
    want_mask = _expected_mask(ops, cabi, mask0, teacher, fused)
    protos0 = loss_fn._prototypes._prototypes_tensors.clone()
    counts0 = loss_fn._prototypes._count_features.clone()
    grad_key = "sem" if fused else "logits"

    def step():
        for v in leaves.values():
            v.grad = None
        loss, preds = loss_fn.compute_loss(batch, net, train=True)
        loss.backward()
        return loss, preds

    def reset():
        loss_fn._prototypes._prototypes_tensors.copy_(protos0)
        loss_fn._prototypes._count_features.copy_(counts0)
        mask.copy_(mask0)

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
    graph_loss, graph_preds, graph_mask = float(gl), gp.clone(), mask.clone()
    graph_grad = leaves[grad_key].grad.clone()
    assert torch.equal(graph_mask, want_mask)
    reset()
    eager_loss, eager_preds = step()
    assert graph_loss == float(eager_loss)
    assert torch.equal(graph_preds, eager_preds)
    assert torch.equal(mask, graph_mask)
    if fused:   # (d sem_logits: fp32 atomics, equal up to the summation order)
        w = leaves[grad_key].grad
        assert torch.allclose(graph_grad, w, rtol=0, atol=1e-6 * float(w.abs().max()))
    else:
        assert torch.equal(graph_grad, leaves[grad_key].grad)
    reset()
    torch.cuda.set_sync_debug_mode("error")
    try:
        step()
    finally:
        torch.cuda.set_sync_debug_mode(0)
    assert torch.equal(mask, want_mask)
