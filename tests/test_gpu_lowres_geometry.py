"""GPU parity of the fused low-res path at inputs that are not a multiple of the output stride: lh = ceil(H / s),
lw = ceil(W / s) for s = 16 or 8 (a DeepLab backbone's padded stride-2 convolutions), and wide maps whose staging
only fits at one image row per CTA.

Reference: the reference's data flow, torch's F.interpolate(sem, size=(H, W), mode="bilinear", align_corners=False)
feeding the full-resolution kernel (ops.pixel_loss, whose parity with the oracle is pinned elsewhere); the gradient
reference is torch's interpolate backward of that kernel's dlogits.  Tolerances: loss 1e-5 relative, d sem_logits
2e-5 of max |grad| (one storage ulp of max |grad| for 16-bit logits), pixel counts exact, arg-max identical except
at fp32 near-ties.  Every output pixel is checked: before each fused call the outputs' blocks are pre-filled with a
sentinel through the caching allocator, so a pixel no thread writes reads back as the sentinel."""
import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu

RTOL = 1e-5
K = 21
OLD_CL = 11
SENTINEL = 0xA5

# name: (B, H, W, lh, lw)
GEOMETRIES = {
    "500x375-s16": (2, 500, 375, 32, 24),
    "375x500-s16": (2, 375, 500, 24, 32),
    "513x513-s16": (2, 513, 513, 33, 33),
    "500x375-s8": (2, 500, 375, 63, 47),
    "512x500-s16": (2, 512, 500, 32, 32),     # exact in y, ceil in x
    "500x512-s16": (2, 500, 512, 32, 32),     # ceil in y, exact in x
    "17x17-s16": (3, 17, 17, 2, 2),           # short, uneven spans; both borders clamped
    "9x9-s16": (3, 9, 9, 1, 1),               # lh = lw = 1: one column owns the whole row
    "16x40-s16": (3, 16, 40, 1, 3),
}
MODES = ["ce", "ce_fwd", "ce_weighted", "unbiased_ce", "score", "weighted_ce_seen_max", "ce_distill_mask"]
DTYPES = {"f32": torch.float32, "bf16": torch.bfloat16, "f16": torch.float16}


@pytest.fixture(scope="module")
def ops():
    from bacs_b200 import ops as _ops
    return _ops


@pytest.fixture(scope="module")
def cabi():
    from bacs_b200 import _cabi
    return _cabi


def close(got, want, rtol=RTOL, atol=None, what=""):
    got = torch.as_tensor(got).detach().double().cpu()
    want = torch.as_tensor(want).detach().double().cpu()
    if atol is None:
        atol = rtol * max(1e-30, float(want.abs().max()))
    err = float((got - want).abs().max()) if got.numel() else 0.0
    assert torch.allclose(got, want, rtol=rtol, atol=atol), "%s max abs err %.3e (atol %.3e)" % (what, err, atol)


def _labels(B, H, W, seed):
    """~30 % background, ~10 % ignored, a few out-of-range labels (counted as invalid), the rest uniform."""
    g = torch.Generator().manual_seed(seed)
    lab = torch.randint(1, K, (B, H, W), generator=g)
    u = torch.rand(B, H, W, generator=g)
    lab = torch.where(u < 0.3, torch.zeros_like(lab), lab)
    lab = torch.where(u > 0.9, torch.full_like(lab, 255), lab)
    lab = torch.where(u > 0.997, torch.full_like(lab, K + 3), lab)
    lab[0, 0, 0] = 255                           # a border pixel of each kind
    lab[0, 0, W - 1] = 0
    lab[-1, H - 1, W - 1] = K - 1
    return lab


def _sentinel_outputs(sem, B, H, W, want_grad, want_preds, want_mask, want_score):
    """Allocate blocks of the sizes ops.pixel_loss allocates, in its order, fill them with the sentinel and free them;
    returns the data pointers of the preds / distill-mask / score blocks."""
    dev = sem.device
    sizes = []
    if want_grad:
        sizes.append(("dlogits", sem.numel() * sem.element_size()))
    if want_preds:
        sizes.append(("preds", B * H * W * 8))
    sizes.append(("acc", 8 * 8))
    if want_mask:
        sizes.append(("distill_mask", B * H * W))
    if want_score:
        sizes.append(("score", B * 8))
    blocks = [(name, torch.full((n,), SENTINEL, dtype=torch.uint8, device=dev)) for name, n in sizes]
    ptrs = {name: t.data_ptr() for name, t in blocks}
    del blocks
    return ptrs


def _check_preds(preds, full):
    """identical except where the two largest up-sampled logits are within fp32 rounding"""
    want = full.argmax(1)
    top2 = full.topk(2, dim=1)[0]
    gap = top2[:, 0] - top2[:, 1]
    diff = preds != want
    tie = gap <= 1e-6 * top2[:, 0].abs().clamp_min(1.0)
    assert int((diff & ~tie).sum()) == 0, "arg-max differs away from near-ties (%d pixels)" % int(diff.sum())


def _mode_kwargs(cabi, mode, B, H, W, dev, seed):
    g = torch.Generator().manual_seed(seed + 100)
    if mode in ("ce", "ce_fwd"):
        return cabi.PIX_CE, dict(want_grad=mode == "ce")
    if mode == "ce_weighted":
        w = torch.rand(K, generator=g) + 0.5
        w[3] = 0.0
        return cabi.PIX_CE, dict(want_grad=True, class_w=w.to(dev))
    if mode == "unbiased_ce":
        return cabi.PIX_UNBIASED_CE, dict(want_grad=True, old_cl=OLD_CL)
    if mode == "score":
        w = torch.ones(K)
        w[0] = 0.0
        return cabi.PIX_SCORE, dict(want_grad=False, class_w=w.to(dev), want_score=True)
    if mode == "weighted_ce_seen_max":
        smax = torch.rand(B, H, W, generator=g).to(dev)
        return cabi.PIX_WEIGHTED_CE, dict(want_grad=True, seen_max=smax, old_cl=OLD_CL, want_distill_mask=True)
    if mode == "ce_distill_mask":
        return cabi.PIX_CE, dict(want_grad=True, want_distill_mask=True, lkd_threshold=-1.0)
    raise ValueError(mode)


def _compare(ops, cabi, sem, labels, mode_id, kw, grad_scale=1.0):
    """the fused call against torch's up-sample + the full-resolution kernel (+ the up-sample's backward)"""
    B, lh, lw = sem.shape[0], sem.shape[2], sem.shape[3]
    H, W = labels.shape[1], labels.shape[2]
    want_grad = kw["want_grad"]
    x = sem.float().clone().requires_grad_(want_grad)
    full = F.interpolate(x, size=(H, W), mode="bilinear", align_corners=False)
    ref = ops.pixel_loss(full.detach(), labels, mode_id, grad_scale=grad_scale, **kw)
    if want_grad:
        full.backward(ref["dlogits"])
    torch.cuda.synchronize()
    ptrs = _sentinel_outputs(sem, B, H, W, want_grad, True, kw.get("want_distill_mask", False),
                             kw.get("want_score", False))
    out = ops.pixel_loss(sem, labels, mode_id, lowres=True, grad_scale=grad_scale, **kw)
    torch.cuda.synchronize()
    assert out["variant"] == 3
    # the outputs landed on the sentinel blocks (otherwise the coverage checks below would prove nothing)
    assert out["preds"].data_ptr() == ptrs["preds"]
    if out["distill_mask"] is not None:
        assert out["distill_mask"].data_ptr() == ptrs["distill_mask"]
    if out["score"] is not None:
        assert out["score"].data_ptr() == ptrs["score"]
    acc, racc = out["acc"].cpu(), ref["acc"].cpu()
    for i in (cabi.ACC_KEPT, cabi.ACC_VALID, cabi.ACC_BG, cabi.ACC_INVALID):
        assert float(acc[i]) == float(racc[i]), "pixel count %d: %s vs %s" % (i, float(acc[i]), float(racc[i]))
    close(acc[cabi.ACC_LOSS], racc[cabi.ACC_LOSS], what="loss")
    close(acc[cabi.ACC_WSUM], racc[cabi.ACC_WSUM], what="weight sum")
    _check_preds(out["preds"], full.detach())
    if out["distill_mask"] is not None:
        assert torch.equal(out["distill_mask"], ref["distill_mask"])
    if out["score"] is not None:
        close(out["score"], ref["score"], what="score")
    if want_grad:
        dt = sem.dtype
        wg = x.grad.to(dt).float()
        tol = {torch.float32: 2e-5, torch.bfloat16: 2.0 ** -7, torch.float16: 2.0 ** -10}[dt]
        assert out["dlogits"].dtype == dt and tuple(out["dlogits"].shape) == tuple(sem.shape)
        close(out["dlogits"].float(), wg, atol=tol * float(wg.abs().max()), what="d sem_logits")
    return out


@pytest.mark.parametrize("dtype", list(DTYPES))
@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("geom", list(GEOMETRIES))
def test_lowres_any_input_size(ops, cabi, geom, mode, dtype):
    B, H, W, lh, lw = GEOMETRIES[geom]
    dt = DTYPES[dtype]
    seed = sum(map(ord, geom + mode + dtype)) % 1000
    g = torch.Generator().manual_seed(seed)
    sem = (torch.randn(B, K, lh, lw, generator=g) * 3.0).to(dt).cuda()
    labels = _labels(B, H, W, seed + 1).cuda()
    mode_id, kw = _mode_kwargs(cabi, mode, B, H, W, sem.device, seed)
    _compare(ops, cabi, sem, labels, mode_id, kw, grad_scale=1024.0 if dt == torch.float16 else 1.0)


@pytest.mark.parametrize("W", [2040, 2048])
def test_lowres_wide_map_many_classes(ops, cabi, W):
    """ADE20K's 151 classes at lw = 128: the staging fits at one image row per CTA only (about 170 KB)"""
    B, H, Kw = 1, 37, 151
    lh, lw = (H + 15) // 16, (W + 15) // 16
    g = torch.Generator().manual_seed(W)
    sem = (torch.randn(B, Kw, lh, lw, generator=g) * 3.0).cuda()
    lab = torch.randint(0, Kw, (B, H, W), generator=g)
    lab[:, :, :5] = 255
    for mode_id, kw in ((cabi.PIX_CE, dict(want_grad=True)), (cabi.PIX_CE, dict(want_grad=False))):
        _compare(ops, cabi, sem, lab.cuda(), mode_id, kw)


def test_eval_step_through_bacs_loss(cabi):
    """BACSLoss(fused_logit_upsample=True).compute_loss(train=False) on an uncropped 500x375 batch: the same loss and
    arg-max as the unfused loss fed the up-sampled logits, and the same confusion matrix"""
    from bacs_b200 import synth
    from bacs_b200.training.metrics import IoU
    cfg = synth.StepConfig("eval500x375", B=2, K=K, old_cl=20, T=6, H=500, W=375, D=32, A=16)
    inp = synth.make_step_inputs(cfg, seed=4, with_replay=False)
    g = torch.Generator().manual_seed(6)
    sem = torch.randn(cfg.B, cfg.K, 32, 24, generator=g) * 3.0
    inp.logits = F.interpolate(sem.cuda(), size=(cfg.H, cfg.W), mode="bilinear", align_corners=False).cpu()
    results = {}
    for fused in (False, True):
        loss_fn, net, batch, _ = synth.build_bacs_step(cfg, inp, fused_logit_upsample=fused)
        if fused:
            net.register_sem(batch[0], sem.cuda())
        loss, preds = loss_fn.compute_loss(batch, net, train=False)
        iou = IoU(num_classes=cfg.K).cuda()
        iou.update(preds, batch[1])
        results[fused] = (loss.detach(), preds, iou.confmat.clone())
    (lu, pu, cu), (lf, pf, cf) = results[False], results[True]
    close(lf, lu, what="eval loss")
    _check_preds(pf, inp.logits.cuda())
    _check_preds(pu, inp.logits.cuda())
    assert torch.equal(pf, pu)
    assert torch.equal(cf, cu)


@pytest.mark.parametrize("H,W,lh,lw", [(32, 32, 8, 8), (500, 375, 31, 23), (500, 375, 31, 24), (500, 375, 32, 23),
                                         (513, 513, 32, 32)])
def test_lowres_still_rejects(ops, cabi, H, W, lh, lw):
    """neither W == s * lw (H a multiple of lh) nor lh == ceil(H / s), lw == ceil(W / s), s in {8, 16}"""
    sem = torch.randn(1, 5, lh, lw).cuda()
    lab = torch.zeros(1, H, W, dtype=torch.int64).cuda()
    with pytest.raises(cabi.BacsError):
        ops.pixel_loss(sem, lab, cabi.PIX_CE, want_grad=False, lowres=True)


def test_lowres_seen_logits_need_multiples_of_16(ops, cabi):
    """the seen heads z (focal term, weighted CE's seen probabilities) keep needing H, W = 16 h, 16 w"""
    sem = torch.randn(1, K, 32, 24).cuda()
    lab = torch.zeros(1, 500, 375, dtype=torch.int64).cuda()
    z = torch.randn(1, 2, 31, 23).cuda()
    with pytest.raises(cabi.BacsError):
        ops.pixel_loss(sem, lab, cabi.PIX_WEIGHTED_CE, want_grad=False, z=z, old_cl=OLD_CL, lowres=True)
    z = torch.randn(1, 2, 32, 24).cuda()          # x16 of the low-res map: still not the label size
    with pytest.raises(cabi.BacsError):
        ops.pixel_loss(sem, lab, cabi.PIX_WEIGHTED_CE, want_grad=False, z=z, old_cl=OLD_CL, focal_head=1,
                       lowres=True)
