"""Pins oracle/bacs_oracle.py against the *imported* reference code (CPU, fp32).

The tests marked ``reference`` import the upstream BACS code and run only where its source tree
is found (tests/golden/ref_shim.py).  Of what they check, only the reference's outputs for the
full step at the ``tiny`` shape, the label remap, the class -> task map of five class splits and
the IoU vector are stored (tests/golden/*.npz, checked by test_golden.py); the rest is checked
nowhere else.  The other tests compare with PyTorch's own ops and run everywhere."""
import math
import warnings

import numpy as np
import pytest
import torch

import ref_shim
from fake_net import FakeNet
from oracle import bacs_oracle as O
from bacs_b200 import synth


@pytest.fixture(scope="module")
def ref():
    if not ref_shim.reference_available():
        pytest.skip("upstream BACS source tree not found (set BACS_REFERENCE_ROOT)")
    warnings.filterwarnings("ignore")
    return ref_shim.install()


def _close(a, b, rtol=1e-5, atol=None):
    a = torch.as_tensor(a).double()
    b = torch.as_tensor(b).double()
    if atol is None:
        atol = 1e-6 * max(1.0, float(b.abs().max()))
    assert torch.allclose(a, b, rtol=rtol, atol=atol), float((a - b).abs().max())


class _Accel:
    root_device = torch.device("cpu")


def _ref_loss(ref, cfg, **kw):
    L = ref["loss.bacs_loss"].BACSLoss(name="ref", bg_weighted_ce=True, **kw)
    L.init_prototype_compute()
    L.set_continual_task_size(cfg.initial_classes, cfg.increment)
    return L


def _ref_seen_net(ref, inp):
    cfg = inp.cfg
    bg = ref["networks.bg_detector"].BgDetector(cfg.D * 4)
    heads = torch.nn.ModuleList([bg.get_classification_head(1) for _ in range(cfg.T)])
    with torch.no_grad():
        for t, head in enumerate(heads):
            head.conv.weight.copy_(inp.head_w[t].view(1, cfg.D, 1, 1))
            head.conv.bias.copy_(inp.head_b[t].view(1))
    bg.seen_not_seen_clf = heads
    return bg


def test_label_downsample_matches_interpolate():
    for (H, W, h, w) in [(512, 512, 32, 32), (528, 528, 33, 33), (513, 513, 33, 33), (64, 96, 4, 6), (100, 75, 7, 5)]:
        t = torch.randint(0, 256, (2, H, W))
        want = torch.nn.functional.interpolate(t.unsqueeze(1).double(), size=(h, w), mode="nearest").long()[:, 0]
        assert torch.equal(O.downsample_labels(t, h, w), want)


@pytest.mark.reference
def test_class_to_task_matches(ref):
    for init, inc in [(16, 1), (16, 5), (11, 1), (101, 50), (15, 2), (20, 0)]:
        L = ref["loss.base_loss"].BaseLoss("x")
        L.set_continual_task_size(init, inc)
        labels = torch.arange(0, 255)
        want = L.label_to_task_num(labels)
        got = O.class_to_task(labels.numpy(), init, inc)
        assert np.array_equal(np.broadcast_to(np.asarray(want).astype(np.int64), got.shape), got), (init, inc)


@pytest.mark.reference
@pytest.mark.parametrize("name,B", [("tiny", 1), ("tiny", 2), ("small", 3)])
def test_prototype_update_matches(ref, name, B):
    cfg = synth.CONFIGS[name]
    inp = synth.make_step_inputs(cfg, seed=3)
    P = ref["loss.prototypes"].Prototypes()
    P.set_continual_task_size(cfg.initial_classes, cfg.increment)
    for t in range(cfg.T):
        P._init_prototypes(t, _Accel(), cfg.D)
    # labels from several tasks so several prototype rows move
    gen = torch.Generator().manual_seed(5)
    mask = synth.make_labels(cfg, gen, classes=list(range(1, cfg.K)), B=B)
    pen = inp.pen[:B]
    protos = torch.zeros(cfg.T, cfg.D)
    counts = P._count_features.clone()
    assert counts.dtype == torch.float32            # Q3: float after the first cat
    for step in range(2):
        P.update_feats_prototypes(pen, mask)
        sums, n = O.proto_accumulate(pen, mask, cfg.initial_classes, cfg.increment, cfg.T, mode="exact")
        protos, counts = O.proto_update(protos, counts, sums, n)
        _close(protos, P._prototypes_tensors)
        _close(counts, P._count_features)
        assert O.prototypes_ready(counts) == bool(P.are_prototypes_ready())
    if B == 1:
        s2, _ = O.proto_accumulate(pen, mask, cfg.initial_classes, cfg.increment, cfg.T, mode="channel")
        _close(s2, sums)


@pytest.mark.reference
def test_seen_probs_match(ref):
    inp = synth.make_step_inputs(synth.CONFIGS["tiny"], seed=1)
    bg = _ref_seen_net(ref, inp)
    want = bg.get_seen_probs(inp.pen, inp.protos, bg_detect=True)
    got = O.seen_probs(inp.pen, inp.protos, inp.head_w, inp.head_b)
    _close(got, want)
    want_t = bg.get_seen_map_task(inp.pen, inp.protos, 1)
    z = O.seen_logits_lowres(inp.pen, inp.protos[1:2], inp.head_w[1:2], inp.head_b[1:2])
    _close(O.bilinear_upsample(z, want_t.shape[-2:], True), want_t)


def test_bilinear_matches_interpolate():
    x = torch.randn(2, 3, 5, 7)
    for ac in (True, False):
        want = torch.nn.functional.interpolate(x, size=(80, 112), mode="bilinear", align_corners=ac)
        _close(O.bilinear_upsample(x, (80, 112), ac), want)
    up = torch.nn.Upsample(scale_factor=16, mode="bilinear", align_corners=True)
    _close(O.bilinear_upsample(x, (80, 112), True), up(x))


@pytest.mark.parametrize("shape,stride", [((2, 7, 4, 6), 16), ((1, 21, 33, 33), 16), ((2, 5, 8, 10), 8)])
def test_upsample_sem_logits_matches_network_op(shape, stride):
    """networks/deeplab_v3.py:157-160: F.interpolate(sem_logits, size=input_shape, mode="bilinear",
    align_corners=False) -- values and the gradient autograd sends back to sem_logits (oracle of the fused low-res path)"""
    g = torch.Generator().manual_seed(shape[1])
    x = torch.randn(*shape, generator=g)
    out_hw = (shape[2] * stride, shape[3] * stride)
    upstream = torch.randn(shape[0], shape[1], *out_hw, generator=g)
    a = x.clone().requires_grad_(True)
    want = torch.nn.functional.interpolate(a, size=out_hw, mode="bilinear", align_corners=False)
    want.backward(upstream)
    b = x.clone().requires_grad_(True)
    got = O.upsample_sem_logits(b, out_hw)
    got.backward(upstream)
    _close(got, want)
    _close(b.grad, a.grad, atol=1e-5 * float(a.grad.abs().max()))


@pytest.mark.reference
@pytest.mark.parametrize("ukd", [True, False])
@pytest.mark.parametrize("name", ["tiny", "small"])
def test_weighted_ce_matches(ref, name, ukd):
    cfg = synth.CONFIGS[name]
    inp = synth.make_step_inputs(cfg, seed=2)
    gen = torch.Generator().manual_seed(9)
    mask = synth.make_labels(cfg, gen, classes=list(range(1, cfg.K)))
    seen = torch.rand(cfg.B, cfg.T, cfg.H, cfg.W, generator=gen)
    W = ref["training.loss_utils"].WeightedCrossEntropy(gamma=2, old_cl=cfg.old_cl, threshold=0.5, ukd=ukd)
    x1 = inp.logits.clone().requires_grad_(True)
    want = W(x1, mask, seen, 0)
    want.backward()
    x2 = inp.logits.clone().requires_grad_(True)
    got = O.weighted_ce(x2, mask, seen.max(1)[0], cfg.old_cl, 2.0, 0.5, ukd)
    got.backward()
    _close(got, want)
    _close(x2.grad, x1.grad, atol=1e-6 * float(x1.grad.abs().max()))


def _cross_entropy_case():
    cfg = synth.CONFIGS["small"]
    inp = synth.make_step_inputs(cfg, seed=4)
    gen = torch.Generator().manual_seed(2)
    mask = synth.make_labels(cfg, gen, classes=list(range(1, cfg.K)))
    return cfg, inp, gen, mask


def test_cross_entropy_matches_torch():
    cfg, inp, _, mask = _cross_entropy_case()
    F = torch.nn.functional
    w = torch.zeros(cfg.K)
    w[1:cfg.old_cl] = 1
    _close(O.cross_entropy(inp.logits, mask), F.cross_entropy(inp.logits, mask, ignore_index=255))
    _close(O.cross_entropy(inp.logits, mask, w), F.cross_entropy(inp.logits, mask, ignore_index=255, weight=w))
    w2 = torch.ones(cfg.K)
    w2[0] = 0
    want = -1 * F.cross_entropy(inp.logits, mask, ignore_index=255, weight=w2, reduction="none").view(cfg.B, -1).mean(1)
    _close(O.cross_entropy_per_image_score(inp.logits, mask, w2), want)


@pytest.mark.reference
def test_cross_entropy_variants_match(ref):
    cfg, inp, gen, mask = _cross_entropy_case()
    U = ref["training.loss_utils"].UnbiasedCrossEntropy(old_cl=cfg.old_cl)
    _close(O.unbiased_ce(inp.logits, mask, cfg.old_cl), U(inp.logits, mask))
    KD = ref["training.loss_utils"].UnbiasedKnowledgeDistillationLoss(alpha=1.0)
    old = torch.randn(cfg.B, cfg.old_cl, cfg.H, cfg.W, generator=gen)
    _close(O.unbiased_kd(inp.logits, old), KD(inp.logits, old))
    pm = mask == 0
    _close(O.unbiased_kd(inp.logits, old, mask=pm), KD(inp.logits, old, mask=pm))


@pytest.mark.reference
@pytest.mark.parametrize("with_seen", [True, False])
def test_teacher_distill_matches(ref, with_seen):
    cfg = synth.CONFIGS["tiny"]
    inp = synth.make_step_inputs(cfg, seed=6)
    L = _ref_loss(ref, cfg)
    gen = torch.Generator().manual_seed(1)
    seen = torch.rand(cfg.B, cfg.T, cfg.H, cfg.W, generator=gen) if with_seen else None
    n1 = inp.new_att.clone().requires_grad_(True)
    want = L._teacher_distill([inp.old_att], [n1], seen, inp.mask)
    want.backward()
    n2 = inp.new_att.clone().requires_grad_(True)
    got = O.teacher_distill(inp.old_att, n2, inp.mask, None if seen is None else seen.max(1)[0])
    got.backward()
    _close(got, want)
    _close(n2.grad, n1.grad, atol=1e-6 * float(n1.grad.abs().max()))


@pytest.mark.reference
def test_der_mse_matches(ref):
    cfg = synth.CONFIGS["tiny"]
    for seed, ncls in [(0, [5, 6]), (1, [7, 7]), (2, [4, 7])]:
        inp = synth.make_step_inputs(cfg, seed=seed)
        rp = inp.replay
        n_classes = torch.tensor(ncls, dtype=torch.uint8)
        L = _ref_loss(ref, cfg)
        L._init_dark_criterion(torch.device("cpu"))
        L.logit_transforms = lambda x: x
        net = FakeNet()
        s1 = rp["sem_logits"].clone().requires_grad_(True)
        img = torch.zeros(cfg.Br, 3, 4, 4)
        net.register_sem(img, s1)
        mem = rp["memory_logits"].long()                 # preprocess_batch (Q4)
        want = L._dark_logits(net, (None, img, mem, None, n_classes, None))
        want.backward()
        s2 = rp["sem_logits"].clone().requires_grad_(True)
        got = O.der_mse(s2, rp["memory_logits"], n_classes.numpy())
        got.backward()
        _close(got, want)
        _close(s2.grad, s1.grad, atol=1e-7)


@pytest.mark.reference
def test_der_transplant_quirk_bigger_batch(ref):
    # Br=5 with repeated class counts: exercises the sample-index-vs-mask quirk (Q5)
    K, Br = 9, 5
    gen = torch.Generator().manual_seed(3)
    cfg = synth.CONFIGS["tiny"]
    L = _ref_loss(ref, cfg)
    L._init_dark_criterion(torch.device("cpu"))
    L.logit_transforms = lambda x: x
    for ncls in ([6, 6, 8, 7, 9], [9, 9, 9, 9, 9], [5, 6, 7, 8, 9], [8, 5, 5, 8, 6]):
        s = torch.randn(Br, K, 4, 4, generator=gen)
        m = (torch.randn(Br, K, 4, 4, generator=gen) * 2)
        net = FakeNet()
        img = torch.zeros(Br, 3, 4, 4)
        net.register_sem(img, s)
        want = L._dark_logits(net, (None, img, m.long(), None, torch.tensor(ncls, dtype=torch.uint8), None))
        got = O.der_mse(s, m, np.array(ncls))
        _close(got, want)


@pytest.mark.reference
def test_focal_seen_loss_matches(ref):
    cfg = synth.CONFIGS["tiny"]
    inp = synth.make_step_inputs(cfg, seed=8)
    for alpha in (None, 0.25):
        L = _ref_loss(ref, cfg, seen_focal_alpha=alpha)
        bg = _ref_seen_net(ref, inp)
        net = FakeNet(bg)
        L._prototypes._prototypes_tensors = inp.protos.clone()
        L._prototypes._count_features = inp.counts.clone()
        L.first_task = False
        want = L._compute_seen_fg_loss(inp.pen, inp.mask, net, task_num=1)
        z = O.seen_logits_lowres(inp.pen, inp.protos[1:2], inp.head_w[1:2], inp.head_b[1:2])
        zf = O.bilinear_upsample(z, (cfg.H, cfg.W), True)
        _close(O.focal_seen_loss(zf, inp.mask, 2.0, alpha), want)
    no_bg = torch.where(inp.mask == 0, torch.full_like(inp.mask, 255), inp.mask)
    assert L._compute_seen_fg_loss(inp.pen, no_bg, net, task_num=1) == 0
    assert float(O.focal_seen_loss(zf, no_bg)) == 0.0


def test_confmat_known_answer():
    # the reference's only known-answer vector: training/metrics.py:159-183
    label = np.zeros((1, 4, 4), dtype=np.int64)
    pred = np.zeros((1, 4, 4), dtype=np.float32)
    label[:, :3, :3] = 1
    pred[:, -3:, -3:] = 1
    C = O.confusion_matrix(pred, label, 2)
    assert C.tolist() == [[2, 5], [5, 4]]
    m = O.iou_metrics(C)
    assert np.allclose(m["iou_per_class"], [2.0 / 12, 4.0 / 14], atol=1e-6)


@pytest.mark.reference
def test_transform_label_sequential(ref):
    TL = __import__("training.utils", fromlist=["TransformLabel"]).TransformLabel
    rng = np.random.RandomState(0)
    for trial in range(20):
        keys = rng.choice(34, size=12, replace=False)
        d1 = {int(k): int(rng.randint(0, 20)) for k in keys}
        d2 = {int(k): int(v) for k, v in zip(rng.choice(20, 6, replace=False), rng.randint(0, 8, 6))}
        d2[255] = 255
        lbl = torch.from_numpy(rng.randint(0, 34, size=(16, 16)).astype(np.int64))
        want = TL(d1, 255, d2, 0)(lbl.clone())
        got = O.transform_label(lbl.numpy(), d1, 255, d2, 0)
        assert np.array_equal(got, want.numpy())
        present = np.zeros(256, dtype=bool)
        present[np.unique(lbl.numpy())] = True
        lut1 = O.effective_sequential_lut(present, d1, 255, 0, 256)
        mid = lut1[lbl.numpy()]
        present2 = np.zeros(256, dtype=bool)
        present2[np.unique(mid)] = True
        lut2 = O.effective_sequential_lut(present2, d2, 0, 0, 256)
        assert np.array_equal(lut2[mid], want.numpy())


@pytest.mark.reference
@pytest.mark.parametrize("name,first_task", [("tiny", False), ("tiny", True), ("small", False)])
def test_full_step_matches(ref, name, first_task):
    cfg = synth.CONFIGS[name]
    inp = synth.make_step_inputs(cfg, seed=11)
    task_num = cfg.T - 1
    L = _ref_loss(ref, cfg)
    for t in range(cfg.T):
        L._prototypes._init_prototypes(t, _Accel(), cfg.D)
    L._prototypes._prototypes_tensors = inp.protos.clone()
    L._prototypes._count_features = inp.counts.clone()
    L._update_task(task_num)
    L.old_classes, L.nb_current_classes = cfg.old_cl, cfg.K
    L.first_task = first_task
    L._use_der_loss = True
    L.set_device(torch.device("cpu"))
    L._init_dark_criterion(torch.device("cpu"))
    L.logit_transforms = lambda x: x
    L.on_train_batch_start(epoch=3, max_epochs=30, batch_idx=0)
    bg = _ref_seen_net(ref, inp)
    net, prev = FakeNet(bg), FakeNet(bg)
    leaf = lambda t: t.clone().requires_grad_(True)
    lg, pn, na = leaf(inp.logits), leaf(inp.pen), leaf(inp.new_att)
    rp = inp.replay
    rlg, rsem = leaf(rp["logits"]), leaf(rp["sem_logits"])
    img, rimg, limg = torch.zeros(cfg.B, 3, 2, 2), torch.zeros(cfg.Br, 3, 2, 2), torch.zeros(cfg.Br, 3, 2, 2)
    net.register(img, lg, pn, [na])
    net.register(rimg, rlg, rp["pen"], [na])
    net.register_sem(limg, rsem)
    prev.register(img, inp.logits, inp.pen, [inp.old_att])
    L.prev_model = prev
    batch = {"main": [img, inp.mask.clone()], "buffer": [rimg, rp["mask"].clone()],
             "bufferlogits": [limg, rp["memory_logits"].clone(), rp["n_classes"]]}
    batch = L.preprocess_batch(batch)
    batch["main"][0], batch["buffer"][0], batch["bufferlogits"][0] = img, rimg, limg  # keep ids
    want, want_preds = L.compute_loss(batch, net, train=True)
    want.backward()

    hw = [leaf(inp.head_w), leaf(inp.head_b)]
    lg2, pn2, na2, rlg2, rsem2 = leaf(inp.logits), leaf(inp.pen), leaf(inp.new_att), leaf(rp["logits"]), leaf(rp["sem_logits"])
    rp2 = dict(rp, logits=rlg2, sem_logits=rsem2, n_classes=rp["n_classes"].numpy())
    out = O.bacs_step(lg2, pn2, inp.old_att, na2, inp.mask, inp.protos, inp.counts, hw[0], hw[1],
                      initial_classes=cfg.initial_classes, increment=cfg.increment, old_cl=cfg.old_cl,
                      task_num=task_num, first_task=first_task, epoch=3, max_epochs=30, replay=rp2,
                      nb_current_classes=cfg.K)
    out["loss"].backward()
    _close(out["loss"], want)
    assert torch.equal(out["preds"], want_preds)
    _close(out["protos"], L.prototypes)
    _close(out["counts"], L._prototypes._count_features)
    _close(lg2.grad, lg.grad, atol=1e-6 * float(lg.grad.abs().max()))
    _close(na2.grad, na.grad, atol=1e-6 * float(na.grad.abs().max()))
    _close(rlg2.grad, rlg.grad, atol=1e-6 * float(rlg.grad.abs().max()))
    _close(rsem2.grad, rsem.grad, atol=1e-6 * float(rsem.grad.abs().max()))
    head = bg.seen_not_seen_clf[task_num]
    _close(hw[0].grad[task_num], head.conv.weight.grad.view(-1), atol=1e-6 * float(head.conv.weight.grad.abs().max()))
    _close(hw[1].grad[task_num], head.conv.bias.grad.view(()), atol=1e-7)
    if first_task:
        _close(pn2.grad, pn.grad, atol=1e-6 * float(pn.grad.abs().max()))
    else:
        assert pn.grad is None or float(pn.grad.abs().max()) == 0.0
