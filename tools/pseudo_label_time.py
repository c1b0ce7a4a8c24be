"""Times the pseudo-labelled background (bacs_pseudo_label / bacs_pseudo_label_lowres, bacs_loss.py:205-210) next to
what it replaces.  CUDA events after warm-up; the card's name and power limit are printed with the numbers.

  * full resolution, B=24 512x512: the previous path (the CE kernel's arg-max over a zero label tensor, then the
    boolean gather / index_put with its two nonzero() synchronisations), torch.where(mask == 0, argmax, mask), and the
    kernel -- also as a share of the measured HBM copy bandwidth for its K_t * s + 8 + 8 * f0 bytes per pixel
    (f0: background fraction), on synth.make_labels labels and on labels drawn per pixel at random;
  * low resolution, from [B,K_t,32,32] at 512x512 and [B,K_t,33,33] at 513x513: the kernel against
    F.interpolate + argmax + where;
  * the whole compute_loss + backward step with pseudo_label=True at VOC 15-1 (B=24, 512x512, bg_weighted_ce off):
    previous path against the kernel, eager, and the kernel's step replayed from a CUDA graph.

The labels are rewritten in place, so every timed call is preceded by a copy from pristine labels; the copy is timed
on its own and subtracted.  The full-resolution teachers (252 MB and more) exceed the 126 MB L2.

    python tools/pseudo_label_time.py [--iters N]"""
import argparse
import os
import subprocess
import sys

import torch
import torch.nn.functional as F

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from bacs_b200 import _cabi, ops, synth  # noqa: E402


def card():
    name = torch.cuda.get_device_name()
    try:
        limit = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i",
                                str(torch.cuda.current_device())], capture_output=True, text=True,
                               timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        limit = "unknown"
    return name, limit or "unknown"


def timeit(fn, iters, warmup=3):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / iters * 1000.0      # us per call


def previous_path(mask, teacher):
    """the code this replaces (BACSLoss.post_process_mask before the kernel): _argmax of the teacher logits"""
    pseudo = ops.pixel_loss(teacher, torch.zeros(teacher.shape[0], *teacher.shape[2:], dtype=torch.int64,
                                                 device=teacher.device), _cabi.PIX_CE, want_grad=False)["preds"]
    mask[mask == 0] = pseudo[mask == 0]


def hbm_copy_bandwidth(iters):
    src = torch.empty(2 << 30, dtype=torch.uint8, device="cuda")
    dst = torch.empty_like(src)
    t = timeit(lambda: dst.copy_(src), iters)
    return 2 * src.numel() / (t * 1e-6)


def random_labels(B, H, W, K, gen):
    return torch.randint(0, K, (B, H, W), generator=gen).cuda()


def full_resolution(iters, peak, gen):
    B, H, W = 24, 512, 512
    cfg = synth.CONFIGS["voc15-1_b24"]
    for what, Kt, dt in (("VOC", 20, torch.bfloat16), ("VOC", 20, torch.float32), ("ADE20K", 150, torch.bfloat16)):
        teacher = torch.randn(B, Kt, H, W, generator=gen).to(dt).cuda()
        am = teacher.float().argmax(1)
        for kind, pristine in (("make_labels", synth.make_labels(cfg, gen).cuda()),
                               ("random", random_labels(B, H, W, Kt + 1, gen))):
            mask = pristine.clone()
            assert torch.equal(ops.pseudo_label_inplace(mask, teacher), torch.where(pristine == 0, am, pristine))
            f0 = float((pristine == 0).float().mean())
            t_copy = timeit(lambda: mask.copy_(pristine), iters)

            def new():
                mask.copy_(pristine)
                ops.pseudo_label_inplace(mask, teacher)

            def prev():
                mask.copy_(pristine)
                previous_path(mask, teacher)

            def where():
                mask.copy_(pristine)
                torch.where(mask == 0, teacher.argmax(1), mask)

            t_new = timeit(new, iters) - t_copy
            t_prev = timeit(prev, iters) - t_copy
            t_where = timeit(where, iters) - t_copy
            nbytes = B * H * W * (Kt * teacher.element_size() + 8 + 8 * f0)
            print("full-res %-6s K_t=%-3d %-8s %-11s (f0 %.2f): previous %8.1f us | torch.where %8.1f us | kernel "
                  "%7.1f us = %.0f GB/s, %.0f%% of the measured copy bandwidth"
                  % (what, Kt, str(dt).replace("torch.", ""), kind, f0, t_prev, t_where, t_new,
                     nbytes / (t_new * 1e-6) / 1e9, 100.0 * nbytes / (t_new * 1e-6) / peak))
        del teacher, am
        torch.cuda.empty_cache()


def low_resolution(iters, gen):
    for what, Kt, dt, H, lh in (("VOC", 20, torch.bfloat16, 512, 32), ("VOC", 20, torch.float32, 512, 32),
                                ("ADE20K", 150, torch.bfloat16, 512, 32), ("VOC", 20, torch.bfloat16, 513, 33),
                                ("ADE20K", 150, torch.bfloat16, 513, 33)):
        B = 24
        sem = torch.randn(B, Kt, lh, lh, generator=gen).to(dt).cuda()
        c = synth.StepConfig("t", B=B, K=21, old_cl=20, T=1, H=H, W=H)
        pristine = synth.make_labels(c, gen).cuda()
        mask = pristine.clone()
        t_copy = timeit(lambda: mask.copy_(pristine), iters)

        def new():
            mask.copy_(pristine)
            ops.pseudo_label_inplace(mask, sem, lowres=True)

        def interp():
            mask.copy_(pristine)
            up = F.interpolate(sem, size=(H, H), mode="bilinear", align_corners=False)
            torch.where(mask == 0, up.argmax(1), mask)

        t_new = timeit(new, iters) - t_copy
        t_int = timeit(interp, iters) - t_copy
        print("low-res  %-6s K_t=%-3d %-8s %dx%d -> %dx%d: F.interpolate + argmax + where %8.1f us | kernel %7.1f us "
              "(%.1fx)" % (what, Kt, str(dt).replace("torch.", ""), lh, lh, H, H, t_int, t_new, t_int / t_new))
        del sem
        torch.cuda.empty_cache()


def whole_step(iters):
    from bacs_b200.loss import BACSLoss
    cfg = synth.CONFIGS["voc15-1_b24"]
    inp = synth.make_step_inputs(cfg, seed=3)
    loss_fn, net, batch, leaves = synth.build_bacs_step(cfg, inp, bg_weighted_ce=False, pseudo_label=True)
    img, mask = batch[0], batch[1]                 # (no replay in this config: a plain [img, mask] batch)
    gen = torch.Generator().manual_seed(4)
    teacher = torch.randn(cfg.B, cfg.old_cl, cfg.H, cfg.W, generator=gen).cuda()
    prev = loss_fn.prev_model
    _, pen, atts = prev(img, return_penultimate=True, return_attentions=True)
    prev.register(img, teacher, pen, atts)
    pristine = mask.clone()
    protos0 = loss_fn._prototypes._prototypes_tensors.clone()
    counts0 = loss_fn._prototypes._count_features.clone()

    def step():
        mask.copy_(pristine)
        loss_fn._prototypes._prototypes_tensors.copy_(protos0)
        loss_fn._prototypes._count_features.copy_(counts0)
        for v in leaves.values():
            v.grad = None
        loss, preds = loss_fn.compute_loss(batch, net, train=True)
        loss.backward()
        return loss, preds

    def previous_mask(self, img_, mask_):
        with torch.no_grad():
            previous_path(mask_, self.prev_model(img_))
        return mask_

    t_new = timeit(step, iters)
    BACSLoss.post_process_mask, saved = previous_mask, BACSLoss.post_process_mask
    try:
        t_prev = timeit(step, iters)
    finally:
        BACSLoss.post_process_mask = saved
    t_new2 = timeit(step, iters)
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        step()
    torch.cuda.current_stream().wait_stream(s)
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        step()
    t_graph = timeit(g.replay, iters)
    print("step     VOC 15-1 B=24 512x512 K=21, teacher K_t=20 fp32, pseudo_label=True (incl. restoring mask, "
          "prototypes): previous %8.1f us | kernel eager %8.1f / %8.1f us | kernel graph replay %8.1f us"
          % (t_prev, t_new, t_new2, t_graph))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=50)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("pseudo_label_time.py needs a CUDA device")
    name, limit = card()
    print("card: %s, power limit %s" % (name, limit))
    peak = hbm_copy_bandwidth(args.iters)
    print("measured HBM copy bandwidth (2 GiB device-to-device copy, read + write): %.0f GB/s" % (peak / 1e9))
    gen = torch.Generator().manual_seed(0)
    full_resolution(args.iters, peak, gen)
    low_resolution(args.iters, gen)
    whole_step(max(10, args.iters // 5))


if __name__ == "__main__":
    main()
