"""Times the fused low-res pixel kernel (bacs_pixel_loss_lowres) at input sizes that are not a multiple of the output
stride (lh = ceil(H/16), lw = ceil(W/16)), next to what it replaces -- torch's bilinear up-sample feeding the
full-resolution kernel, plus the up-sample's backward where a gradient is wanted -- and, for scale, the fused kernel
at the exact geometry of the next multiple-of-16 size.  CE mode with the arg-max; CUDA events after warm-up.

    python tools/lowres_geometry_time.py [--iters N]"""
import argparse
import os
import subprocess
import sys

import torch
import torch.nn.functional as F

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from bacs_b200 import ops, _cabi  # noqa: E402

# (what, B, K, H, W, want_grad, dtype)
CASES = [
    ("eval VOC 500x375", 1, 21, 500, 375, False, torch.float32),
    ("eval ADE20K 512x683", 1, 151, 512, 683, False, torch.float32),
    ("train 513x513 bf16", 24, 21, 513, 513, True, torch.bfloat16),
    ("train 513x513 fp32", 24, 21, 513, 513, True, torch.float32),
    ("ADE20K lw=128 1020x2040 bf16", 4, 151, 1020, 2040, True, torch.bfloat16),
    ("ADE20K lw=128 1020x2040 eval", 4, 151, 1020, 2040, False, torch.bfloat16),
]


def card():
    name = torch.cuda.get_device_name()
    try:
        limit = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i",
                                str(torch.cuda.current_device())], capture_output=True, text=True,
                               timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        limit = "unknown"
    return name, limit or "unknown"


def timeit(fn, iters, warmup=5):
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


def labels(B, K, H, W, gen):
    lab = torch.randint(0, K, (B, H, W), generator=gen)
    return torch.where(torch.rand(B, H, W, generator=gen) < 0.05, torch.full_like(lab, 255), lab).cuda()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=20)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("lowres_geometry_time.py needs a CUDA device")
    name, limit = card()
    print("card: %s, power limit %s" % (name, limit))
    gen = torch.Generator().manual_seed(0)
    for what, B, K, H, W, grad, dt in CASES:
        lh, lw = (H + 15) // 16, (W + 15) // 16
        sem = torch.randn(B, K, lh, lw, generator=gen).to(dt).cuda()
        lab = labels(B, K, H, W, gen)
        He, We = 16 * lh, 16 * lw
        lab_e = labels(B, K, He, We, gen)

        def fused():
            ops.pixel_loss(sem, lab, _cabi.PIX_CE, want_grad=grad, lowres=True)

        def exact():
            ops.pixel_loss(sem, lab_e, _cabi.PIX_CE, want_grad=grad, lowres=True)

        def torch_path():
            s = sem.detach().requires_grad_(grad)
            full = F.interpolate(s, size=(H, W), mode="bilinear", align_corners=False)
            out = ops.pixel_loss(full.detach(), lab, _cabi.PIX_CE, want_grad=grad)
            if grad:
                full.backward(out["dlogits"])

        t_fused, t_torch, t_exact = timeit(fused, args.iters), timeit(torch_path, args.iters), timeit(exact, args.iters)
        print("%-30s B=%-2d K=%-3d %dx%d -> %dx%d %s%s: fused %8.1f us | F.interpolate%s + full-res kernel %8.1f us "
              "(%.1fx) | fused at %dx%d (exact) %8.1f us"
              % (what, B, K, H, W, lh, lw, str(dt).replace("torch.", ""), " +grad" if grad else "", t_fused,
                 " + backward" if grad else "", t_torch, t_torch / t_fused, He, We, t_exact))
        del sem, lab, lab_e
        torch.cuda.empty_cache()


if __name__ == "__main__":
    main()
