"""Times the full-resolution pixel kernel (bacs_pixel_loss) at a named config and checks it against the device oracle.
usage: pixel_time.py [config] [bf16|f16|f32] [B]      (BACS_NO_REGS=1 selects the two streaming passes)"""
import sys, torch
sys.path.insert(0, '/root/repo')
from bacs_b200 import synth, ops, _cabi
name = sys.argv[1] if len(sys.argv) > 1 else "ade100-50"
dtype = {"bf16": torch.bfloat16, "f16": torch.float16, "f32": torch.float32}[sys.argv[2] if len(sys.argv) > 2 else "bf16"]
cfg = synth.CONFIGS[name]
B = int(sys.argv[3]) if len(sys.argv) > 3 else cfg.B
g = torch.Generator(device="cuda").manual_seed(0)
logits = torch.randn(B, cfg.K, cfg.H, cfg.W, device="cuda", generator=g).to(dtype)
mask = synth.make_labels(cfg, torch.Generator().manual_seed(1), classes=list(range(1, cfg.K)), B=B).cuda()
z = torch.randn(B, cfg.T, cfg.h, cfg.w, device="cuda")
kw = dict(want_grad=True, z=z, want_distill_mask=True, old_cl=cfg.old_cl, focal_head=cfg.T - 1)
def timeit(fn, n=20):
    for _ in range(3): fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(n): fn()
    e1.record(); torch.cuda.synchronize()
    return e0.elapsed_time(e1) / n * 1000
out = ops.pixel_loss(logits, mask, _cabi.PIX_WEIGHTED_CE, **kw)
t = timeit(lambda: ops.pixel_loss(logits, mask, _cabi.PIX_WEIGHTED_CE, **kw))
t_fwd = timeit(lambda: ops.pixel_loss(logits, mask, _cabi.PIX_WEIGHTED_CE, want_grad=False, z=z, old_cl=cfg.old_cl))
px = B * cfg.H * cfg.W
es = logits.element_size()
alg = px * (2 * cfg.K * es + 17)
print("%s %s B=%d variant %d: fwd+grad %.1f us = %.0f GB/s algorithmic (%.1f%% of 6546) | fwd only %.1f us"
      % (name, sys.argv[2] if len(sys.argv) > 2 else "bf16", B, out["variant"], t, alg / t / 1e3, alg / t / 1e3 / 65.46, t_fwd))
