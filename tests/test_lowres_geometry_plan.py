"""CPU test of the fused low-res path's geometry rule.  bacs_pixel_lowres_workspace_bytes is host code (the plan of
bacs_pixel_loss_lowres): non-zero for a shape the kernel serves, zero for one it refuses.

Accepted: W == s * lw with s = 8 or 16 and H a multiple of lh, or lh == ceil(H / s) and lw == ceil(W / s) for s = 8
or 16 -- what a backbone with padded stride-2 convolutions returns for any input -- with lw <= 256, K <= 255 and the
staging of one row group within 200 KB of shared memory.  The seen logits z need the first form."""
import ctypes as C

import pytest

# (H, W, lh, lw, K, accepted)
TABLE = [
    # W == s * lw, H a multiple of lh
    (512, 512, 32, 32, 21, True),
    (512, 512, 64, 64, 21, True),
    (528, 528, 33, 33, 21, True),
    (512, 1024, 32, 64, 21, True),
    (1024, 2048, 64, 128, 19, True),
    (64, 64, 2, 4, 21, True),
    (8, 8, 1, 1, 21, True),
    (512, 512, 32, 32, 255, True),
    # lh == ceil(H / s), lw == ceil(W / s)
    (500, 375, 32, 24, 21, True),
    (375, 500, 24, 32, 21, True),
    (513, 513, 33, 33, 21, True),
    (500, 375, 63, 47, 21, True),
    (512, 500, 32, 32, 21, True),
    (500, 512, 32, 32, 21, True),
    (512, 683, 32, 43, 151, True),
    (17, 17, 2, 2, 21, True),
    (9, 9, 1, 1, 21, True),
    (16, 40, 1, 3, 21, True),
    (5, 7, 1, 1, 21, True),
    (37, 2040, 3, 128, 151, True),      # fit at one image row per CTA only (about 170 KB)
    (37, 2048, 3, 128, 151, True),
    (1000, 2040, 63, 128, 151, True),
    (4100, 4090, 257, 256, 21, True),
    # neither rule
    (32, 32, 8, 8, 5, False),           # x4
    (500, 375, 31, 23, 21, False),      # floor(H / 16), floor(W / 16)
    (500, 375, 31, 24, 21, False),      # floor in y
    (500, 375, 32, 23, 21, False),      # floor in x
    (513, 513, 32, 32, 21, False),
    (500, 375, 32, 47, 21, False),      # s = 16 in y, s = 8 in x
    (500, 375, 64, 48, 21, False),
    (512, 512, 32, 32, 256, False),     # K > 255
    (513, 513, 33, 33, 256, False),
    (4112, 4112, 257, 257, 21, False),  # lw > 256
    (64, 4096, 4, 256, 255, False),     # beyond 200 KB of shared memory at one row per CTA
    (40, 4090, 3, 256, 255, False),
]


def _args(H, W, K, z=False):
    from bacs_b200 import _cabi
    a = _cabi.PixelArgs()
    a.B, a.K, a.H, a.W = 2, K, H, W
    a.dtype, a.mode = _cabi.F32, _cabi.PIX_CE
    a.ignore_index, a.seen_scale = 255, 16
    if z:                                # the plan only looks at the pointer and the head-map size
        a.z, a.T, a.h, a.w = 0x1000, 2, max(1, H // 16), max(1, W // 16)
    return a


@pytest.mark.parametrize("H,W,lh,lw,K,accepted", TABLE)
def test_lowres_geometry_rule(H, W, lh, lw, K, accepted):
    from bacs_b200 import _cabi
    lib = _cabi.load()
    nbytes = lib.bacs_pixel_lowres_workspace_bytes(C.byref(_args(H, W, K)), lh, lw)
    assert (nbytes != 0) == accepted, (H, W, lh, lw, K, nbytes)


@pytest.mark.parametrize("H,W,lh,lw,accepted", [
    (512, 512, 32, 32, True), (512, 512, 64, 64, True),
    (500, 375, 32, 24, False), (513, 513, 33, 33, False), (500, 512, 32, 32, False)])
def test_lowres_seen_logits_need_exact_geometry(H, W, lh, lw, accepted):
    from bacs_b200 import _cabi
    lib = _cabi.load()
    nbytes = lib.bacs_pixel_lowres_workspace_bytes(C.byref(_args(H, W, 21, z=True)), lh, lw)
    assert (nbytes != 0) == accepted, (H, W, lh, lw, nbytes)
