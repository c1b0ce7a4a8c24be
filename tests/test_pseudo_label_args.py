"""CPU tests of the pseudo-label entry points' host side: argument checks and the low-res geometry rule, answered
before any CUDA call.  Only requests the entry points refuse are made here (placeholder pointers are never
dereferenced); the low-res rule must be the one of bacs_pixel_loss_lowres without seen logits, so every geometry
refused here also has bacs_pixel_lowres_workspace_bytes == 0, and every one it serves a non-zero workspace."""
import ctypes as C

import pytest
import torch

INVALID, UNSUPPORTED = -1, -2
PTR = 0x1000           # placeholder: only passed where the call is refused


@pytest.fixture(scope="module")
def cabi():
    from bacs_b200 import _cabi
    return _cabi


def _pixel_args(cabi, B, K, H, W):
    a = cabi.PixelArgs()
    a.B, a.K, a.H, a.W = B, K, H, W
    a.dtype, a.mode = cabi.F32, cabi.PIX_CE
    a.ignore_index, a.seen_scale = 255, 16
    return a


def _full(cabi, teacher, dtype, B, K, H, W, labels):
    return cabi.load().bacs_pseudo_label(teacher, dtype, B, K, H, W, labels, None)


def _low(cabi, sem, dtype, B, K, lh, lw, H, W, labels):
    return cabi.load().bacs_pseudo_label_lowres(sem, dtype, B, K, lh, lw, H, W, labels, None)


@pytest.mark.parametrize("teacher,labels", [(None, PTR), (PTR, None), (None, None)])
def test_null_pointers(cabi, teacher, labels):
    assert _full(cabi, teacher, cabi.F32, 2, 21, 64, 64, labels) == INVALID
    assert cabi.last_error().startswith("bacs_pseudo_label:")
    assert _low(cabi, teacher, cabi.F32, 2, 21, 4, 4, 64, 64, labels) == INVALID
    assert cabi.last_error().startswith("bacs_pseudo_label_lowres:")


@pytest.mark.parametrize("B,K,H,W", [(0, 21, 64, 64), (2, 0, 64, 64), (2, 21, 0, 64), (2, 21, 64, 0),
                                     (-1, 21, 64, 64), (2, -3, 64, 64)])
def test_bad_shapes(cabi, B, K, H, W):
    assert _full(cabi, PTR, cabi.BF16, B, K, H, W, PTR) == INVALID
    assert cabi.last_error().startswith("bacs_pseudo_label:")
    assert _low(cabi, PTR, cabi.BF16, B, K, 4, 4, H, W, PTR) == INVALID
    assert cabi.last_error().startswith("bacs_pseudo_label_lowres:")


@pytest.mark.parametrize("dtype", [-1, 3])
def test_unknown_dtype(cabi, dtype):
    assert _full(cabi, PTR, dtype, 2, 21, 64, 64, PTR) == INVALID
    assert cabi.last_error().startswith("bacs_pseudo_label:")
    assert _low(cabi, PTR, dtype, 2, 21, 4, 4, 64, 64, PTR) == INVALID
    assert cabi.last_error().startswith("bacs_pseudo_label_lowres:")


def test_lowres_refuses_256_teacher_channels(cabi):
    lib = cabi.load()
    assert lib.bacs_pixel_lowres_workspace_bytes(C.byref(_pixel_args(cabi, 2, 255, 512, 512)), 32, 32) != 0
    assert lib.bacs_pixel_lowres_workspace_bytes(C.byref(_pixel_args(cabi, 2, 256, 512, 512)), 32, 32) == 0
    assert _low(cabi, PTR, cabi.F32, 2, 256, 32, 32, 512, 512, PTR) == UNSUPPORTED
    assert cabi.last_error().startswith("bacs_pseudo_label_lowres: unsupported geometry")


# (H, W, lh, lw, K_t, served)
GEOMETRIES = [
    (512, 512, 32, 32, 20, True),
    (512, 512, 64, 64, 20, True),
    (500, 375, 32, 24, 20, True),
    (513, 513, 33, 33, 20, True),
    (500, 375, 63, 47, 20, True),
    (9, 9, 1, 1, 20, True),
    (16, 40, 1, 3, 20, True),
    (37, 2048, 3, 128, 151, True),
    (500, 375, 31, 24, 20, False),      # floor in y
    (500, 375, 31, 23, 20, False),      # floor in both
    (500, 375, 32, 23, 20, False),      # floor in x
    (513, 513, 32, 32, 20, False),
    (500, 375, 32, 47, 20, False),      # s = 16 in y, s = 8 in x
    (32, 32, 8, 8, 20, False),          # stride 4
    (512, 512, 16, 16, 20, False),      # stride 32
    (480, 480, 20, 20, 20, False),      # stride 24
    (4112, 4112, 257, 257, 20, False),  # lw > 256
    (64, 4096, 4, 256, 255, False),     # staging beyond 200 KB of shared memory
    (512, 512, 0, 32, 20, False),
    (512, 512, 32, -1, 20, False),
]


@pytest.mark.parametrize("H,W,lh,lw,K,served", GEOMETRIES)
def test_lowres_geometry_is_the_loss_kernels(cabi, H, W, lh, lw, K, served):
    nbytes = cabi.load().bacs_pixel_lowres_workspace_bytes(C.byref(_pixel_args(cabi, 2, K, H, W)), lh, lw)
    assert (nbytes != 0) == served, (H, W, lh, lw, K, nbytes)
    if not served:
        assert _low(cabi, PTR, cabi.BF16, 2, K, lh, lw, H, W, PTR) == UNSUPPORTED
        assert cabi.last_error().startswith("bacs_pseudo_label_lowres: unsupported geometry")


def test_op_has_no_cpu_path():
    from bacs_b200 import ops
    with pytest.raises(RuntimeError, match="no CPU path"):
        ops.pseudo_label_inplace(torch.zeros(1, 8, 8, dtype=torch.int64), torch.zeros(1, 3, 8, 8))
