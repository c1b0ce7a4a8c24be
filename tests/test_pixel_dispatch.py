"""CPU test of the fused pixel loss's host side: which kernel bacs_pixel_loss picks, the workspace it needs, and the
argument checks of its two entry points.  Nothing here launches a kernel: the calls plan only, or return before any
launch, so the pointers are fake (suitably aligned) values.

The route table was recorded with the library as it was before the kernel choice moved into one function.  The plans
size their persistent grids by the SM count, and the library uses 148, the B200's count, when it cannot query a
device; so the workspace sizes are the same on a machine without a GPU and on a B200.  Variants 2 (the training-step
kernel) and 5 (the register-column kernel) need the driver's tensor-map encoder, which a machine without a GPU driver
does not have (there those shapes report 1 and 4); their rows are marked gpu."""
import ctypes as C

import pytest

from bacs_b200 import _cabi

LOGITS, LABELS, DLOGITS, ACC, HIST = 0x10000000, 0x20000000, 0x30000000, 0x40000000, 0x50000000
Z, SEEN_MAX, SCORE, GZ, WORKSPACE = 0x60000000, 0x70000000, 0x80000000, 0x90000000, 0xA0000000


def _args(**kw):
    """bacs_pixel_args of a CE step with gradient (B=2, K=21, 512x512, fp32); `kw` overrides fields.  z=True adds
    seen logits of T heads at h, w = H/16, W/16."""
    a = _cabi.PixelArgs()
    a.B, a.K, a.H, a.W = 2, 21, 512, 512
    a.dtype, a.mode = _cabi.F32, _cabi.PIX_CE
    a.logits, a.labels, a.dlogits, a.acc, a.hist = LOGITS, LABELS, DLOGITS, ACC, HIST
    a.ignore_index, a.seen_scale = 255, 16
    z, T = kw.pop("z", False), kw.pop("T", 2)
    if z:
        a.z, a.T, a.h, a.w = Z, T, kw.get("H", 512) // 16, kw.get("W", 512) // 16
    for k, v in kw.items():
        setattr(a, k, v)
    return a


BF16, F16 = _cabi.BF16, _cabi.F16
gpu = pytest.mark.gpu


def _wce(**kw):
    """the training step: WEIGHTED_CE with the seen logits, 16 old classes, bf16"""
    return dict(dict(mode=_cabi.PIX_WEIGHTED_CE, old_cl=16, z=True, dtype=BF16), **kw)


def _score(**kw):
    """per-image scores: no gradient"""
    return dict(dict(mode=_cabi.PIX_SCORE, score=SCORE, dlogits=None), **kw)


# (fields, variant, workspace bytes): 0 generic tiles, 1 K <= 24 in registers, 2 training step, 4 streaming passes,
# 5 register column, -1 no shared-memory tile fits
ROUTES = [
    pytest.param(dict(K=24), 1, 9472, id="K24"),
    pytest.param(dict(K=25), 0, 9472, id="K25"),
    pytest.param(dict(K=63), 0, 18944, id="K63"),
    pytest.param(dict(K=64), 4, 12615680, id="K64-f32"),
    pytest.param(dict(K=64, dtype=BF16), 5, 37888, id="K64-bf16", marks=gpu),
    pytest.param(dict(K=152, dtype=BF16), 5, 37888, id="K152-bf16", marks=gpu),
    pytest.param(dict(K=153, dtype=BF16), 4, 12599296, id="K153-bf16"),
    pytest.param(dict(K=151), 4, 12615680, id="K151-f32"),
    pytest.param(dict(K=151, dtype=F16, **_score()), 4, 16384, id="K151-f16-score"),
    pytest.param(dict(K=151, dtype=BF16, **_score()), 4, 16384, id="K151-bf16-score"),
    pytest.param(dict(**_score()), 1, 65536, id="K21-score"),
    pytest.param(dict(H=24, W=32), 0, 256, id="hw768"),
    pytest.param(dict(K=151, dtype=BF16, H=24, W=32), 5, 768, id="hw768-K151-bf16", marks=gpu),
    pytest.param(dict(K=151, dtype=BF16, H=24, W=36), 4, 41728, id="hw864-K151-bf16"),
    pytest.param(dict(H=33, W=33), 0, 768, id="odd"),
    pytest.param(dict(K=151, H=33, W=33), 0, 768, id="odd-K151"),
    pytest.param(dict(dtype=BF16, logits=LOGITS + 2), 0, 9472, id="logits+2"),
    pytest.param(dict(K=151, dtype=BF16, logits=LOGITS + 2), 0, 18944, id="logits+2-K151"),
    pytest.param(dict(z=True), 1, 9472, id="ce-z-rowtile"),
    pytest.param(_wce(), 2, 18944, id="wce", marks=gpu),
    pytest.param(_wce(W=1024, T=8), 2, 18944, id="wce-3stage", marks=gpu),
    pytest.param(_wce(seen_max=SEEN_MAX), 1, 18944, id="wce-seen_max"),
    pytest.param(dict(K=300, H=33, W=33), -1, 0, id="K300-odd"),
]


@pytest.mark.parametrize("fields,variant,nbytes", ROUTES)
def test_pixel_route(fields, variant, nbytes):
    lib = _cabi.load()
    a = _args(**fields)
    assert lib.bacs_pixel_kernel_variant(C.byref(a)) == variant
    assert lib.bacs_pixel_workspace_bytes(C.byref(a)) == nbytes


# Each row breaks one rule of a valid request (a CE step with gradient; seen logits where a row needs them).
INVALID = [
    pytest.param(dict(logits=None), id="null-logits"),
    pytest.param(dict(labels=None), id="null-labels"),
    pytest.param(dict(acc=None), id="null-acc"),
    pytest.param(dict(H=0), id="empty-shape"),
    pytest.param(dict(dtype=3), id="dtype"),
    pytest.param(dict(mode=4), id="mode"),
    pytest.param(dict(mode=-1), id="mode-negative"),
    pytest.param(dict(ignore_index=0), id="ignore_index-0"),
    pytest.param(dict(ignore_index=20), id="ignore_index-K-1"),
    pytest.param(dict(z=True, T=0), id="z-without-T"),
    pytest.param(dict(z=True, seen_scale=8), id="z-H-not-h-times-scale"),
    pytest.param(dict(z=True, gz=GZ, focal_head=2), id="focal-head-T"),
    pytest.param(dict(z=True, gz=GZ, focal_head=-1), id="focal-head-negative"),
    pytest.param(dict(gz=GZ), id="focal-without-z"),
    pytest.param(dict(mode=_cabi.PIX_WEIGHTED_CE, old_cl=16), id="wce-without-seen"),
    pytest.param(dict(hist=None), id="ce-grad-without-hist"),
    pytest.param(_score(score=None), id="score-without-score"),
    pytest.param(_score(dlogits=DLOGITS), id="score-with-grad"),
]

LH = LW = 32  # low-res logits of the 512x512 request at output stride 16


def _call(entry, a, workspace, nbytes):
    lib = _cabi.load()
    if entry == "bacs_pixel_loss":
        return lib.bacs_pixel_loss(C.byref(a), workspace, nbytes, None)
    return lib.bacs_pixel_loss_lowres(C.byref(a), LH, LW, workspace, nbytes, None)


@pytest.mark.parametrize("entry", ["bacs_pixel_loss", "bacs_pixel_loss_lowres"])
@pytest.mark.parametrize("fields", INVALID)
def test_pixel_args_rejected(entry, fields):
    # no workspace: a request that passed the checks would stop at BACS_ERR_WORKSPACE, before any launch
    assert _call(entry, _args(**fields), None, 0) == -1  # BACS_ERR_INVALID
    assert _cabi.last_error().startswith(entry + ":"), _cabi.last_error()


# bacs_pixel_workspace_bytes rounds the tile kernels' partial rows up to 256 bytes, while bacs_pixel_loss checks them
# unrounded.  The tile request here has 148 rows of 64 bytes, a multiple of 256, so the two sizes agree.  The streaming
# passes (K = 151) need the rounded size, because their coefficient planes start after it.
@pytest.mark.parametrize("fields", [pytest.param({}, id="tiles"), pytest.param(dict(K=151), id="stream")])
@pytest.mark.parametrize("entry", ["bacs_pixel_loss", "bacs_pixel_loss_lowres"])
def test_pixel_workspace_one_byte_short(entry, fields):
    lib = _cabi.load()
    a = _args(**fields)
    need = (lib.bacs_pixel_workspace_bytes(C.byref(a)) if entry == "bacs_pixel_loss"
            else lib.bacs_pixel_lowres_workspace_bytes(C.byref(a), LH, LW))
    assert need > 0
    assert _call(entry, a, WORKSPACE, need - 1) == -4  # BACS_ERR_WORKSPACE
    assert _cabi.last_error().startswith(entry + ":"), _cabi.last_error()
