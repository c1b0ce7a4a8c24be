"""The fused full-resolution pixel loss (bacs_pixel_loss) at every kernel variant, template instantiation, mode and
optional output, against a float64 reference evaluated on the host from the exact values the kernels read: logits
rounded to their storage type and widened, fp32 seen logits, fp32 seen probabilities, fp32 class weights, and the
align_corners=True up-sample geometry in fp32 as ATen computes it (test_gpu_seen_heads.ac_geometry).

Labels are cleaned as the kernels treat them: ignore_index is ignored; a label in [0, K) is valid; anything else
(negative, >= K, 2^32 + 1, 255 when ignore_index is -1) is counted in INVALID and otherwise ignored.

Error model (per value, never normalised by the largest entry):
  * A sum (LOSS, WSUM, FOCAL, a gz cell, a score) may be off by 1e-5 x the sum of its terms' absolute values: the
    kernels' fp32 summation order changes with the variant and the pixels per thread.  A log-sum-exp term is
    lse_A - lse_B; its "absolute values" are |lse_A| + |lse_B|.  On top, every pixel's loss is allowed 2^-19 per
    unit of loss weight for the fast intrinsics (ex2.approx, lg2.approx, __logf, __fdividef, rcp.approx: absolute
    error ~2^-21 near 1, up to four of them per pixel), and every focal term 2^-20 (1 + |z|) for the intrinsics
    and the fp32 interpolation of the seen logits (|z| = the interpolated absolute head values).
  * The seen weight (1 - s)^gamma is evaluated from a seen probability s that the kernel interpolates in fp32 and
    passes through an approximate sigmoid: s may be off by 2^-20 (1 + |z|).  The loss allows that error times
    d mod / ds, and a pixel whose s lies within that band of `threshold` may take either branch (mod or 0).
  * Gradients are checked per element against a bound scaled per pixel: each element is a sum of coefficient x
    softmax terms, and may be off by 1e-5 x the sum of those terms' absolute values (plus 2^-100 per unit of weight
    for flushed subnormal exponentials).  In 16-bit storage an element must be within one ulp of the storage type
    of the float64 value rounded to that type, plus that fp32 allowance.
  * Counts and preds are exact.  The distill mask is exact outside the band above around lkd_threshold (zero width
    when the seen probabilities are given as seen_max).
  * Every gradient element is checked, at ignored and invalid pixels too (where it must be 0); a NaN or an
    unwritten element fails.  The one exception: a pixel with a foreground label (1 <= y < K) whose foreground mass
    sum_{c >= 1} exp(x_c - max) underflows in fp32 has no fp32 value for the closed form of its gradient.  Such
    pixels are left out of the gradient check, and the test prints how many.  Their loss is still checked: the
    kernels clamp the flushed mass to 1e-37, and the reference evaluates the same clamp.

The host copy of the plan (pixel_plan) returns the variant, the instantiation key and the workspace bytes of a
request; every case checks it against bacs_pixel_kernel_variant and bacs_pixel_workspace_bytes.  Cases whose plan
needs no tensor-map encoder run on the CPU too (with no device the library assumes 148 SMs)."""
import ctypes as C
import math
from dataclasses import dataclass, replace
from typing import Optional

import pytest
import torch

from test_gpu_seen_heads import ac_geometry, up_ac64  # noqa: F401  (up_ac64 interpolates with ac_geometry)

RTOL = 1e-5
EPS_LOG = 2.0 ** -19
EPS_SUB = 2.0 ** -100
DTYPES = {"f32": torch.float32, "bf16": torch.bfloat16, "f16": torch.float16}
ES = {"f32": 4, "bf16": 2, "f16": 2}
DT_ID = {"f32": 0, "bf16": 1, "f16": 2}
WCE, CE, UCE, SCORE = 0, 1, 2, 3
KREGS = (4, 8, 12, 16, 20, 21, 24)
CPU_SMS = 148
gpu = pytest.mark.gpu


def _on_gpu():
    return torch.cuda.is_available()


def sm_count():
    return torch.cuda.get_device_properties(0).multi_processor_count if _on_gpu() else CPU_SMS


# --------------------------------------------------------------------------------------
# requests
# --------------------------------------------------------------------------------------
@dataclass(frozen=True)
class Req:
    """One bacs_pixel_loss request.  z = (T, h, w, seen_scale) of the seen logits; focal_head >= 0 adds the focal
    term; labels names a label recipe of make_inputs; logit_off / mask_off are element / byte offsets of the logits
    and the distill mask past their allocations."""
    name: str
    dtype: str
    B: int
    K: int
    H: int
    W: int
    mode: int = CE
    grad: bool = True
    preds: bool = True
    mask: bool = False
    z: Optional[tuple] = None
    focal_head: int = -1
    seen_max: bool = False
    class_w: Optional[str] = None       # None, "w" (positive) or "w0" (some zeros)
    old_cl: int = 0
    ukd: bool = True
    gamma: float = 2.0
    threshold: float = 0.5
    focal_gamma: float = 2.0
    focal_alpha: Optional[float] = None
    lkd: float = 0.5
    grad_scale: float = 1.0
    ignore_index: int = 255
    labels: str = "mix"
    logits: str = "int"                 # "int": a few integers (arg-max ties); "conf": confident, see make_inputs
    logit_off: int = 0
    mask_off: int = 0
    epilogue: Optional[tuple] = None    # (ready: None / 0 / 1, over_wsum, focal_weight, loss_coef)
    seed: int = 0

    @property
    def gz(self):
        return self.focal_head >= 0


def _std(r):
    return r.gamma == 2.0 and r.ukd and (not r.gz or (r.focal_gamma == 2.0 and r.focal_alpha is None))


def _align256(n):
    return (n + 255) // 256 * 256


def pixel_plan(r, sms, tmap=True):
    """(variant, instantiation key, workspace bytes) that pixel_route (csrc/pixel_loss.cu) picks for `r` on `sms` SMs,
    with or without the driver's tensor-map encoder.  Labels, gradient and preds tensors are 512-byte aligned."""
    es, HW, K, dt = ES[r.dtype], r.H * r.W, r.K, r.dtype
    lg = r.logit_off * es
    T, h, w, sc = r.z if r.z else (0, 0, 0, 0)
    # 5: register column
    if tmap and dt != "f32" and 64 <= K <= 152 and HW % 256 == 0 and r.mode != SCORE and lg % 16 == 0:
        bx = min(HW // 128 * r.B, sms * 4)
        return 5, ("regs", dt), _align256(bx * 64)
    # 4: streaming passes
    n = 4 if dt == "f32" else 8
    if K >= 64 and HW % n == 0 and lg % 16 == 0 and (not r.mask or r.mask_off % 4 == 0):
        bx = min((HW // n + 255) // 256, max(1, sms * 4))
        return 4, ("stream", dt, r.grad), _align256(bx * r.B * 64) + (_align256(6 * HW * r.B * 4) if r.grad else 0)
    cap = 220 * 1024
    two_fit = lambda s: 2 * (s + 1024 + 512) <= 228 * 1024  # noqa: E731
    fast_ok = K <= 24 and HW % 512 == 0 and (HW * es) % 16 == 0 and lg % 16 == 0 and (not r.mask or r.mask_off % 2 == 0)
    if fast_ok:
        kreg = next(k for k in KREGS if k >= K)
        zrows = (T * 2 * w * 4 + 127) // 128 * 128 if r.z else 0
        stage = kreg * 512 * es + 4096 + zrows
        tail = (8 * T * 64 if r.z else 0) + 64
        rowtile = bool(r.z) and r.W % 512 == 0 and sc >= 16 and w % 4 == 0
        wce = rowtile and r.mode == WCE and not r.seen_max and tmap and w <= 256 and T <= 256
        stages = 3 if wce and not two_fit(4 * stage + tail) and two_fit(3 * stage + tail) else 4
        smem = stages * stage + tail
        if smem + 1024 <= cap:
            grid = min(HW // 512 * r.B, sms * (2 if two_fit(smem) else 1))
            ws = _align256((HW // 512 * r.B if r.mode == SCORE else grid) * 64)
            if wce:
                return 2, ("wce", dt, kreg, _std(r), stages), ws
            return 1, ("fast", dt, kreg, rowtile), ws
    extra = T * w * 4 + (w + 1) * 4 + 64
    for min_stages in (2, 1):
        for ppt in (2, 1):
            if ppt == 2 and HW % 2:
                continue
            P = ppt * 256
            coop = ppt == 1 and HW % 2 == 0 and K >= 2
            tile = K * (P * es + (64 if coop else 0))
            stages = next((st for st in (3, 2, 1) if st >= min_stages and st * tile + extra + 1024 <= cap), 0)
            if not stages:
                continue
            per_sm = 1
            if ppt == 1:
                for st in range(min(stages, 2), 0, -1):
                    if two_fit(st * tile + extra):
                        stages, per_sm = st, 2
                        break
            tpi = (HW + P - 1) // P
            grid = min(tpi * r.B, sms * per_sm)
            rowtile = bool(r.z) and P <= r.W and r.W % P == 0
            return 0, ("tile", dt, ppt, rowtile, coop, stages), _align256((tpi * r.B if r.mode == SCORE else grid) * 64)
    return -1, None, 0


def all_instantiations():
    """every kernel instantiation bacs_pixel_loss can launch, as pixel_plan keys"""
    keys = set()
    for dt in DTYPES:
        for (ppt, coop) in ((2, False), (1, True), (1, False)):
            for rt in (False, True):
                for st in (1, 2, 3):
                    keys.add(("tile", dt, ppt, rt, coop, st))
        for kreg in KREGS:
            for rt in (False, True):
                keys.add(("fast", dt, kreg, rt))
            for std in (False, True):
                for st in (3, 4):
                    keys.add(("wce", dt, kreg, std, st))
        for g in (False, True):
            keys.add(("stream", dt, g))
        if dt != "f32":
            keys.add(("regs", dt))
    return keys


# Instantiations that no request reaches, with the arithmetic.  two_fit(s): two CTAs of s bytes of dynamic shared
# memory fit an SM, 2 (s + 1536) <= 228 KB, i.e. s <= 115200.
def why_unreachable():
    why = {}
    for kreg in (20, 21, 24):
        stage = kreg * 512 * 4 + 4096
        for std in (False, True):
            why[("wce", "f32", kreg, std, 3)] = (
                "fp32 KREG %d: one stage is at least %d*512*4 + 4096 = %d bytes, so three stages (%d) never let two CTAs "
                "share an SM (s <= 115200) and the plan keeps four" % (kreg, kreg, stage, 3 * stage))
    return why


# --------------------------------------------------------------------------------------
# the reference
# --------------------------------------------------------------------------------------
def make_inputs(r):
    """host tensors of a request: logits [B,K,H,W] in the storage type, labels int64, z fp32, seen_max fp32,
    class weights fp32"""
    g = torch.Generator().manual_seed(1000 + r.seed * 7 + r.K)
    B, K, H, W = r.B, r.K, r.H, r.W
    if r.logits == "conf":
        # confident logits, multiples of 10; at 5 % of the pixels the background leads every other channel by 90 or
        # more, so that exp(x_c - max) flushes to zero in fp32 for every foreground channel (90 / ln 2 > 126)
        x = torch.randint(-4, 5, (B, K, H, W), generator=g).float() * 10.0
        sure = (torch.rand(B, 1, H, W, generator=g) < 0.05).expand(B, K, H, W).clone()
        sure[:, 0] = False
        x[:, 0] = torch.where(sure[:, 1], torch.full_like(x[:, 0], 60.0), x[:, 0])
        x = torch.where(sure, -30.0 - 10.0 * torch.randint(0, 4, (B, K, H, W), generator=g).float(), x)
    else:
        x = torch.randint(-3, 4, (B, K, H, W), generator=g).float()
        x = x + (torch.rand(B, K, H, W, generator=g) < 0.5).float() * torch.randn(B, K, H, W, generator=g) * 0.5
    logits = x.to(DTYPES[r.dtype])
    u = torch.rand(B, H, W, generator=g)
    lab = torch.randint(0, K, (B, H, W), generator=g)
    lab[u < 0.3] = 0
    if r.labels in ("mix", "noig"):
        specials = [r.ignore_index, K, K + 7, -1, 2 ** 32 + 1, 255, -3]
        for i, v in enumerate(specials):
            sel = (u >= 0.9 + 0.012 * i) & (u < 0.9 + 0.012 * (i + 1))
            lab[sel] = v
    if r.labels == "nobg":
        lab[lab == 0] = 1 if K > 1 else r.ignore_index
        lab[u > 0.9] = r.ignore_index
    if r.labels in ("mix", "nobg") and B >= 2:
        lab[1] = r.ignore_index                                  # one image all ignored
    z = sm = cw = None
    if r.z:
        T, h, w, _ = r.z
        z = torch.randn(B, T, h, w, generator=g) * 2.0
    if r.seen_max:
        sm = torch.rand(B, H, W, generator=g)
        sm[torch.rand(B, H, W, generator=g) < 0.05] = r.threshold   # exactly at the thresholds: strict compares
        sm[torch.rand(B, H, W, generator=g) < 0.05] = r.lkd
    if r.class_w:
        cw = torch.rand(K, generator=g) + 0.25
        if r.class_w == "w0":
            cw[::3] = 0.0
    return logits, lab, z, sm, cw


def _lse(x, sel):
    """log-sum-exp over the channels in boolean [K] `sel` (float64), and the matching softmax"""
    xs = x[:, sel]
    return torch.logsumexp(xs, 1), torch.softmax(xs, 1)


def reference(r, logits, lab, z, sm, cw):
    """float64 values of everything bacs_pixel_loss writes, with per-value error bounds (see the module docstring)"""
    B, K, H, W = r.B, r.K, r.H, r.W
    HW = H * W
    x = logits.double()
    lab = lab.clone()
    ign = lab == r.ignore_index
    valid = (lab >= 0) & (lab < K) & ~ign
    invalid = ~ign & ~valid
    y = torch.where(valid, lab, torch.zeros_like(lab))
    bg = valid & (y == 0)
    old = min(max(r.old_cl, 0), K)
    chan = torch.arange(K)
    xm = x.max(1, keepdim=True)[0]
    e = torch.exp(x - xm)                                              # [B,K,H,W]
    lse = torch.logsumexp(x, 1)
    p = torch.softmax(x, 1)
    xy = x.gather(1, y.unsqueeze(1)).squeeze(1)
    onehot = torch.nn.functional.one_hot(y, K).permute(0, 3, 1, 2).double()
    have_seen = r.z is not None or r.seen_max
    out = {}

    # seen probability, its error band, and the focal head's interpolated logit
    s = torch.zeros(B, H, W, dtype=torch.float64)
    s_err = torch.zeros_like(s)
    zabs = torch.zeros_like(s)
    up = None
    if r.z:
        T, h, w, sc = r.z
        up = up_ac64(z.double(), sc)
        zabs = up_ac64(z.double().abs(), sc).max(1)[0]
        if not r.seen_max:
            s = torch.sigmoid(up.max(1)[0])
            s_err = 2.0 ** -20 * (1 + zabs)
    if r.seen_max:
        s = sm.double()

    # loss components: a list of (weight [B,H,W], lse_A, softmax_A over sel_A, lse_B, softmax_B over sel_B);
    # the pixel's loss is sum w (lse_A - lse_B), its gradient sum w (softmax_A - softmax_B) (scattered to channels)
    zero = torch.zeros(B, H, W, dtype=torch.float64)
    comps = []
    fg = chan >= 1
    oldm = chan < old
    lse_fg, p_fg = (_lse(x, fg) if K > 1 else (zero, None))
    # foreground mass flushed to zero in fp32 (ex2.approx.ftz flushes results below 2^-126): the kernels clamp it to
    # 1e-37, so their log of it is ln(1e-37) and their max is the background logit
    under_fg = torch.zeros(B, H, W, dtype=torch.bool)
    if r.mode == WCE and K > 1:
        under_fg = ~(((x[:, 1:] - xm) * (1 / math.log(2))) >= -126).any(1)
        clamp = float(torch.tensor(1e-37, dtype=torch.float32).double().log())
        lse_fg = torch.where(under_fg, xm[:, 0] + clamp, lse_fg)
    lse_old, p_old = (_lse(x, oldm) if old > 0 else (zero, None))
    # "single channel" lse: x_c, softmax = one-hot
    x0 = x[:, 0]
    oh0 = torch.zeros_like(x)
    oh0[:, 0] = 1.0
    mod_band = torch.zeros_like(s)
    if r.mode == WCE:
        u = 1.0 if r.ukd else 0.0
        smod = torch.where(s > r.threshold, torch.ones_like(s), s)
        mod = (1 - smod) ** r.gamma
        # either branch inside the band around threshold; d mod / ds <= gamma (1 - s)^(gamma - 1)
        near = ((s - r.threshold).abs() <= s_err) & (s_err > 0)   # seen_max: exact fp32 compare, no band
        alt = torch.where(s > r.threshold, (1 - s) ** r.gamma, torch.zeros_like(s))
        mod_band = torch.where(near, (mod - alt).abs(), torch.zeros_like(s)) + \
            s_err * r.gamma * (1 - s).clamp(min=0) ** (r.gamma - 1) * (s <= r.threshold)
        isold = valid & (y >= 1) & (y < old)
        isnew = valid & (y >= old)
        comps.append((torch.where(bg, mod, zero), lse, p, x0, oh0))
        comps.append((torch.where(bg | isold, torch.full_like(s, u), zero), lse, p, lse_old, p_old))
        comps.append((torch.where(isold | isnew, torch.ones_like(s), zero), lse, p, lse_fg, p_fg))
        comps.append((torch.where(isnew, torch.ones_like(s), zero), lse, p, xy, onehot))
        gs = float(torch.tensor(1.0 / (B * HW), dtype=torch.float32)) * r.grad_scale
        gsc = torch.full_like(s, gs)
        wsum = 0.0
    else:
        wy = cw.double()[y] if cw is not None else torch.ones_like(s)
        wy = torch.where(valid, wy, zero)
        if r.mode == UCE:
            wy = valid.double()
            isold = valid & (y < old)
            comps.append((torch.where(isold, wy, zero), lse, p, lse_old, p_old))
            comps.append((torch.where(~isold, wy, zero), lse, p, xy, onehot))
        else:
            comps.append((wy, lse, p, xy, onehot))
        wsum = float(wy.sum())
        s_norm = float(torch.tensor(1.0 / wsum, dtype=torch.float32)) if wsum > 0 else 0.0
        gsc = torch.full_like(s, s_norm * r.grad_scale)

    loss_pix = torch.zeros_like(s)
    loss_abs = torch.zeros_like(s)
    wtot = torch.zeros_like(s)
    g = torch.zeros_like(x)
    gabs = torch.zeros_like(x)
    for (wgt, la, pa, lb, pb) in comps:
        if pb is None:
            continue
        loss_pix += wgt * (la - lb)
        loss_abs += wgt.abs() * (la.abs() + lb.abs())
        wtot += wgt.abs()
        wa = (wgt * gsc).unsqueeze(1)
        g += wa * pa
        gabs += wa.abs() * pa
        if pb.shape[1] == K:
            sel = slice(None)
            g -= wa * pb
            gabs += wa.abs() * pb
        else:
            sel = (chan >= 1) if pb is p_fg else (chan < old)
            g[:, sel] -= wa * pb
            gabs[:, sel] += wa.abs() * pb
    # foreground labels whose foreground mass underflows: no fp32 value of the gradient's closed form
    under = valid & (y >= 1) & under_fg
    out["excluded"] = int(under.sum())
    loss_err = (RTOL * loss_abs + EPS_LOG * wtot + mod_band * (lse - x0).abs() * bg) * valid
    out["LOSS"] = (float((loss_pix * valid).sum()), float(loss_err.sum()))
    out["WSUM"] = wsum
    out["KEPT"] = out["VALID"] = int(valid.sum())
    out["BG"] = int(bg.sum())
    out["INVALID"] = int(invalid.sum())
    out["preds"] = x.argmax(1)                                       # first maximum
    out["dlogits"] = (g, RTOL * gabs + EPS_SUB * gsc.unsqueeze(1) * (1 + wtot.unsqueeze(1)), ~under)

    # distill mask, with its band
    thr_ok = s > r.lkd if have_seen else torch.ones_like(valid)
    m = bg & thr_ok
    band = bg & ((s - r.lkd).abs() <= s_err) & (s_err > 0)
    out["mask"] = (m, band)
    out["DISTILL"] = (int((m & ~band).sum()), int(band.sum()))   # certain pixels, pixels that may go either way

    # focal term of head focal_head, and gz
    if r.gz:
        Z = up[:, r.focal_head].clone().requires_grad_(True)
        t = (~bg).double()
        bce = torch.nn.functional.softplus(Z) - t * Z
        pt = torch.exp(-bce)
        term = (1 - pt) ** r.focal_gamma * bce
        if r.focal_alpha is not None:
            term = term * (r.focal_alpha * t + (1 - r.focal_alpha) * (1 - t))
        term = term * valid
        (dterm,) = torch.autograd.grad(term.sum(), Z)
        term = term.detach()
        floor = 2.0 ** -20 * (1 + zabs) * valid
        out["FOCAL"] = (float(term.sum()), float((RTOL * term.abs() + floor).sum()))
        T, h, w, sc = r.z
        out["gz"] = (_scatter_up(dterm, B, h, w, sc), _scatter_up(RTOL * dterm.abs() + floor, B, h, w, sc))
    else:
        out["FOCAL"] = (0.0, 0.0)

    if r.mode == SCORE:
        per = (loss_pix * valid).sum((1, 2))
        err = loss_err.sum((1, 2))
        out["score"] = (-per / HW, err / HW)

    if r.epilogue is not None:
        ready, over, fw, coef = r.epilogue
        kept = out["KEPT"]
        on = (ready is None or ready != 0) and out["BG"] > 0 and kept > 0
        fs = fw / kept if on else 0.0
        main, main_err = coef * out["LOSS"][0], abs(coef) * out["LOSS"][1]
        if over:
            main, main_err = main / wsum, main_err / wsum
        val = main + fs * out["FOCAL"][0]
        out["focal_scale"] = fs
        out["loss"] = (val, main_err + fs * out["FOCAL"][1] + 2.0 ** -23 * abs(val))
    return out


def _scatter_up(v, B, h, w, s):
    """adjoint of up_ac64 applied to a per-pixel [B,H,W] map (float64)"""
    zz = torch.zeros(B, 1, h, w, dtype=torch.float64, requires_grad=True)
    (gg,) = torch.autograd.grad((up_ac64(zz, s)[:, 0] * v).sum(), zz)
    return gg[:, 0]


def _ulp(v, dtype):
    """spacing of `dtype` at the float64 values v (their rounded magnitudes), subnormals included"""
    fi = torch.finfo(dtype)
    mant = {torch.bfloat16: 7, torch.float16: 10, torch.float32: 23}[dtype]
    a = v.abs().clamp(min=fi.tiny)
    return torch.exp2(torch.floor(torch.log2(a)) - mant).clamp(min=fi.tiny * 2.0 ** -mant)


# --------------------------------------------------------------------------------------
# the request as C-ABI arguments, and a run on the device
# --------------------------------------------------------------------------------------
FAKE = 0x10000000   # a 512-byte aligned fake address: plan-only calls never touch memory


def _args(r, ptrs=None):
    """bacs_pixel_args of `r`; ptrs maps field -> device address (fake aligned addresses + the offsets when None)"""
    from bacs_b200 import _cabi
    a = _cabi.PixelArgs()
    fake = {"logits": FAKE + r.logit_off * ES[r.dtype], "labels": 2 * FAKE, "acc": 3 * FAKE,
            "dlogits": 4 * FAKE if r.grad else None, "preds": 5 * FAKE if r.preds else None,
            "distill_mask": 6 * FAKE + r.mask_off if r.mask else None, "z": 7 * FAKE if r.z else None,
            "seen_max": 8 * FAKE if r.seen_max else None, "gz": 9 * FAKE if r.gz else None,
            "class_w": 10 * FAKE if r.class_w else None,
            "hist": 11 * FAKE if r.grad and r.mode in (CE, UCE) else None,
            "score": 12 * FAKE if r.mode == SCORE else None}
    for k, v in (ptrs or fake).items():
        setattr(a, k, v)
    a.B, a.K, a.H, a.W = r.B, r.K, r.H, r.W
    a.T, a.h, a.w, a.seen_scale = r.z if r.z else (0, 0, 0, 16)
    a.dtype, a.mode = DT_ID[r.dtype], r.mode
    a.old_cl, a.ukd, a.focal_head, a.ignore_index = r.old_cl, int(r.ukd), r.focal_head, r.ignore_index
    a.gamma, a.threshold, a.focal_gamma = r.gamma, r.threshold, r.focal_gamma
    a.focal_alpha = -1.0 if r.focal_alpha is None else r.focal_alpha
    a.lkd_threshold, a.grad_scale = r.lkd, r.grad_scale
    return a


def _dev(host, off):
    """host tensor on the device, `off` elements past the start of its allocation"""
    flat = torch.zeros(host.numel() + off, dtype=host.dtype)
    flat[off:] = host.reshape(-1)
    return flat.cuda()[off:].view(host.shape)


def run_kernel(r, inputs):
    """bacs_pixel_loss on the device through the C ABI; returns the host copies of everything it wrote"""
    from bacs_b200 import _cabi, ops
    lib = _cabi.load()
    logits, lab, z, sm, cw = inputs
    B, H, W = r.B, r.H, r.W
    d = {"logits": _dev(logits, r.logit_off), "labels": lab.cuda(), "acc": torch.zeros(8, dtype=torch.float64).cuda()}
    if r.grad:
        d["dlogits"] = torch.full_like(d["logits"], float("nan"))
    if r.preds:
        d["preds"] = torch.full((B, H, W), -7, dtype=torch.int64, device="cuda")
    if r.mask:
        d["distill_mask"] = _dev(torch.full((B, H, W), 9, dtype=torch.uint8), r.mask_off)
    if r.z:
        d["z"] = z.cuda()
    if r.seen_max:
        d["seen_max"] = sm.cuda()
    if r.gz:
        d["gz"] = torch.zeros(B, r.z[1], r.z[2], dtype=torch.float32, device="cuda")
    if r.class_w:
        d["class_w"] = cw.cuda()
    if r.grad and r.mode in (CE, UCE):
        d["hist"] = ops.label_hist(d["labels"])
    if r.mode == SCORE:
        d["score"] = torch.full((B,), float("nan"), dtype=torch.float64, device="cuda")
    a = _args(r, {k: v.data_ptr() for k, v in d.items()})
    if r.epilogue is not None:
        ready, over, fw, coef = r.epilogue
        d["focal_scale"] = torch.full((1,), float("nan"), device="cuda")
        d["loss"] = torch.full((1,), float("nan"), device="cuda")
        if ready is not None:
            d["ready"] = torch.tensor([ready], dtype=torch.int32, device="cuda")
            a.ready = d["ready"].data_ptr()
        a.focal_scale_out, a.loss_out = d["focal_scale"].data_ptr(), d["loss"].data_ptr()
        a.focal_weight, a.loss_coef, a.loss_over_wsum = fw, coef, int(over)
    variant = lib.bacs_pixel_kernel_variant(C.byref(a))
    nbytes = lib.bacs_pixel_workspace_bytes(C.byref(a))
    ws = torch.empty(max(nbytes, 16), dtype=torch.uint8, device="cuda")
    _cabi.check(lib.bacs_pixel_loss(C.byref(a), ws.data_ptr(), nbytes, ops._stream()), "bacs_pixel_loss")
    torch.cuda.synchronize()
    got = {k: v.cpu() for k, v in d.items()}
    got["variant"], got["workspace"] = variant, nbytes
    return got


# --------------------------------------------------------------------------------------
# checks
# --------------------------------------------------------------------------------------
ACC = dict(LOSS=0, WSUM=1, FOCAL=2, KEPT=3, BG=4, INVALID=5, DISTILL=6, VALID=7)
WORST = {}   # output -> worst ratio of error to bound seen in this session


def _ratio(what, err, bound):
    rt = float(err / bound) if bound > 0 else (0.0 if err == 0 else math.inf)
    if rt != rt:          # NaN: an unwritten or non-finite output
        rt = math.inf
    WORST[what] = max(WORST.get(what, 0.0), rt)
    return rt


def check_against_reference(r, got, want):
    acc = got["acc"]
    for k in ("KEPT", "VALID", "BG", "INVALID"):
        assert int(acc[ACC[k]]) == want[k] and float(acc[ACC[k]]) == want[k], (k, float(acc[ACC[k]]), want[k])
    v, e = want["LOSS"]
    assert _ratio("LOSS", abs(float(acc[ACC["LOSS"]]) - v), e) <= 1, ("LOSS", float(acc[ACC["LOSS"]]), v, e)
    if r.mode != WCE:
        assert _ratio("WSUM", abs(float(acc[ACC["WSUM"]]) - want["WSUM"]), RTOL * want["WSUM"]) <= 1
    fv, fe = want["FOCAL"]
    assert _ratio("FOCAL", abs(float(acc[ACC["FOCAL"]]) - fv), fe) <= 1, ("FOCAL", float(acc[ACC["FOCAL"]]), fv, fe)
    if r.preds:
        assert torch.equal(got["preds"], want["preds"]), "preds: %d wrong" % int((got["preds"] != want["preds"]).sum())
    if r.mask:
        m, band = want["mask"]
        gm = got["distill_mask"]
        assert int(((gm != m.to(torch.uint8)) & ~band).sum()) == 0, "distill mask"
        assert int(acc[ACC["DISTILL"]]) == int(gm.sum())
        assert int(((gm != 0) & (gm != 1)).sum()) == 0
    # DISTILL: the mask's pixel count.  Without a mask only the training-step kernel (variant 2) still counts it;
    # the others leave it at 0.
    certain, either = want["DISTILL"]
    got_d = float(acc[ACC["DISTILL"]])
    if r.mask or got["variant"] == 2:
        assert certain <= got_d <= certain + either and got_d == int(got_d), ("DISTILL", got_d, certain, either)
    else:
        assert got_d == 0.0, ("DISTILL without a mask", got_d)
    if r.grad:
        g64, gb, keep = want["dlogits"]
        gk = got["dlogits"].double()
        dt = DTYPES[r.dtype]
        if dt != torch.float32:
            g64r = g64.to(dt).double()
            gb = gb + _ulp(g64r, dt)
            g64 = g64r
        ok = keep.unsqueeze(1).expand_as(gk)
        err = (gk - g64).abs()
        bad = ~(err <= gb) & ok                     # NaN-safe: an unwritten (NaN) element fails
        assert not bool(bad.any()), "dlogits: %d of %d out of bounds (worst ratio %.3g)" % (
            int(bad.sum()), int(ok.sum()), float((err / gb)[ok].nan_to_num(math.inf).max()))
        if bool(ok.any()):
            _ratio("dlogits", float((err / gb)[ok].max()), 1.0)
    if r.gz:
        gz64, gzb = want["gz"]
        err = (got["gz"].double() - gz64).abs()
        bad = ~(err <= gzb)                         # NaN-safe
        assert not bool(bad.any()), "gz: %d cells out of bounds (worst ratio %.3g)" % (
            int(bad.sum()), float((err / gzb).nan_to_num(math.inf).max()))
        _ratio("gz", float((err / gzb.clamp(min=1e-300)).max()), 1.0)
    if r.mode == SCORE:
        sv, se = want["score"]
        err = (got["score"] - sv).abs()
        assert bool((err <= se).all()), ("score", got["score"], sv, se)
        _ratio("score", float((err / se.clamp(min=1e-300)).max()), 1.0)
    if r.epilogue is not None:
        assert float(got["focal_scale"][0]) == float(torch.tensor(want["focal_scale"], dtype=torch.float32))
        lv, le = want["loss"]
        assert _ratio("loss_out", abs(float(got["loss"][0]) - lv), le) <= 1, ("loss_out", float(got["loss"][0]), lv)


# --------------------------------------------------------------------------------------
# the case table
# --------------------------------------------------------------------------------------
# One request per generic-tile instantiation (dtype, K, H, W, seen logits (T, h, w, seen_scale), logit offset): the
# cheapest found by searching the plan.  One pixel per thread without the lane-pair walk on row tiles needs K = 1
# and more than 210 heads of seen-logit rows in shared memory; odd images need seen_scale 1 for the seen logits.
TILE_WITNESS = [
    ("f32", 57, 3, 7, None, 0), ("f32", 1, 3, 7, None, 0), ("f32", 53, 63, 63, (241, 63, 63, 1), 0),
    ("f32", 55, 6, 43, None, 0), ("f32", 61, 64, 64, (192, 64, 64, 1), 0), ("f32", 50, 64, 64, (237, 64, 64, 1), 0),
    ("f32", 1, 16, 4096, (216, 1, 256, 16), 0), ("f32", 1, 16, 4096, (215, 1, 256, 16), 0),
    ("f32", 1, 16, 4096, (214, 1, 256, 16), 0), ("f32", 55, 16, 256, (1, 1, 16, 16), 0),
    ("f32", 61, 16, 1024, (192, 1, 64, 16), 0), ("f32", 50, 16, 1024, (237, 1, 64, 16), 0),
    ("f32", 104, 6, 43, None, 0), ("f32", 37, 6, 43, None, 0), ("f32", 1, 6, 43, None, 0),
    ("f32", 63, 16, 1536, (226, 1, 96, 16), 0), ("f32", 37, 16, 512, (1, 1, 32, 16), 0),
    ("f32", 25, 16, 512, (1, 1, 32, 16), 0),
]
for _dt in ("bf16", "f16"):
    TILE_WITNESS += [
        (_dt, 113, 3, 7, None, 0), (_dt, 1, 3, 7, None, 0), (_dt, 106, 63, 63, (241, 63, 63, 1), 0),
        (_dt, 110, 6, 43, None, 0), (_dt, 178, 34, 34, (96, 34, 34, 1), 0), (_dt, 63, 112, 112, (212, 112, 112, 1), 0),
        (_dt, 1, 16, 4096, (217, 1, 256, 16), 0), (_dt, 1, 16, 3584, (248, 1, 224, 16), 0),
        (_dt, 1, 16, 4096, (216, 1, 256, 16), 0), (_dt, 63, 16, 2560, (249, 1, 160, 16), 0),
        (_dt, 63, 16, 2048, (225, 1, 128, 16), 0), (_dt, 63, 16, 1536, (247, 1, 96, 16), 0),
        (_dt, 196, 6, 43, None, 0), (_dt, 73, 6, 43, None, 0), (_dt, 1, 6, 43, None, 0),
        (_dt, 63, 16, 2560, (236, 1, 160, 16), 0), (_dt, 63, 16, 512, (239, 1, 32, 16), 0),
        (_dt, 25, 16, 512, (1, 1, 32, 16), 0),
    ]

NON_STD = [dict(focal_alpha=0.25), dict(gamma=1.5), dict(ukd=False), dict(focal_gamma=1.5)]
EPILOGUES = [(None, False, 0.5, 0.7), (0, False, 0.5, 0.7), (1, True, 0.25, 1.3)]


def _wce_geom(dt, kreg, stages):
    """the smallest (T, w) whose training-step plan has `stages` stages (None if there is none)"""
    for T, w in sorted(((T, w) for T in (1, 2, 4, 8, 16, 32, 64) for w in (32, 64, 96, 128, 256)),
                       key=lambda tw: tw[0] * tw[1]):
        r = Req("x", dt, 1, kreg, 16, 16 * w, mode=WCE, old_cl=1, z=(T, 1, w, 16))
        if pixel_plan(r, CPU_SMS)[1][4] == stages:
            return T, w
    return None


def _cases():
    cases = []
    # generic tiles: all four modes in turn, every option somewhere
    for i, (dt, K, H, W, z, off) in enumerate(TILE_WITNESS):
        mode = (CE, UCE, SCORE, WCE)[i % 4]
        big = z is not None and z[0] * H * W > 200000
        kw = dict(logit_off=off, z=z, mask=i % 4 != 1, seed=i)
        if mode == SCORE and big:
            mode = CE
        if mode == SCORE:
            kw.update(B=3, grad=False)
        if mode == WCE:
            kw.update(old_cl=max(1, K // 2), seen_max=z is None or i % 8 == 7, ukd=i % 3 != 0,
                      gamma=(2.0, 1.5)[i % 2])
        if mode == UCE:
            kw.update(old_cl=(1, max(1, K // 2), K)[i % 3])
        if mode == CE:
            kw.update(class_w=(None, "w0", "w")[i % 3])
        if z is not None and i % 2 == 0:
            kw.update(focal_head=z[0] - 1, focal_alpha=(None, 0.25)[i % 4 == 0])
        if i % 5 == 0:
            kw.update(grad_scale=4.0)
        if i % 6 == 1:
            kw.update(ignore_index=-1)
        if i % 7 == 3:
            kw.update(labels="nobg")
        if i % 5 == 2 and mode != WCE:
            kw.update(epilogue=EPILOGUES[i % 3])
        kw.setdefault("B", 1 if big else 2)
        cases.append(Req("tile%d" % i, dt, K=K, H=H, W=W, mode=mode, **kw))
    # K <= 24 in registers: row tiles (CE with seen logits, or WEIGHTED_CE from seen_max) and whole-image tiles
    i = 0
    for dt in DTYPES:
        for kreg in KREGS:
            for rowtile in (False, True):
                K = kreg if i % 2 else wce_kmin(kreg)
                mode = (CE, UCE, SCORE, WCE)[i % 4]
                if rowtile:
                    geo = dict(H=16, W=512, z=(2, 1, 32, 16))
                elif i % 3 == 0:
                    geo = dict(H=16, W=256, z=(3, 1, 16, 16))         # seen logits on whole-image tiles
                else:
                    geo = dict(H=16, W=64)
                kw = dict(geo, mask=True, seed=100 + i, B=3 if mode == SCORE else 2)
                if mode == SCORE:
                    kw.update(grad=False)
                if mode == WCE:
                    kw.update(old_cl=max(1, K // 2), seen_max=True, ukd=i % 3 != 1, gamma=(2.0, 1.5)[i % 2])
                if mode == UCE:
                    kw.update(old_cl=(1, max(1, K // 2), K)[i % 3])
                if mode == CE:
                    kw.update(class_w=(None, "w0")[i % 2])
                if "z" in kw and i % 2 == 0:
                    kw.update(focal_head=kw["z"][0] - 1, focal_alpha=(None, 0.25)[i % 4 == 0])
                if i % 5 == 1:
                    kw.update(grad_scale=0.5, ignore_index=-1)
                if i % 7 == 2 and mode != WCE:
                    kw.update(epilogue=EPILOGUES[i % 3])
                cases.append(Req("fast%d" % i, dt, K=K, mode=mode, **kw))
                i += 1
    # the training-step kernel: every (dtype, KREG, STD, ring depth) the plan can produce
    i = 0
    for dt in DTYPES:
        for kreg in KREGS:
            for stages in (4, 3):
                tw = _wce_geom(dt, kreg, stages)
                if tw is None:
                    continue
                T, w = tw
                for std in (True, False):
                    K = kreg if i % 2 else wce_kmin(kreg)
                    kw = dict(B=2, H=16, W=16 * w, z=(T, 1, w, 16), mode=WCE, old_cl=max(1, K // 2), mask=True,
                              focal_head=(T - 1, -1)[i % 5 == 4], seed=200 + i)
                    if not std:
                        kw.update(NON_STD[(i // 2) % 4])
                        if "focal_alpha" in NON_STD[(i // 2) % 4] or "focal_gamma" in NON_STD[(i // 2) % 4]:
                            kw["focal_head"] = T - 1
                    if i % 3 == 1:
                        kw.update(grad_scale=8.0)
                    if i % 6 == 2:
                        kw.update(ignore_index=-1)
                    if i % 7 == 5:
                        kw.update(labels="nobg")
                    if i % 4 == 3:
                        kw.update(epilogue=EPILOGUES[i % 3][:1] + (False, 0.5, 0.7))
                    if i % 9 == 8:
                        kw.update(lkd=0.7, threshold=0.3)
                    cases.append(Req("wce%d" % i, dt, K=K, **kw))
                    i += 1
    # K >= 64: streaming passes and the register column
    cases += [
        Req("stream-f32-ce", "f32", 2, 70, 16, 64, class_w="w0", mask=True),
        Req("stream-f32-score", "f32", 3, 70, 16, 64, mode=SCORE, grad=False, mask=True, class_w="w"),
        Req("stream-bf16-uce", "bf16", 2, 160, 16, 64, mode=UCE, old_cl=80, grad_scale=2.0),
        Req("stream-bf16-score", "bf16", 3, 100, 16, 64, mode=SCORE, grad=False),
        Req("stream-f16-wce", "f16", 2, 153, 16, 64, mode=WCE, old_cl=100, seen_max=True, mask=True, ukd=False),
        Req("stream-f16-nograd", "f16", 2, 170, 16, 64, mode=WCE, old_cl=9, grad=False, z=(2, 1, 4, 16),
            focal_head=1, mask=True, epilogue=(1, False, 0.5, 0.7)),
        Req("stream-f32-K300", "f32", 2, 300, 16, 64, grad=False, ignore_index=-1, labels="noig"),
        Req("regs-bf16-wce", "bf16", 2, 80, 16, 256, mode=WCE, old_cl=40, z=(3, 1, 16, 16), focal_head=2, mask=True),
        Req("regs-f16-ce", "f16", 2, 152, 16, 256, class_w="w0", mask=True, ignore_index=-1),
        Req("regs-bf16-uce", "bf16", 2, 64, 16, 256, mode=UCE, old_cl=64, grad_scale=3.0),
        # edges: confident logits (the foreground mass underflows in fp32 at some pixels), a single tile, an odd
        # distill-mask pointer
        Req("conf-wce", "bf16", 2, 21, 16, 512, mode=WCE, old_cl=16, z=(2, 1, 32, 16), focal_head=1, mask=True,
            logits="conf"),
        Req("conf-tile", "f32", 2, 30, 16, 64, mode=WCE, old_cl=15, seen_max=True, mask=True, logits="conf"),
        Req("single-tile", "bf16", 1, 30, 16, 32, mode=WCE, old_cl=15, z=(2, 1, 2, 16), focal_head=0, mask=True),
        Req("mask-odd", "bf16", 2, 30, 16, 64, mode=WCE, old_cl=15, seen_max=True, mask=True, mask_off=1),
        Req("mask-odd-fast", "f32", 2, 12, 16, 64, mode=CE, mask=True, mask_off=1),
        # logits one element past their allocation: plain copies instead of bulk copies on the tile kernel, on
        # shapes that aligned logits would send to the register path, the training-step kernel, the streaming passes
        # and the register column
        Req("off-tile-bf16", "bf16", 2, 30, 16, 64, mode=WCE, old_cl=15, seen_max=True, mask=True, logit_off=1),
        Req("off-fast-f32", "f32", 2, 12, 16, 64, class_w="w0", mask=True, logit_off=1, ignore_index=-1),
        Req("off-wce-bf16", "bf16", 2, 21, 16, 512, mode=WCE, old_cl=16, z=(2, 1, 32, 16), focal_head=1, mask=True,
            logit_off=1),
        Req("off-wce-f16-conf", "f16", 2, 8, 16, 512, mode=WCE, old_cl=4, z=(1, 1, 32, 16), focal_head=0, mask=True,
            logit_off=1, logits="conf"),
        Req("off-stream-f32", "f32", 2, 70, 16, 64, mode=UCE, old_cl=35, mask=True, logit_off=1),
        Req("off-regs-f16", "f16", 2, 100, 16, 256, mode=CE, class_w="w", mask=True, logit_off=1, grad_scale=2.0),
        Req("off-score-f16", "f16", 3, 40, 16, 64, mode=SCORE, grad=False, mask=True, logit_off=1),
        # per-image scores on the generic tile kernel with more tiles (180) than CTAs (148 per SM count)
        Req("score-many-tiles", "bf16", 3, 30, 120, 256, mode=SCORE, grad=False, mask=True),
    ]
    return cases


def wce_kmin(kreg):
    return {4: 1, 8: 5, 12: 9, 16: 13, 20: 17, 21: 21, 24: 22}[kreg]


CASES = _cases()


def _needs_tmap(r):
    return pixel_plan(r, CPU_SMS, tmap=True) != pixel_plan(r, CPU_SMS, tmap=False)


def _marks(r):
    return [gpu] if _needs_tmap(r) else []


@pytest.fixture(scope="module", autouse=True)
def _report_worst():
    yield
    if WORST:
        print("\nworst error / bound: " + ", ".join("%s %.3g" % kv for kv in sorted(WORST.items())))


def test_pixel_case_table_covers_every_kernel():
    """The cases reach every instantiation the host code can launch (with this device's SM count); the others are
    listed with the reason no request reaches them."""
    sms = sm_count()
    reached = {pixel_plan(r, sms)[1] for r in CASES}
    why = why_unreachable()
    want = all_instantiations() - set(why)
    for key, reason in sorted(why.items(), key=str):
        print("unreachable %s: %s" % (key, reason))
    print("reached %d of %d kernel instantiations" % (len(reached & want), len(want)))
    assert not (reached & set(why)), "listed as unreachable but reached: %s" % sorted(reached & set(why), key=str)
    assert reached >= want, "not reached: %s" % sorted(want - reached, key=str)
    for dt in DTYPES:   # the tile kernel's ring depths 1, 2 and 3, in every dtype
        assert {k[5] for k in reached if k[0] == "tile" and k[1] == dt} == {1, 2, 3}


def test_pixel_plan_unreachable_arithmetic():
    """fp32 WEIGHTED_CE with 16 or more heads at K = 22..24 overflows the register path's shared memory and lands
    on the generic tile kernel; fp32 training-step stages never come to three at KREG >= 20."""
    from bacs_b200 import _cabi
    lib = _cabi.load()
    for K in (22, 23, 24):
        r = Req("x", "f32", 2, K, 16, 512, mode=WCE, old_cl=8, z=(16, 1, 32, 16))
        assert pixel_plan(r, CPU_SMS)[0] == 0 and pixel_plan(r, CPU_SMS, tmap=False)[0] == 0
        assert lib.bacs_pixel_kernel_variant(C.byref(_args(r))) == 0
    for kreg in (20, 21, 24):
        for T in (1, 2, 4, 8, 16, 32, 64, 128, 256):
            for w in (32, 64, 128, 256):
                r = Req("x", "f32", 1, kreg, 16, 16 * w, mode=WCE, old_cl=1, z=(T, 1, w, 16))
                key = pixel_plan(r, CPU_SMS)[1]
                assert key is None or key[0] != "wce" or key[4] == 4


@pytest.mark.parametrize("r", [pytest.param(r, id=r.name, marks=_marks(r)) for r in CASES])
def test_pixel_plan_matches_library(r):
    """variant and workspace bytes of the host plan equal the library's (fake, suitably aligned pointers)"""
    from bacs_b200 import _cabi
    lib = _cabi.load()
    tmap = _on_gpu()
    v, _, ws = pixel_plan(r, sm_count(), tmap=tmap)
    a = _args(r)
    assert lib.bacs_pixel_kernel_variant(C.byref(a)) == v
    assert lib.bacs_pixel_workspace_bytes(C.byref(a)) == ws


@gpu
@pytest.mark.parametrize("r", CASES, ids=[r.name for r in CASES])
def test_pixel_variant_against_fp64(r):
    inputs = make_inputs(r)
    want = reference(r, *inputs)
    v, key, ws = pixel_plan(r, sm_count())
    for rr in (r, replace(r, grad=False, preds=False, mask=False, mask_off=0)):
        got = run_kernel(rr, inputs)
        vv, _, wws = pixel_plan(rr, sm_count())
        assert (got["variant"], got["workspace"]) == (vv, wws), (key, got["variant"], got["workspace"])
        check_against_reference(rr, got, want)
    if want["excluded"]:
        print("%s: %d confident pixels excluded (foreground mass underflows in fp32)" % (r.name, want["excluded"]))


@gpu
def test_pixel_ce_gradient_refused_above_256_classes():
    """CE-type gradients normalise by the 257-bin label histogram, which counts labels >= 256 together: K = 300 with
    a gradient is refused (it used to run with a normaliser missing the labels 256..299)."""
    from bacs_b200 import _cabi
    for mode in (CE, UCE):
        r = Req("K300", "f32", 2, 300, 16, 64, mode=mode, old_cl=150, ignore_index=-1, labels="noig")
        inputs = make_inputs(r)
        with pytest.raises(_cabi.BacsError, match="257-bin"):
            run_kernel(r, inputs)


@gpu
def test_pixel_counters_past_128_tiles_per_cta():
    """bf16, K = 4, 512-pixel row tiles: more than 128 tiles per CTA, so the training-step kernel's 8-bit pixel
    counters are flushed many times; the counts are exact (reference on the device)."""
    from bacs_b200 import _cabi
    B, K, H, W = 80, 4, 512, 512
    r = Req("big", "bf16", B, K, H, W, mode=WCE, old_cl=2, z=(1, 32, 32, 16), mask=True)
    v, key, _ = pixel_plan(r, sm_count())
    assert key == ("wce", "bf16", 4, True, 4)
    grid = min(H * W // 512 * B, 2 * sm_count())
    assert H * W // 512 * B // grid > 128
    g = torch.Generator(device="cuda").manual_seed(5)
    logits = torch.randint(-3, 4, (B, K, H, W), generator=g, device="cuda").to(torch.bfloat16)
    lab = torch.randint(0, K, (B, H, W), generator=g, device="cuda")
    u = torch.rand(B, H, W, generator=g, device="cuda")
    lab[u < 0.5] = 0
    # ignored and invalid labels only in the last images: the first 128 tiles of every CTA hold 256 valid pixels per
    # thread, which an 8-bit counter flushed every 128 tiles would wrap
    late = torch.arange(B, device="cuda").view(B, 1, 1) >= 78
    lab[(u > 0.9) & late] = 255
    lab[(u > 0.95) & late] = K + 1
    z = torch.randn(B, 1, 32, 32, generator=g, device="cuda")
    from bacs_b200 import ops
    out = ops.pixel_loss(logits, lab, _cabi.PIX_WEIGHTED_CE, want_grad=False, z=z, want_distill_mask=True, old_cl=2)
    assert out["variant"] == 2
    acc = out["acc"].cpu()
    valid = (lab >= 0) & (lab < K)
    assert int(acc[ACC["KEPT"]]) == int(valid.sum()) == int(acc[ACC["VALID"]])
    assert int(acc[ACC["BG"]]) == int((lab == 0).sum())
    assert int(acc[ACC["INVALID"]]) == int((lab == K + 1).sum())
    assert int(acc[ACC["DISTILL"]]) == int(out["distill_mask"].sum())
    assert torch.equal(out["preds"], logits.float().argmax(1))
