"""The per-class prototype family -- bacs_class_distance (one tcgen05 kernel) and bacs_class_sums (the one-hot
mma.sync kernel at NT = 4..20 and the shared-memory table kernel at every vector path and warp count) -- at every
plan, tile count and path, against float64 references evaluated from the exact values the kernels read: bf16
features and prototypes for the distances, the stored feature type for the sums.

Both ops are called through the C ABI with output buffers owned here: every output is pre-filled with a sentinel
(NaN distances, -1 nearest classes, NaN sums, an all-NaN workspace) and has a guard band before and after it.  Every
entry must be written and every guard must stay untouched.

Error model (per element, never normalised by the largest entry):
  * dist2[b,k,p] = |f|^2 + |c_k|^2 - 2 f.c_k may be off by 1e-5 M with M = |f|^2 + |c_k|^2 + 2 sum_d |f_d c_kd|:
    the fp32 expansion cancels terms of size M (the bf16 products are exact, the fp32 sums are not).  dist2 >= 0.
    The fp64 reference is evaluated as the same expansion, image by image; its own error is ~2^-50 M.
  * nearest[b,p] is in [0, Kc), it is the lowest class among the kernel's own smallest distances, and its fp64
    distance is within the allowances of its class and of the fp64 arg-min above the fp64 minimum -- so it is the
    fp64 arg-min wherever the gap to the runner-up exceeds twice the allowance.
  * Integer features and prototypes in [-8, 8] keep every product and partial sum an integer below 2^24: dist2 is
    bit-equal to float64 and nearest is the fp64 arg-min (lowest class on ties) exactly.
  * The distances do not depend on how the batch is split or where a tile falls in its CTA's run: a batched call,
    per-image calls, two halves and a call without nearest give the same bits.
  * sums[k][c] may be off by 1e-5 x the sum of its terms' absolute values; on integer features they are bit-equal
    to float64, a class present at one pixel sums to that feature exactly and an absent class to exactly 0.  Counts
    (ops.class_sums) are exact.

The host copies of the plans (cd_plan, cs_plan) follow bacs_class_distance / bacs_class_sums; the coverage test
prints what the case tables reach, and the profiler test confirms the class-sums plan by the kernel names.  The
refusal rows are rejected before the tensor-map encoder and run without a device too."""
import re
from dataclasses import dataclass

import pytest
import torch

gpu = pytest.mark.gpu
RTOL = 1e-5
CPU_SMS = 148
F32, BF16, F16 = 0, 1, 2
DTYPES = {"f32": torch.float32, "bf16": torch.bfloat16, "f16": torch.float16}
DT_ID = {"f32": F32, "bf16": BF16, "f16": F16}
GUARD = 64                 # elements of guard band before and after every output
GUARD_F, GUARD_I = -1234.5, -7777
WORST = {}                 # quantity -> worst ratio of error to allowance seen in this session


def _on_gpu():
    return torch.cuda.is_available()


def sm_count():
    return torch.cuda.get_device_properties(0).multi_processor_count if _on_gpu() else CPU_SMS


def _dev():
    return "cuda" if _on_gpu() else "cpu"


def _lib():
    from bacs_b200 import _cabi
    return _cabi.load()


def _stream():
    from bacs_b200 import ops
    return ops._stream()


def _ratio(what, r):
    WORST[what] = max(WORST.get(what, 0.0), r)


@pytest.fixture(scope="module", autouse=True)
def _report_worst():
    yield
    if WORST:
        print("\nworst error / allowance: " + ", ".join("%s %.3g" % kv for kv in sorted(WORST.items())))


def _guarded(n, dtype, fill, guard):
    """[GUARD | n entries | GUARD] on the device: the entries hold `fill`, the guards `guard`"""
    buf = torch.full((n + 2 * GUARD,), fill, dtype=dtype, device=_dev())
    buf[:GUARD] = guard
    buf[GUARD + n:] = guard
    return buf


def _guards_intact(buf, n, guard):
    return bool((buf[:GUARD] == guard).all()) and bool((buf[GUARD + n:] == guard).all())


def _bits(t):
    return t.view(torch.int32) if t.dtype == torch.float32 else t


# --------------------------------------------------------------------------------------
# bacs_class_distance: the plan
# --------------------------------------------------------------------------------------
TILE_M, CHUNK_K, MAX_CHUNKS, STAGE_BYTES, SMEM_CAP = 128, 32, 16, 32 * 128 * 2, 224 * 1024


def cd_smem(Np, Dp, stages):
    """shared-memory bytes of class_distance_kernel: ring | B operand with a spare row per k-block | norms | xx, best,
    arg | barriers"""
    return stages * STAGE_BYTES + (Np + 1) * 16 * (Dp // 8) + Np * 4 + 3 * 4 * TILE_M * 4 + (MAX_CHUNKS + 2 + 16) * 8 + 16


@dataclass(frozen=True)
class CdPlan:
    ok: bool
    Np: int
    Dp: int
    nchunks: int
    stages: int
    smem: int
    n_tiles: int
    grid: int
    tiles_min: int        # tiles of the least loaded CTA
    tiles_max: int
    laps: int             # complete passes of the least loaded CTA over the ring


def cd_plan(B, D, hw, Kc, sms):
    Np, Dp = (Kc + 31) // 32 * 32, (D + 15) // 16 * 16
    nchunks = (Dp + CHUNK_K - 1) // CHUNK_K
    stages = 8 if cd_smem(Np, Dp, 8) <= SMEM_CAP else 4
    smem = cd_smem(Np, Dp, stages)
    ok = 0 < Kc <= 256 and D % 8 == 0 and hw % 8 == 0 and Dp <= MAX_CHUNKS * CHUNK_K and smem <= SMEM_CAP
    n_tiles = (hw + TILE_M - 1) // TILE_M * B
    grid = min(n_tiles, sms)
    tmin, tmax = n_tiles // grid, (n_tiles + grid - 1) // grid
    return CdPlan(ok, Np, Dp, nchunks, stages, smem, n_tiles, grid, tmin, tmax, tmin * nchunks // stages)


@dataclass(frozen=True)
class Cd:
    """one class-distance case: data is "randn", "int" (integers in [-8, 8]), "tie" (integers, duplicate prototypes
    in three accumulator quarters), "trap" (features near 0, every prototype far) or "offset" (randn + 50)"""
    name: str
    B: int
    D: int
    h: int
    w: int
    Kc: int
    data: str

    @property
    def hw(self):
        return self.h * self.w

    def plan(self, sms):
        return cd_plan(self.B, self.D, self.hw, self.Kc, sms)


def cd_cases(sms):
    return [
        # the ADE20K shape of bench.py (4 stages, 192 tiles) and twice its batch
        Cd("ade", 24, 512, 32, 32, 150, "randn"),
        Cd("ade-x2-int", 48, 512, 32, 32, 150, "int"),
        # tiles per CTA: two laps of the 8-stage ring with one chunk per tile; 1 (last tile of an image partial);
        # 2; 3 or more with an uneven split
        Cd("laps", 16 * sms + 3, 8, 2, 4, 1, "int"),
        Cd("one-tile", 2, 64, 25, 40, 31, "randn"),
        Cd("two-tiles", sms + 5, 128, 8, 16, 32, "int"),
        Cd("three-uneven", 3 * sms + 7, 24, 8, 15, 33, "randn"),
        # chunk counts 3, 5, 7 (last chunk of 16 channels) and 12 (also 16), several tiles per CTA
        Cd("nch3", sms, 96, 8, 17, 97, "int"),
        Cd("nch5", 40, 160, 25, 40, 255, "randn"),
        Cd("nch7", 2 * sms + 1, 200, 8, 16, 256, "int"),
        Cd("nch12-224k", sms + 1, 368, 8, 15, 256, "randn"),       # 4 stages, exactly 224 KB
        # shared-memory boundaries
        Cd("np160-d512", 3, 512, 25, 40, 160, "int"),               # 4 stages
        Cd("np224-d416", 4, 416, 8, 17, 224, "randn"),              # 4 stages
        Cd("np160-d480", 2 * sms, 480, 8, 16, 160, "randn"),        # the largest 8-stage shape at Np = 160
        Cd("kc1-d32", 5, 32, 2, 4, 1, "randn"),
        # ties across the builder warpgroups, the padding trap, cancellation
        Cd("ties", sms // 4 + 1, 64, 25, 40, 150, "tie"),
        Cd("trap", 2 * sms + 3, 96, 8, 16, 33, "trap"),
        Cd("trap-97", 5, 200, 25, 40, 97, "trap"),
        Cd("offset50", 10, 256, 25, 40, 97, "offset"),
    ]


# rejected before the tensor-map encoder: (name, overrides of the base call, part of the error message)
CD_BASE = dict(dtype=BF16, B=2, D=64, h=4, w=8, Kc=10, feat_off=0, proto_off=0, null=None)
CD_REFUSALS = [
    ("dtype-f32", dict(dtype=F32), "bf16"),
    ("dtype-f16", dict(dtype=F16), "bf16"),
    ("kc0", dict(Kc=0), "bad shape"),
    ("kc257", dict(Kc=257), "bad shape"),
    ("d12", dict(D=12), "multiples of 8"),
    ("hw12", dict(h=3, w=4), "multiples of 8"),
    ("d520", dict(D=520), "do not fit one SM"),
    ("kc161-d512", dict(Kc=161, D=512), "do not fit one SM"),
    ("kc256-d376", dict(Kc=256, D=376), "do not fit one SM"),
    ("kc224-d432", dict(Kc=224, D=432), "do not fit one SM"),
    ("feat-off8", dict(feat_off=8), "16-byte aligned"),
    ("proto-off8", dict(proto_off=8), "16-byte aligned"),
    ("null-feat", dict(null="feat"), "null pointer"),
    ("null-protos", dict(null="protos"), "null pointer"),
    ("null-dist2", dict(null="dist2"), "null pointer"),
]


# --------------------------------------------------------------------------------------
# bacs_class_distance: inputs, reference, run, checks
# --------------------------------------------------------------------------------------
def cd_inputs(c, seed=0):
    """bf16 features [B, D, hw] and prototypes [Kc, D] on the host"""
    g = torch.Generator().manual_seed(7 * c.Kc + c.D + seed)
    B, D, hw, Kc = c.B, c.D, c.hw, c.Kc
    if c.data in ("randn", "offset"):
        f, p = torch.randn(B, D, hw, generator=g), torch.randn(Kc, D, generator=g)
        if c.data == "offset":
            f, p = f + 50.0, p + 50.0
    elif c.data in ("int", "tie"):
        f, p = torch.randint(-8, 9, (B, D, hw), generator=g).float(), torch.randint(-8, 9, (Kc, D), generator=g).float()
    else:   # trap: |f - c|^2 >= 49 D for every real class, |f|^2 <= D for a zero (padded) row
        f = torch.randint(-1, 2, (B, D, hw), generator=g).float()
        p = (torch.randint(0, 2, (Kc, D), generator=g) * 16 - 8).float()
    if c.data == "tie":
        # equal rows in three of the four accumulator quarters; every 7th pixel sits on them (distance 0)
        j, q = 5, (Kc + 31) // 32 * 8
        assert j + 3 * q < Kc
        p[j + q] = p[j]
        p[j + 3 * q] = p[j]
        f[:, :, ::7] = p[j].view(1, D, 1)
    if c.data != "trap":
        p[0] = f[B - 1, :, hw - 1]            # the last pixel of the last (partial) tile sits on class 0
    return f.to(torch.bfloat16), p.to(torch.bfloat16)


def cd_reference(f, p):
    """fp64 (dist2, M) [B, Kc, hw] from the bf16 values; on the device when there is one"""
    F, P = f.to(_dev()).double(), p.to(_dev()).double()
    ff = (F * F).sum(1).unsqueeze(1)                      # [B, 1, hw]
    cc = (P * P).sum(1).view(1, -1, 1)                    # [1, Kc, 1]
    ref = ff + cc - 2.0 * torch.matmul(P, F)
    M = ff + cc + 2.0 * torch.matmul(P.abs(), F.abs())
    return ref, M


def run_distance(fd, pd, B, D, h, w, Kc, want_nearest=True):
    """bacs_class_distance through the C ABI on device tensors; (dist2 [B, Kc, hw], nearest [B, hw] or None)"""
    from bacs_b200 import _cabi
    lib = _lib()
    hw = h * w
    nd, nn = B * Kc * hw, B * hw
    d = _guarded(nd, torch.float32, float("nan"), GUARD_F)
    n = _guarded(nn, torch.int64, -1, GUARD_I)
    ws = torch.empty(256, dtype=torch.uint8, device="cuda")
    _cabi.check(lib.bacs_class_distance(fd.data_ptr(), BF16, B, D, h, w, pd.data_ptr(), Kc, d[GUARD:].data_ptr(),
                                        n[GUARD:].data_ptr() if want_nearest else None, ws.data_ptr(), 256, _stream()),
                "bacs_class_distance")
    torch.cuda.synchronize()
    assert _guards_intact(d, nd, GUARD_F), "dist2 guard band written"
    assert _guards_intact(n, nn, GUARD_I), "nearest guard band written"
    if not want_nearest:
        assert bool((n[GUARD:GUARD + nn] == -1).all()), "nearest written although NULL was passed"
    return d[GUARD:GUARD + nd].view(B, Kc, hw), (n[GUARD:GUARD + nn].view(B, hw) if want_nearest else None)


def check_distance(c, got, near, ref, M):
    exact = c.data in ("int", "tie")
    assert not bool(torch.isnan(got).any()), "dist2: %d entries unwritten" % int(torch.isnan(got).sum())
    tol = RTOL * M
    g64 = got.double()
    err = (g64 - ref).abs()
    bad = ~(err <= tol)
    assert not bool(bad.any()), "dist2: %d of %d out of bounds (worst ratio %.3g)" % (
        int(bad.sum()), bad.numel(), float((err / tol.clamp(min=1e-300)).max()))
    _ratio("dist2", float((err / tol.clamp(min=1e-300)).max()))
    assert float(got.min()) >= 0.0
    if exact:
        assert torch.equal(g64, ref), "dist2 (integers): %d not bit-equal to fp64" % int((g64 != ref).sum())
    if c.data != "trap":
        assert float(got[c.B - 1, 0, c.hw - 1]) <= float(tol[c.B - 1, 0, c.hw - 1])
    if near is None:
        return
    assert int(near.min()) >= 0 and int(near.max()) < c.Kc, "nearest outside [0, Kc): %d..%d" % (
        int(near.min()), int(near.max()))
    own = got.argmin(1)                                  # the first (lowest) class among the smallest distances
    assert torch.equal(near, own), "nearest: %d pixels not the lowest class of the smallest distance" % int(
        (near != own).sum())
    rmin, amin = ref.min(1)[0], ref.argmin(1)
    rn = ref.gather(1, near.unsqueeze(1))[:, 0]
    allow = tol.gather(1, near.unsqueeze(1))[:, 0] + tol.gather(1, amin.unsqueeze(1))[:, 0]
    gap = rn - rmin
    assert bool((gap <= allow).all()), "nearest: %d pixels not within the allowance of the minimum" % int(
        (gap > allow).sum())
    _ratio("nearest", float((gap / allow.clamp(min=1e-300)).max()))
    if exact:
        assert torch.equal(near, amin), "nearest (integers): %d pixels differ from the fp64 arg-min" % int(
            (near != amin).sum())


# --------------------------------------------------------------------------------------
# bacs_class_sums: the plan
# --------------------------------------------------------------------------------------
NTS = (4, 8, 12, 16, 20)


def cs_plan(dt, D, hw, K, feat_off=0, lab_off=0, no_mma=False):
    """("mma", dtype, NT) or ("table", dtype, vec, warps) as bacs_class_sums picks them (byte offsets of features and
    labels past 512-byte aligned allocations)"""
    aligned = feat_off % 16 == 0 and lab_off % 16 == 0
    if dt != "f32" and hw % 32 == 0 and D % 16 == 0 and K <= 160 and aligned and not no_mma:
        nt = (K + 7) // 8
        return ("mma", dt, next(n for n in NTS if n >= nt))
    warps = min(8, 200 * 1024 // (K * 32 * 4))
    return ("table", dt, int(hw % 8 == 0 and aligned), warps)


@dataclass(frozen=True)
class Cs:
    name: str
    dt: str
    B: int
    D: int
    h: int
    w: int
    K: int
    feat_off: int = 0       # bytes
    lab_off: int = 0        # bytes
    feats: str = "randn"    # or "int": integers in [-8, 8]

    @property
    def hw(self):
        return self.h * self.w

    def plan(self, no_mma=False):
        return cs_plan(self.dt, self.D, self.hw, self.K, self.feat_off, self.lab_off, no_mma)


# mma shapes: D/16 odd (the block's second warp idle) or even; h*w = 32 and h*w % 64 = 32 (the second half of the
# two-chunk unroll finds no pixels) or a multiple of 64
MMA_SHAPES = [(3, 16, 4, 8), (2, 48, 8, 12), (3, 32, 8, 8), (2, 80, 10, 16), (4, 64, 16, 16)]


def cs_cases():
    cases = []
    for di, dt in enumerate(("bf16", "f16")):
        for i, nt in enumerate(NTS):
            for hi, K in enumerate((nt * 8 - 31 if nt > 4 else 1, nt * 8)):
                B, D, h, w = MMA_SHAPES[(2 * i + hi + di) % len(MMA_SHAPES)]
                cases.append(Cs("mma-%s-nt%d-k%d" % (dt, nt, K), dt, B, D, h, w, K, feats=("int", "randn")[hi]))
    cases += [
        Cs("ade-bf16-k151", "bf16", 4, 512, 32, 32, 151),
        Cs("k161-bf16", "bf16", 3, 32, 8, 8, 161),                             # mma shape, one class too many
        Cs("k161-f16-int", "f16", 2, 48, 8, 12, 161, feats="int"),
        Cs("f32-vec", "f32", 3, 20, 8, 8, 21),
        Cs("f32-odd-hw", "f32", 2, 40, 7, 9, 21, feats="int"),
        Cs("f32-feat-off8", "f32", 2, 24, 8, 8, 33, feat_off=8),
        Cs("f32-lab-off8", "f32", 2, 24, 8, 8, 33, lab_off=8),
        Cs("bf16-vec", "bf16", 3, 24, 5, 8, 100),
        Cs("bf16-odd-hw", "bf16", 2, 40, 5, 7, 151, feats="int"),
        Cs("bf16-feat-off8", "bf16", 2, 32, 8, 8, 21, feat_off=8),             # mma shape, misaligned features
        Cs("f16-vec", "f16", 2, 24, 8, 8, 21),
        Cs("f16-lab-off8", "f16", 2, 32, 8, 8, 64, lab_off=8),                 # mma shape, misaligned labels
        Cs("f16-odd-k256", "f16", 1, 8, 3, 3, 256),
        Cs("bf16-k256-int", "bf16", 3, 16, 8, 16, 256, feats="int"),
        Cs("f32-w6-k256", "f32", 2, 32, 8, 8, 256),
        Cs("bf16-w4-k400", "bf16", 2, 10, 8, 8, 400),
        Cs("f16-w2-k800", "f16", 2, 7, 8, 8, 800, feats="int"),
        Cs("f32-w1-k1024", "f32", 2, 3, 6, 6, 1024),
    ]
    return cases


CS_CASES = cs_cases()
CS_PARAMS = [(c, False) for c in CS_CASES] + [(c, True) for c in CS_CASES if c.plan()[0] == "mma"]


# --------------------------------------------------------------------------------------
# bacs_class_sums: inputs, reference, run, checks
# --------------------------------------------------------------------------------------
def cs_inputs(c):
    """features [B, D, h, w] in the storage type and int64 labels [B, h, w] on the host.  Labels: random classes,
    a long run of class K - 1 (255 at K = 256), values to skip (negative, K, 255 when K <= 255, +-2^40), class 0 at
    exactly one pixel and class 1 absent (K >= 3)."""
    g = torch.Generator().manual_seed(31 * c.K + c.D + c.hw)
    B, D, h, w, K = c.B, c.D, c.h, c.w, c.K
    if c.feats == "int":
        f = torch.randint(-8, 9, (B, D, h, w), generator=g).float()
    else:
        f = torch.randn(B, D, h, w, generator=g)
    f = f.to(DTYPES[c.dt])
    lab = torch.randint(0, K, (B, h, w), generator=g)
    flat = lab.view(B, -1)
    flat[0, : (h * w) // 2] = K - 1
    u = torch.rand(B, h, w, generator=g)
    for i, v in enumerate((-1, -(2 ** 40), K, 2 ** 40, 255, -3)):
        lab[(u >= 0.88 + 0.02 * i) & (u < 0.9 + 0.02 * i)] = v
    if K >= 3:
        lab[(lab == 0) | (lab == 1)] = -1
        lab[B - 1, h - 1, w - 1] = 0
    return f, lab


def cs_reference(f, lab, K):
    """fp64 (sums [K, D], sums of |terms| [K, D], counts [K])"""
    B, D = f.shape[:2]
    x = f.double().permute(0, 2, 3, 1).reshape(-1, D)
    ll = lab.reshape(-1)
    keep = (ll >= 0) & (ll < K)
    s = torch.zeros(K, D, dtype=torch.float64).index_add_(0, ll[keep], x[keep])
    a = torch.zeros(K, D, dtype=torch.float64).index_add_(0, ll[keep], x[keep].abs())
    return s, a, torch.bincount(ll[keep], minlength=K)


def _at_offset(host, off_bytes):
    """host tensor on the device, `off_bytes` past the start of a 512-byte aligned allocation"""
    es = host.element_size()
    assert off_bytes % es == 0
    o = off_bytes // es
    flat = torch.zeros(host.numel() + o, dtype=host.dtype, device="cuda")
    flat[o:] = host.reshape(-1).cuda()
    return flat[o:].view(host.shape)


def run_sums(c, fd, ld):
    """bacs_class_sums through the C ABI on device tensors (workspace all NaN); sums [K, D]"""
    from bacs_b200 import _cabi
    lib = _lib()
    B, D, K = c.B, c.D, c.K
    nbytes = lib.bacs_class_sums_workspace_bytes(B, D, K)
    ws = torch.full((nbytes,), 0xFF, dtype=torch.uint8, device="cuda")
    n = K * D
    s = _guarded(n, torch.float64, float("nan"), GUARD_F)
    _cabi.check(lib.bacs_class_sums(fd.data_ptr(), DT_ID[c.dt], B, D, c.h, c.w, ld.data_ptr(), K, s[GUARD:].data_ptr(),
                                    ws.data_ptr(), nbytes, _stream()), "bacs_class_sums")
    torch.cuda.synchronize()
    assert _guards_intact(s, n, GUARD_F), "sums guard band written"
    return s[GUARD:GUARD + n].view(K, D)


def check_sums(c, got, f, lab, want, absw):
    got = got.cpu()
    assert not bool(torch.isnan(got).any()), "sums: %d entries unwritten" % int(torch.isnan(got).sum())
    tol = RTOL * absw
    err = (got - want).abs()
    bad = ~(err <= tol)
    assert not bool(bad.any()), "sums: %d of %d out of bounds (worst ratio %.3g)" % (
        int(bad.sum()), bad.numel(), float((err / tol.clamp(min=1e-300)).max()))
    _ratio("sums", float((err / tol.clamp(min=1e-300)).max()))
    if c.feats == "int":
        assert torch.equal(got, want), "sums (integers): %d not bit-equal to fp64" % int((got != want).sum())
    if c.K >= 3:
        assert torch.equal(got[0], f[c.B - 1, :, c.h - 1, c.w - 1].double()), "one-pixel class"
        assert bool((got[1] == 0).all()), "absent class"


# --------------------------------------------------------------------------------------
# coverage of the plans
# --------------------------------------------------------------------------------------
CD_BOUNDARIES = {(160, 512): 4, (256, 368): 4, (224, 416): 4, (160, 480): 8}      # accepted (Kc, D) -> stages


def cd_reached(sms):
    items = set()
    for c in cd_cases(sms):
        p = c.plan(sms)
        assert p.ok, c.name
        if p.tiles_max == 1:
            items.add("tiles/CTA 1")
        if p.tiles_max == 2:
            items.add("tiles/CTA 2")
        if p.tiles_max >= 3 and p.n_tiles % p.grid:
            items.add("tiles/CTA >= 3, uneven")
        if p.laps >= 2:
            items.add("two laps of the ring")
        if p.tiles_max >= 2:
            items.add("nearest NULL and given, tiles/CTA >= 2")
        if p.Dp % 32 == 16:
            items.add("last chunk of 16 channels")
        items.add("nchunks %d" % p.nchunks)
        items.add("stages %d" % p.stages)
        items.add("Kc %d" % c.Kc)
        items.add("hw %d" % c.hw)
        if c.hw > TILE_M and c.hw % TILE_M:
            items.add("multi-tile image, last tile partial")
        if (c.Kc, c.D) in CD_BOUNDARIES and p.stages == CD_BOUNDARIES[(c.Kc, c.D)]:
            items.add("accepted %d x %d, %d stages" % (c.Kc, c.D, p.stages))
        if (c.D, c.hw, c.Kc) == (512, 1024, 150):
            items.add("ADE B=%d" % c.B)
        if c.data == "tie":
            items.add("ties across warpgroups")
        if c.data == "trap" and c.Kc % 32:
            items.add("padding trap")
        if c.data == "offset":
            items.add("offset 50")
        if c.data in ("int", "tie"):
            items.add("exact integers")
    for name, over, msg in CD_REFUSALS:
        a = dict(CD_BASE, **over)
        if "fit one SM" in msg:
            assert not cd_plan(a["B"], a["D"], a["h"] * a["w"], a["Kc"], sms).ok, name
            items.add("refused %d x %d" % (a["Kc"], a["D"]))
    return items


CD_WANT = ({"tiles/CTA 1", "tiles/CTA 2", "tiles/CTA >= 3, uneven", "two laps of the ring",
            "nearest NULL and given, tiles/CTA >= 2", "last chunk of 16 channels", "stages 8", "stages 4",
            "multi-tile image, last tile partial", "ADE B=24", "ADE B=48", "ties across warpgroups", "padding trap",
            "offset 50", "exact integers", "refused 161 x 512", "refused 256 x 376", "refused 224 x 432",
            "refused 10 x 520"}
           | {"nchunks %d" % n for n in (1, 2, 3, 4, 5, 7, 12, 16)}
           | {"Kc %d" % k for k in (1, 31, 32, 33, 97, 150, 255, 256)}
           | {"hw %d" % n for n in (8, 120, 128, 136, 1000)}
           | {"accepted %d x %d, %d stages" % (k, d, s) for (k, d), s in CD_BOUNDARIES.items()})


def cs_reached():
    items = set()
    for c, no_mma in CS_PARAMS:
        p = c.plan(no_mma)
        if p[0] == "mma":
            nt = p[2]
            items.add("mma %s NT %d" % (p[1], nt))
            if c.K in (nt * 8 - 31 if nt > 4 else 1, nt * 8):
                items.add("mma %s NT %d K %d" % (p[1], nt, c.K))
            if (c.D // 16) % 2:
                items.add("mma D/16 odd")
            if c.hw == 32:
                items.add("mma hw 32")
            if c.hw > 32 and c.hw % 64 == 32:
                items.add("mma hw % 64 = 32")
        else:
            _, dt, vec, warps = p
            items.add("table %s vec %d" % (dt, vec))
            if warps == 1 or c.D % warps:
                items.add("table %d warps, D %% warps != 0 or 1 warp" % warps)
            if not vec:
                if c.hw % 8:
                    items.add("vec 0: h*w % 8 != 0")
                if c.feat_off % 16:
                    items.add("vec 0: feature pointer + 8 bytes")
                if c.lab_off % 16:
                    items.add("vec 0: label pointer + 8 bytes")
            mma_shape = c.dt != "f32" and c.hw % 32 == 0 and c.D % 16 == 0 and c.feat_off % 16 == 0 and c.lab_off % 16 == 0
            if mma_shape and c.K == 161 and not no_mma:
                items.add("K 161 on an mma shape: table")
            if no_mma:
                items.add("BACS_NO_SUMS_MMA")
        if c.K == 256:
            items.add("K 256: label 255 summed")
    return items


CS_WANT = ({"mma %s NT %d" % (dt, nt) for dt in ("bf16", "f16") for nt in NTS}
           | {"mma %s NT %d K %d" % (dt, nt, k) for dt in ("bf16", "f16") for nt in NTS
              for k in ((nt * 8 - 31 if nt > 4 else 1), nt * 8)}
           | {"table %s vec %d" % (dt, v) for dt in DTYPES for v in (0, 1)}
           | {"table %d warps, D %% warps != 0 or 1 warp" % w for w in (8, 6, 4, 2, 1)}
           | {"mma D/16 odd", "mma hw 32", "mma hw % 64 = 32", "vec 0: h*w % 8 != 0", "vec 0: feature pointer + 8 bytes",
              "vec 0: label pointer + 8 bytes", "K 161 on an mma shape: table", "BACS_NO_SUMS_MMA",
              "K 256: label 255 summed"})


def test_class_family_coverage():
    """the case tables reach every plan item of both ops on this device's SM count"""
    sms = sm_count()
    if _on_gpu():
        assert _lib().bacs_device_sm_count() == sms
    got = cd_reached(sms)
    print("\nclass_distance: reached %d of %d plan items (%d SMs)" % (len(got & CD_WANT), len(CD_WANT), sms))
    assert got >= CD_WANT, "not reached: %s" % sorted(CD_WANT - got)
    got = cs_reached()
    print("class_sums: reached %d of %d plan items" % (len(got & CS_WANT), len(CS_WANT)))
    assert got >= CS_WANT, "not reached: %s" % sorted(CS_WANT - got)


def test_class_distance_plan_arithmetic():
    """the shared-memory boundaries of the host plan (224 KB = 229376 bytes)"""
    assert cd_smem(256, 368, 4) == SMEM_CAP
    for (Kc, D), stages in CD_BOUNDARIES.items():
        p = cd_plan(1, D, 8, Kc, CPU_SMS)
        assert p.ok and p.stages == stages, (Kc, D, p)
    for Kc, D in ((161, 512), (256, 376), (224, 432), (1, 520)):
        assert not cd_plan(1, D, 8, Kc, CPU_SMS).ok
    assert cd_plan(1, 496, 8, 160, CPU_SMS).stages == 4           # one k-block past the largest 8-stage shape


# --------------------------------------------------------------------------------------
# bacs_class_distance tests
# --------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("c", cd_cases(sm_count()), ids=lambda c: c.name)
def test_class_distance_against_fp64(c):
    f, p = cd_inputs(c)
    fd, pd = f.cuda(), p.cuda()
    ref, M = cd_reference(f, p)
    got, near = run_distance(fd, pd, c.B, c.D, c.h, c.w, c.Kc)
    check_distance(c, got, near, ref, M)
    got2, _ = run_distance(fd, pd, c.B, c.D, c.h, c.w, c.Kc, want_nearest=False)
    assert torch.equal(_bits(got2), _bits(got)), "dist2 without nearest differs"


@gpu
@pytest.mark.parametrize("D", [96, 160, 200])
def test_class_distance_independent_of_batch_split(D):
    """chunk counts 3, 5 and 7 rotate the builder warpgroups from tile to tile of a CTA: the batched call (2 or 3
    tiles per CTA) gives the same bits as per-image calls, two halves, a second call and a call without nearest"""
    sms = sm_count()
    B = 5 * sms // 16 + 1
    c = Cd("split-d%d" % D, B, D, 32, 32, 40, "randn")
    assert c.plan(sms).tiles_min >= 2
    f, p = cd_inputs(c)
    fd, pd = f.cuda(), p.cuda()
    full, near = run_distance(fd, pd, B, D, 32, 32, 40)
    check_distance(c, full, near, *cd_reference(f, p))
    parts = {"per image": [run_distance(fd[b:b + 1], pd, 1, D, 32, 32, 40) for b in range(B)],
             "halves": [run_distance(fd[:B // 2], pd, B // 2, D, 32, 32, 40),
                        run_distance(fd[B // 2:], pd, B - B // 2, D, 32, 32, 40)],
             "again": [run_distance(fd, pd, B, D, 32, 32, 40)]}
    for what, runs in parts.items():
        d2 = torch.cat([r[0] for r in runs])
        nn = torch.cat([r[1] for r in runs])
        diff = int((_bits(d2) != _bits(full)).sum())
        assert diff == 0, "%s: %d distances differ from the batched call" % (what, diff)
        assert torch.equal(nn, near), what
    d2, _ = run_distance(fd, pd, B, D, 32, 32, 40, want_nearest=False)
    assert torch.equal(_bits(d2), _bits(full)), "without nearest"


@pytest.mark.parametrize("row", CD_REFUSALS, ids=[r[0] for r in CD_REFUSALS])
def test_class_distance_refusals(row):
    """refused with a message before any launch; the outputs stay untouched (no device needed)"""
    from bacs_b200 import _cabi
    lib = _lib()
    _, over, msg = row
    a = dict(CD_BASE, **over)
    B, D, h, w, Kc = a["B"], a["D"], a["h"], a["w"], a["Kc"]
    dev = _dev()
    fb = torch.zeros(max(B * D * h * w, 1) + 8, dtype=torch.bfloat16, device=dev)
    pb = torch.zeros(max(Kc * D, 1) + 8, dtype=torch.bfloat16, device=dev)
    nd, nn = max(B * Kc * h * w, 1), B * h * w
    d = _guarded(nd, torch.float32, float("nan"), GUARD_F)
    n = _guarded(nn, torch.int64, -1, GUARD_I)
    ptr = {"feat": fb.data_ptr() + a["feat_off"], "protos": pb.data_ptr() + a["proto_off"], "dist2": d[GUARD:].data_ptr()}
    if a["null"]:
        ptr[a["null"]] = None
    st = lib.bacs_class_distance(ptr["feat"], a["dtype"], B, D, h, w, ptr["protos"], Kc, ptr["dist2"],
                                 n[GUARD:].data_ptr(), None, 0, _stream() if _on_gpu() else None)
    assert st != 0 and msg in _cabi.last_error(), (st, _cabi.last_error())
    if _on_gpu():
        torch.cuda.synchronize()
    assert _guards_intact(d, nd, GUARD_F) and bool(torch.isnan(d[GUARD:GUARD + nd]).all())
    assert _guards_intact(n, nn, GUARD_I) and bool((n[GUARD:GUARD + nn] == -1).all())


# --------------------------------------------------------------------------------------
# bacs_class_sums tests
# --------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("c,no_mma", CS_PARAMS,
                         ids=["%s%s" % (c.name, "-no-mma" if m else "") for c, m in CS_PARAMS])
def test_class_sums_against_fp64(c, no_mma, monkeypatch):
    if no_mma:
        monkeypatch.setenv("BACS_NO_SUMS_MMA", "1")          # read by bacs_class_sums on every call
    else:
        monkeypatch.delenv("BACS_NO_SUMS_MMA", raising=False)
    f, lab = cs_inputs(c)
    want, absw, counts = cs_reference(f, lab, c.K)
    fd, ld = _at_offset(f, c.feat_off), _at_offset(lab, c.lab_off)
    got = run_sums(c, fd, ld)
    check_sums(c, got, f, lab, want, absw)
    if c.K <= 256:
        # ops.class_sums: the same kernel (same bits) and the counts from the label histogram (labels at an 8-byte
        # offset are copied for it)
        from bacs_b200 import ops
        s2, n2 = ops.class_sums(fd, ld, c.K)
        assert torch.equal(s2.cpu(), got.cpu())
        assert torch.equal(n2.cpu(), counts), "counts"


def _sums_kernel_key(name, dt):
    m = re.search(r"class_sums_mma_kernel<\s*([\w:]+)\s*,\s*(\d+)\s*>", name)
    tn = {"__nv_bfloat16": "bf16", "__half": "f16", "float": "f32"}
    if m:
        return ("mma", tn[m.group(1).split("::")[-1]], int(m.group(2)))
    m = re.search(r"class_sums_kernel<\s*([\w:]+)\s*>", name)
    assert m, name
    return ("table", tn[m.group(1).split("::")[-1]])


@gpu
def test_class_sums_plan_matches_kernel_names(monkeypatch):
    """the host plan names the kernel the library launches: one profiled call per instantiation"""
    from torch.profiler import ProfilerActivity, profile
    monkeypatch.delenv("BACS_NO_SUMS_MMA", raising=False)
    first = {}
    for c in CS_CASES:
        p = c.plan()
        first.setdefault(p[:3] if p[0] == "mma" else p[:2], c)
    assert len(first) == 13, sorted(first)
    for key, c in sorted(first.items()):
        f, lab = cs_inputs(c)
        fd, ld = _at_offset(f, c.feat_off), _at_offset(lab, c.lab_off)
        run_sums(c, fd, ld)                                  # warm up outside the profile
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            run_sums(c, fd, ld)
        names = {e.key for e in prof.key_averages() if "class_sums" in e.key and "finalize" not in e.key}
        assert len(names) == 1, (c.name, names)
        assert _sums_kernel_key(names.pop(), c.dt) == key, (c.name, key)
