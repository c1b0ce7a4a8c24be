"""The seen / unseen detector heads (csrc/seen.cu) and the pixel kernels' use of their logits, against a float64
reference evaluated on the host from the exact values the kernels read (features rounded to their storage type, fp32
prototypes, head parameters and logits).

Error model: per element, never normalised by the largest entry.  A value that is a sum of terms is allowed
1e-5 x (the sum of the terms' absolute values) of error: the kernels' fp32 summation order changes with the cluster
size, the table chunking and the pixels per thread, and this bound holds for every order.  Where a kernel uses the
fast fp32 intrinsics (ex2 / rcp / lg2 approximations, absolute error ~2^-21 near 1), the bound adds that absolute
error per term, and says so where it does.  16-bit gradients are within one ulp of the storage type of the float64
value rounded to that type."""
import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu

EPS32 = 2.0 ** -23
RTOL = 1e-5
DTYPES = {"f32": torch.float32, "bf16": torch.bfloat16, "f16": torch.float16}
TMAXES = (2, 4, 6, 8, 12, 16, 32)


@pytest.fixture(scope="module")
def ops():
    from bacs_b200 import ops as _ops
    return _ops


@pytest.fixture(scope="module")
def cabi():
    from bacs_b200 import _cabi
    return _cabi


def sm_count():
    return torch.cuda.get_device_properties(0).multi_processor_count


def on_device(n_elems, dtype, offset, gen, scale=2.0):
    """A contiguous CUDA tensor of n_elems values whose data pointer is `offset` elements past an allocation (the
    caching allocator's blocks are 512-byte aligned, so offset 1 misaligns every vector width)."""
    host = (torch.randn(n_elems + offset, generator=gen) * scale).to(dtype)
    return host.cuda()[offset:]


# --------------------------------------------------------------------------------------
# float64 references
# --------------------------------------------------------------------------------------
def seen_logits64(feat, proto, weight, bias):
    """-> (z64, abs64) [B,T,h,w]: z = bias + sum_c w[t,c] |sig(x) - sig(p[t,c])| and |bias| + sum_c |w[t,c]| |...|,
    one head at a time so that [B,T,D,hw] never exists."""
    x = feat.detach().cpu().double()
    B, D, h, w = x.shape
    sx = torch.sigmoid(x).reshape(B, D, h * w)
    sp = torch.sigmoid(proto.detach().cpu().double())
    W = weight.detach().cpu().double().reshape(-1, D)
    bb = bias.detach().cpu().double().reshape(-1)
    T = W.shape[0]
    z = torch.empty(B, T, h * w, dtype=torch.float64)
    a = torch.empty_like(z)
    for t in range(T):
        d = (sx - sp[t].view(1, D, 1)).abs()
        z[:, t] = torch.einsum("c,bcq->bq", W[t], d) + bb[t]
        a[:, t] = torch.einsum("c,bcq->bq", W[t].abs(), d) + bb[t].abs()
    return z.view(B, T, h, w), a.view(B, T, h, w)


def ac_geometry(n_in, n_out):
    """align_corners=True source geometry exactly as ATen / the kernels compute it: fp32 scale (in-1)/(out-1), fp32
    source coordinate scale*dst, fp32 weights.  The float64 references interpolate with these weights, so only the
    blend's own rounding is left between them and a kernel."""
    scale = torch.tensor(float(n_in - 1), dtype=torch.float32) / float(n_out - 1) if n_out > 1 else \
        torch.tensor(0.0, dtype=torch.float32)
    src = torch.arange(n_out, dtype=torch.float32) * scale
    i0 = src.long().clamp(max=n_in - 1)
    i1 = torch.where(i0 < n_in - 1, i0 + 1, i0)
    w1 = src - i0.float()
    w0 = 1.0 - w1
    return i0, i1, w0.double(), w1.double()


def up_ac64(z, s):
    """float64 align_corners=True x s up-sample of [..., h, w] (ATen's geometry, see ac_geometry)."""
    h, w = z.shape[-2:]
    y0, y1, wy0, wy1 = ac_geometry(h, h * s)
    x0, x1, wx0, wx1 = ac_geometry(w, w * s)
    rows = z[..., y0, :] * wy0.view(-1, 1) + z[..., y1, :] * wy1.view(-1, 1)
    return rows[..., x0] * wx0 + rows[..., x1] * wx1


def up_hp64(x, H, W):
    """float64 align_corners=False up-sample (the network's own sem_logits -> image up-sample), fp32 geometry."""
    def geo(n_in, n_out):
        scale = torch.tensor(float(n_in), dtype=torch.float32) / float(n_out)
        src = ((torch.arange(n_out, dtype=torch.float32) + 0.5) * scale - 0.5).clamp(min=0.0)
        i0 = src.long().clamp(max=n_in - 1)
        i1 = torch.where(i0 < n_in - 1, i0 + 1, i0)
        w1 = src - i0.float()
        return i0, i1, (1.0 - w1).double(), w1.double()
    y0, y1, wy0, wy1 = geo(x.shape[-2], H)
    x0, x1, wx0, wx1 = geo(x.shape[-1], W)
    rows = x[..., y0, :] * wy0.view(-1, 1) + x[..., y1, :] * wy1.view(-1, 1)
    return rows[..., x0] * wx0 + rows[..., x1] * wx1


def head_backward64(feat, proto_t, weight_t, gz, scale):
    """fp64 autograd of scale * sum(gz * z_t): (dW, db, dfeat, |terms| of dW, |terms| of db)."""
    x = feat.detach().cpu().double().requires_grad_(True)
    w = weight_t.detach().cpu().double().requires_grad_(True)
    b = torch.zeros(1, dtype=torch.float64, requires_grad=True)
    B, D, h, wd = x.shape
    g = gz.detach().cpu().double().reshape(B, 1, h, wd)
    d = (torch.sigmoid(x) - torch.sigmoid(proto_t.detach().cpu().double()).view(1, D, 1, 1)).abs()
    z = (d * w.view(1, D, 1, 1)).sum(1, keepdim=True) + b
    (scale * (g * z).sum()).backward()
    dw_abs = abs(scale) * (g.abs() * d.detach()).sum((0, 2, 3))
    db_abs = abs(scale) * g.abs().sum().reshape(1)
    return w.grad, b.grad, x.grad, dw_abs, db_abs


# --------------------------------------------------------------------------------------
# seen_logits: host mirror of the launch plan
# --------------------------------------------------------------------------------------
def seen_plan(T, D, B, h, w, elem_bytes, offset, sms):
    """(TMAX, PX, cs, n_chunks) that seen_logits_impl (csrc/seen.cu:386-401) picks: the head-count bucket TMAX, the
    pixels per lane PX (4 up to 8 heads, 2 up to 16, else 1; 1 when hw % PX != 0 or the feature pointer is not
    PX * elem_bytes aligned), the thread-block cluster size cs (doubled while the grid, at `per_sm` resident CTAs,
    still fits the machine in one wave and every CTA keeps >= 16 channels) and the number of channel-table chunks
    the leader CTA loads (32 KB table of 2*TMAX floats per channel, a multiple of 8 channels)."""
    hw = h * w
    tmax = next(m for m in TMAXES if T <= m)
    px = 4 if tmax <= 8 else (2 if tmax <= 16 else 1)
    if hw % px != 0 or (offset * elem_bytes) % (px * elem_bytes) != 0:
        px = 1
    ps = 32 * px
    n_pb = (hw + ps - 1) // ps
    per_sm = 3 if tmax * px <= 32 else (2 if tmax * px <= 48 else 1)
    cs = 1
    while cs < 8 and n_pb * B * cs * 2 <= per_sm * sms and D // (2 * cs) >= 16:
        cs *= 2
    stride = 2 * tmax
    per = (D + cs - 1) // cs
    chunk = max(8, (32 * 1024 // 4) // stride // 8 * 8)
    if chunk > per:
        chunk = (per + 7) // 8 * 8
    return tmax, px, cs, (per + chunk - 1) // chunk


def push_overlaps_table(T, D, B, h, w, elem_bytes, offset, sms):
    """True when the cluster's partial sums land inside the leader's channel table: the kernel stores the per-warp
    sums at smem[0, 8*T*32*PX) and receives the other CTAs' sums right after them, while every chunk's channel
    table spans up to smem[0, chunk*2*TMAX).  Such a launch depends on the cluster barrier between the table loop and the pushes."""
    tmax, px, cs, _ = seen_plan(T, D, B, h, w, elem_bytes, offset, sms)
    per = (D + cs - 1) // cs
    chunk = min(max(8, (32 * 1024 // 4) // (2 * tmax) // 8 * 8), (per + 7) // 8 * 8)
    return cs > 1 and chunk * 2 * tmax > 8 * T * 32 * px


# (T, D, B, h, w, feature offset in elements): every row runs in fp32, bf16 and fp16.  The path of each row is what
# seen_plan gives on a 148-SM B200; test_seen_case_table_covers_every_path re-derives it on the device at hand.
SEEN_CASES = [
    (1, 64, 2, 16, 16, 0),     # T=1 (first task), TMAX 2, PX 4, cs 4
    (2, 100, 1, 33, 33, 0),    # TMAX 2, odd hw (VOC 513/528 crop at stride 16) -> PX 1; D=100 not a multiple of cs 4
    (2, 64, 2, 16, 16, 1),     # TMAX 2, feature pointer one element past the allocation -> PX 1
    (3, 257, 2, 6, 7, 0),      # TMAX 4, hw=42 (even, not % 4) -> PX 1; D=257: cs 8 with a ragged last CTA
    (4, 48, 3, 20, 20, 0),     # TMAX 4, PX 4, cs 2 (D=48 stops the doubling)
    (5, 64, 8, 32, 32, 0),     # TMAX 6, PX 4, cs 4
    (6, 96, 2, 12, 12, 1),     # TMAX 6, misaligned -> PX 1, cs 4
    (7, 64, 16, 40, 40, 0),    # TMAX 8, PX 4, 1600 pixels = 12.5 CTA spans (partial last span), cs 2
    (8, 32, 24, 48, 48, 0),    # TMAX 8, PX 4, cs 1 (432 CTAs already fill the machine)
    (8, 40, 2, 9, 9, 0),       # TMAX 8, odd hw -> PX 1, cs 2
    (9, 128, 2, 10, 10, 0),    # TMAX 12, PX 2, cs 8
    (11, 256, 2, 33, 33, 0),   # TMAX 12 (VOC 10-1 last task), odd hw -> PX 1, cs 4
    (12, 80, 4, 16, 18, 0),    # TMAX 12, PX 2, 288 pixels = 4.5 CTA spans, cs 4
    (12, 80, 2, 6, 7, 0),      # TMAX 12, hw=42 (even, not % 4): still PX 2, cs 4
    (12, 360, 16, 30, 30, 0),  # TMAX 12, PX 2, cs 1 (240 CTAs), D=360: two table chunks (336 + 24 channels)
    (13, 64, 2, 16, 16, 1),    # TMAX 16, misaligned -> PX 1, cs 4
    (16, 600, 4, 40, 45, 0),   # TMAX 16, PX 2, cs 2: 300 channels per CTA = two chunks of 256
    (16, 48, 2, 7, 7, 0),      # TMAX 16, odd hw -> PX 1, cs 2
    (17, 64, 1, 5, 7, 0),      # TMAX 32 (first count past 16), PX 1, cs 4
    (17, 300, 3, 9, 9, 0),     # TMAX 32, cs 8, 38 channels per CTA (not a multiple of 8)
    # TMAX 32, cs 4: the leader's 80-channel table (5120 floats) reaches into the region the other CTAs push their sums
    # to (from 8*17*32 = 4352 floats).  The pushes used to start without waiting for the leader to finish with its
    # table, a race; every CTA now passes a cluster barrier between its table loop and the pushes.
    (17, 300, 20, 9, 9, 0),
    (24, 300, 3, 9, 9, 0),     # TMAX 32, cs 8
    (32, 288, 8, 30, 30, 0),   # TMAX 32, cs 1: three table chunks (128 + 128 + 32 channels)
    (32, 512, 4, 29, 32, 0),   # TMAX 32, cs 2: 256 channels per CTA = two chunks (push region right after the table)
]


def _seen_inputs(T, D, B, h, w, dtype, offset, seed):
    g = torch.Generator().manual_seed(seed)
    feat = on_device(B * D * h * w, dtype, offset, g).view(B, D, h, w)
    proto = (torch.randn(T, D, generator=g) * 1.5).cuda()
    weight = (torch.randn(T, D, generator=g) * 0.2).cuda()
    bias = torch.randn(T, generator=g).cuda()
    return feat, proto, weight, bias


def _case_id(c):
    return "T%d-D%d-B%d-%dx%d%s" % (c[0], c[1], c[2], c[3], c[4], "-off" if c[5] else "")


def test_seen_case_table_covers_every_path():
    """Every (dtype, TMAX, PX) instantiation of seen_logits_kernel and every cluster size is reached by SEEN_CASES
    (with this device's SM count), and the multi-chunk table is reached with and without a cluster."""
    sms = sm_count()
    reached, sizes, chunked, overlap = set(), set(), set(), 0
    for (T, D, B, h, w, off) in SEEN_CASES:
        for name, dt in DTYPES.items():
            tmax, px, cs, n_chunks = seen_plan(T, D, B, h, w, dt.itemsize, off, sms)
            reached.add((name, tmax, px))
            sizes.add(cs)
            if n_chunks > 1:
                chunked.add((tmax, cs > 1))
            overlap += push_overlaps_table(T, D, B, h, w, dt.itemsize, off, sms)
    want = {(n, tm, px) for n in DTYPES for tm in TMAXES
            for px in ((4, 1) if tm <= 8 else ((2, 1) if tm <= 16 else (1,)))}
    print("seen_logits_kernel instantiations reached: %d of %d; cluster sizes %s; chunked tables %s"
          % (len(reached & want), len(want), sorted(sizes), sorted(chunked)))
    assert reached == want, "not reached: %s" % sorted(want - reached)
    assert sizes == {1, 2, 4, 8}
    assert {c for _, c in chunked} == {False, True}
    assert {tm for tm, _ in chunked} >= {12, 16, 32}
    assert overlap > 0, "no case pushes cluster sums into the leader's table region"


@pytest.mark.parametrize("dname", list(DTYPES))
@pytest.mark.parametrize("case", SEEN_CASES, ids=_case_id)
def test_seen_logits_against_fp64(ops, case, dname):
    T, D, B, h, w, off = case
    dtype = DTYPES[dname]
    feat, proto, weight, bias = _seen_inputs(T, D, B, h, w, dtype, off, seed=T * 1000 + D)
    if off:
        assert feat.data_ptr() % 16 != 0
    z = ops.seen_logits(feat, proto, weight, bias)
    z64, abs64 = seen_logits64(feat, proto, weight, bias)
    err = (z.cpu().double() - z64).abs()
    bound = RTOL * abs64
    bad = err > bound
    assert not bool(bad.any()), "%d of %d entries beyond 1e-5 x sum|terms| (worst ratio %.3g)" % (
        int(bad.sum()), bad.numel(), float((err / bound).max()))
    # the heads as separate parameter tensors: same kernel, same bits; the accumulator cleared over all B*h*w
    ws = [weight[t].clone().reshape(1, D, 1, 1) for t in range(T)]
    bs = [bias[t].clone().reshape(1) for t in range(T)]
    zero = torch.full((B, h, w), float("nan"), device="cuda")
    zh = ops.seen_logits_heads(feat, proto, ws, bs, zero_out=zero)
    assert torch.equal(zh, z)
    assert bool((zero == 0).all()), "%d of %d accumulator entries not cleared" % (int((zero != 0).sum()), zero.numel())
    # fixed summation order: a second call gives the same bits
    assert torch.equal(ops.seen_logits(feat, proto, weight, bias), z)


def test_seen_logits_refuses_head_counts(ops, cabi):
    """The head-count range check itself (every buffer non-empty, so no null-pointer check answers first)."""
    g = torch.Generator().manual_seed(0)
    feat = torch.randn(1, 16, 4, 4, generator=g).cuda()
    proto, weight, bias = torch.zeros(33, 16).cuda(), torch.zeros(33, 16).cuda(), torch.zeros(33).cuda()
    z = torch.empty(1, 33, 4, 4).cuda()
    lib = cabi.load()
    for T in (0, 33):
        with pytest.raises(cabi.BacsError, match=r"T=%d not in \[1,32\]" % T):
            cabi.check(lib.bacs_seen_logits(feat.data_ptr(), cabi.F32, 1, 16, 4, 4, proto.data_ptr(), weight.data_ptr(),
                                            bias.data_ptr(), T, z.data_ptr(), ops._stream()), "bacs_seen_logits")
    with pytest.raises(cabi.BacsError, match=r"T=33 not in \[1,32\]"):
        ops.seen_logits(feat, proto, weight, bias)
    ws = [torch.zeros(1, 16, 1, 1).cuda() for _ in range(33)]
    with pytest.raises(cabi.BacsError, match=r"T=33 not in \[1,32\]"):
        ops.seen_logits_heads(feat, proto, ws, [torch.zeros(1).cuda() for _ in range(33)])


# --------------------------------------------------------------------------------------
# seen_upsample (align_corners=True)
# --------------------------------------------------------------------------------------
@pytest.mark.parametrize("scale", [8, 16])
@pytest.mark.parametrize("B,T,h,w", [(2, 3, 5, 7), (1, 2, 1, 6), (2, 1, 7, 1), (1, 1, 1, 1), (1, 4, 33, 33)])
def test_seen_upsample_against_fp64(ops, B, T, h, w, scale):
    g = torch.Generator().manual_seed(h * 100 + w)
    z = (torch.randn(B, T, h, w, generator=g) * 3).cuda()
    z64 = z.cpu().double()
    want = up_ac64(z64, scale)
    absum = up_ac64(z64.abs(), scale)          # sum of |weight * corner| of every output
    got = ops.seen_upsample(z, scale)
    # three fp32 roundings per level of the blend: <= 2 ulp of the absolute-term sum
    err = (got.cpu().double() - want).abs()
    assert bool((err <= 2 * EPS32 * absum).all()), "fp64: worst %.3g ulp" % float((err / (EPS32 * absum)).max())
    # Not bit-exact with F.interpolate: ATen's CUDA kernel evaluates h0*(w0*v00 + w1*v01) + h1*(w0*v10 + w1*v11) with
    # the products contracted into FMAs, ours rounds every product (the CPU oracle's op order).  Each is within 2 ulp
    # of the absolute-term sum of the fp64 value, so they are within 4 of each other.
    ref = F.interpolate(z, scale_factor=scale, mode="bilinear", align_corners=True)
    err = (got - ref).abs().cpu().double()
    assert bool((err <= 4 * EPS32 * absum).all()), "F.interpolate: worst %.3g ulp" % float((err / (EPS32 * absum)).max())
    # the geometry (source index and fp32 weight) is ATen's exactly: where an output lies on a source sample both
    # return that sample's bits
    Y0, _, _, wy1 = ac_geometry(h, h * scale)
    X0, _, _, wx1 = ac_geometry(w, w * scale)
    on_y, on_x = (wy1 == 0).nonzero().view(-1), (wx1 == 0).nonzero().view(-1)
    exact = got[..., on_y, :][..., on_x].cpu()
    assert torch.equal(exact, ref[..., on_y, :][..., on_x].cpu())
    assert torch.equal(exact, z.cpu()[..., Y0[on_y], :][..., X0[on_x]])
    # with the sigmoid: the blend's error through sigma' <= 1/4, plus a few ulp of the accurate fp32 sigmoid
    gs = ops.seen_upsample(z, scale, apply_sigmoid=True).cpu().double()
    sw = torch.sigmoid(want)
    ratio = (gs - sw).abs() / (0.5 * EPS32 * absum + 4 * EPS32 * sw)
    assert bool((ratio <= 1).all()), "sigmoid: worst ratio %.3g" % float(ratio.max())


# --------------------------------------------------------------------------------------
# seen_head_backward: vectorised (hw % 8 == 0, 16-byte aligned feature / gz / gradient) and scalar kernels
# --------------------------------------------------------------------------------------
# (dtype, B, D, h, w, feature offset, gz offset, want_dfeatures, scale (None: no scale pointer))
HEAD_BWD_CASES = [
    ("f32", 2, 48, 8, 8, 0, 0, True, 0.37),       # vectorised
    ("bf16", 3, 40, 16, 16, 0, 0, True, None),    # vectorised, no scale
    ("f16", 2, 33, 12, 12, 0, 0, True, 0.0),      # vectorised, scale 0: all gradients exactly 0
    ("f32", 1, 16, 48, 48, 0, 0, False, 0.37),    # vectorised, hw > 2048, no feature gradient
    ("bf16", 2, 24, 48, 50, 0, 0, True, 0.37),    # vectorised, hw > 2048
    ("f32", 2, 40, 5, 7, 0, 0, True, 0.37),       # scalar: hw % 8 != 0
    ("bf16", 2, 32, 8, 8, 0, 1, True, 0.37),      # scalar: gz not 16-byte aligned
    ("f16", 2, 32, 8, 8, 1, 0, True, None),       # scalar: features not 16-byte aligned
    ("f32", 2, 32, 8, 8, 1, 0, False, 0.0),       # scalar, no feature gradient, scale 0
    ("f32", 20, 24, 4, 5, 0, 0, True, 0.37),      # scalar, hw < 32, B > 16: 16 images side by side in a block
    ("bf16", 37, 16, 3, 3, 0, 0, True, None),     # scalar, hw = 9: 16 images side by side, B not a multiple
    ("f16", 19, 16, 2, 4, 0, 3, True, 0.37),      # scalar (gz misaligned), hw = 8, 16 images side by side
    ("f16", 2, 8, 45, 47, 0, 0, True, 0.37),      # scalar, hw > 2048 (odd): one image per block, 512 threads
    ("f32", 1, 8, 47, 47, 0, 0, False, None),     # scalar, hw > 2048
]


def _bwd_id(c):
    return "%s-B%d-D%d-%dx%d%s%s%s-s%s" % (c[0], c[1], c[2], c[3], c[4], "-foff" if c[5] else "",
                                            "-goff" if c[6] else "", "" if c[7] else "-nodf", c[8])


def _vec_path(feat, gz, dfeat_ptr_aligned, hw):
    return hw % 8 == 0 and feat.data_ptr() % 16 == 0 and gz.data_ptr() % 16 == 0 and dfeat_ptr_aligned


def _check_dfeat(got, want64, coef_abs, dtype, what):
    """fp32: 1e-5 relative plus the two approximate sigmoids' absolute error in sig*(1-sig) (<= 2^-21) times
    |scale*gz*w|; 16-bit: 1 ulp of the storage type of the rounded fp64 value + 1e-5 max|value| (ulp_check's floor)."""
    g = got.cpu().double()
    if dtype == torch.float32:
        tol = RTOL * want64.abs() + 2.0 ** -21 * coef_abs
        ref = want64
    else:
        ref = want64.to(dtype).double()
        ulp = 2.0 ** (-7 if dtype == torch.bfloat16 else -10)
        tol = ulp * ref.abs() + RTOL * float(want64.abs().max())
    bad = (g - ref).abs() > tol
    assert not bool(bad.any()), "%s: %d of %d elements out of bounds" % (what, int(bad.sum()), bad.numel())


def _bwd_inputs(dname, B, D, h, w, foff, goff, seed):
    dtype = DTYPES[dname]
    g = torch.Generator().manual_seed(seed)
    feat = on_device(B * D * h * w, dtype, foff, g).view(B, D, h, w)
    proto = (torch.randn(D, generator=g) * 1.5).cuda()
    weight = (torch.randn(D, generator=g) * 0.2).cuda()
    gz = on_device(B * h * w, torch.float32, goff, g, scale=1.0).view(B, h, w)
    return dtype, feat, proto, weight, gz


@pytest.mark.parametrize("case", HEAD_BWD_CASES, ids=_bwd_id)
def test_seen_head_backward_against_fp64(ops, case):
    dname, B, D, h, w, foff, goff, want_df, scale = case
    dtype, feat, proto, weight, gz = _bwd_inputs(dname, B, D, h, w, foff, goff, seed=B * 100 + D)
    hw = h * w
    expect_vec = hw % 8 == 0 and not foff and not goff
    assert _vec_path(feat, gz, True, hw) == expect_vec   # (a fresh feature-gradient tensor is always aligned)
    sdev = None if scale is None else torch.tensor([scale], device="cuda")
    s = 1.0 if scale is None else scale
    dw, db, df = ops.seen_head_backward(feat, proto, weight, gz, sdev, want_df)
    assert (df is not None) == want_df
    dw64, db64, df64, dw_abs, db_abs = head_backward64(feat, proto, weight, gz, s)
    if s == 0.0:
        assert not bool(dw.any()) and not bool(db.any()) and (df is None or not bool(df.float().any()))
        return
    assert bool(((dw.cpu().double() - dw64).abs() <= RTOL * dw_abs).all()), "dweight"
    assert bool(((db.cpu().double() - db64).abs() <= RTOL * db_abs).all()), "dbias"
    if want_df:
        coef = (abs(s) * gz.cpu().double().abs().unsqueeze(1) * weight.cpu().double().abs().view(1, D, 1, 1))
        _check_dfeat(df, df64, coef, dtype, "dfeat")


@pytest.mark.parametrize("dname,h,w,foff", [("f32", 8, 8, 0), ("bf16", 16, 16, 0), ("f16", 8, 8, 0),
                                            ("f32", 5, 7, 0), ("bf16", 8, 8, 1), ("f16", 3, 5, 0)],
                         ids=["f32-vec", "bf16-vec", "f16-vec", "f32-scalar", "bf16-scalar", "f16-scalar"])
def test_seen_head_tie_gives_zero_feature_gradient(ops, dname, h, w, foff):
    """Where a feature equals its channel's prototype, |sig(x) - sig(p)| has the subgradient torch's abs gives, 0:
    the kernel must compute exactly 0 for d there (both sigmoids through the same instructions), not +-1 ulp that
    would turn into +-w*sig'*gz.  ReLU features are exactly 0 often, so ties are common.  dW is unaffected: the
    tied terms contribute 0 to it either way.  seen_logits gets the same 0 terms: z equals the fp64 value of the
    untied channels within the usual bound."""
    B, D = 2, 24
    dtype, feat, proto, weight, gz = _bwd_inputs(dname, B, D, h, w, foff, 0, seed=77)
    proto = proto.to(dtype).float()                         # prototypes representable in the feature type
    tie = torch.rand(B, D, h, w, generator=torch.Generator().manual_seed(5)) < 0.3
    tie[0, :, 0, 0] = True                                  # a pixel where every channel ties
    x = feat.cpu().float()
    x = torch.where(tie, proto.cpu().view(1, D, 1, 1).expand(B, D, h, w), x)
    feat.copy_(x.to(dtype).cuda().view_as(feat))
    assert bool((feat.cpu().float()[tie] == proto.cpu().view(1, D, 1, 1).expand(B, D, h, w)[tie]).all())
    dw, db, df = ops.seen_head_backward(feat, proto, weight, gz, torch.tensor([0.37], device="cuda"), True)
    assert _vec_path(feat, gz, True, h * w) == (h * w % 8 == 0 and not foff)
    dfc = df.cpu()
    assert int((dfc[tie] != 0).sum()) == 0, "%d tied features got a nonzero gradient" % int((dfc[tie] != 0).sum())
    dw64, _, df64, dw_abs, _ = head_backward64(feat, proto, weight, gz, 0.37)
    assert bool(((dw.cpu().double() - dw64).abs() <= RTOL * dw_abs).all())
    coef = 0.37 * gz.cpu().double().abs().unsqueeze(1) * weight.cpu().double().abs().view(1, D, 1, 1)
    _check_dfeat(df, df64, coef, dtype, "dfeat")
    # the all-tied pixel: z is exactly the bias in every head (every term is exactly 0)
    z = ops.seen_logits(feat, proto.view(1, D), weight.view(1, D), torch.tensor([0.25], device="cuda"))
    assert float(z[0, 0, 0, 0]) == 0.25
    z64, abs64 = seen_logits64(feat, proto.view(1, D), weight.view(1, D), torch.tensor([0.25]))
    assert bool(((z.cpu().double() - z64).abs() <= RTOL * abs64).all())


# --------------------------------------------------------------------------------------
# the pixel kernels' use of the heads: seen weight, distill mask, focal term and its gradient
# --------------------------------------------------------------------------------------
# name -> (variant, logits dtype, K, B, h, w, lowres): the kernel bacs_pixel_kernel_variant reports for this shape
PIXEL_SHAPES = {
    # 25 <= K <= 63: generic shared-memory tile.  W = 48: a warp's pixels wrap into the next image row and meet the
    # same low-res cells again; the focal gradient's segmented warp reduction used to add such a later run into the
    # earlier one as well, counting it twice (fixed: run_end_lane)
    "tile":      (0, torch.float32, 30, 2, 3, 3, False),
    "fast":      (1, torch.float32, 8, 1, 2, 16, False),     # K <= 24, W = 256 (not 512-pixel rows): register fast path
    "fast_wrap": (1, torch.float32, 8, 2, 2, 3, False),      # the register fast path at W = 48: the same wrap as "tile"
    "rowtile":   (2, torch.bfloat16, 8, 1, 2, 32, False),    # K <= 24, W = 512: row-tile training-step kernel
    "lowres":    (3, torch.float32, 8, 1, 2, 3, True),       # fused x16 up-sample of sem_logits
    "stream":    (4, torch.float32, 64, 1, 2, 2, False),     # fp32, K >= 64: two streaming passes
    "regs":      (5, torch.bfloat16, 80, 1, 2, 2, False),    # 16-bit, 64 <= K <= 152: register column
}
PIXEL_CASES = []
for _name in PIXEL_SHAPES:
    for _T in (1, 2, 8, 16, 32):
        for _head in sorted({0, _T // 2, _T - 1}):
            PIXEL_CASES.append((_name, _T, _head))
# many heads on the 512-pixel row-tile shape: T=64 keeps the row-tile kernel (T*2*w floats of head rows per stage);
# at T=256 the staged rows and the per-warp [T][8] strips exceed shared memory and the plan takes the generic tile
for _T in (64, 256):
    for _head in (0, _T // 2, _T - 1):
        PIXEL_CASES.append(("rowtile", _T, _head))


def _pixel_variant(name, T):
    return 0 if (name == "rowtile" and T == 256) else PIXEL_SHAPES[name][0]


def focal64(Z, t):
    """binary focal loss (gamma 2, no alpha) per pixel: (term, d term / dZ), float64"""
    Z = Z.detach().clone().requires_grad_(True)
    bce = F.softplus(Z) - t * Z
    pt = torch.exp(-bce)
    term = (1.0 - pt) ** 2 * bce
    (dterm,) = torch.autograd.grad(term.sum(), Z)
    return term.detach(), dterm


def _scatter_up(v, B, T, h, w, s):
    """adjoint of up_ac64 applied to a per-pixel [B,H,W] map: sum over the pixels of weight * v, per low-res cell"""
    zz = torch.zeros(B, 1, h, w, dtype=torch.float64, requires_grad=True)
    (g,) = torch.autograd.grad((up_ac64(zz, s)[:, 0] * v).sum(), zz)
    return g[:, 0]


@pytest.mark.parametrize("name,T,head", PIXEL_CASES, ids=["%s-T%d-h%d" % c for c in PIXEL_CASES])
def test_pixel_kernels_read_the_heads(ops, cabi, name, T, head):
    _, dtype, K, B, h, w, lowres = PIXEL_SHAPES[name]
    s = 16
    H, W = h * s, w * s
    old_cl = K // 2
    g = torch.Generator().manual_seed(T * 31 + head + K)
    z = torch.randn(B, T, h, w, generator=g) * 2.0
    lab = torch.randint(1, K, (B, H, W), generator=g)
    u = torch.rand(B, H, W, generator=g)
    lab[u < 0.35] = 0
    lab[u > 0.95] = 255
    if lowres:
        logits = (torch.randn(B, K, h, w, generator=g) * 2).to(dtype)
        x = up_hp64(logits.double(), H, W)
    else:
        logits = (torch.randn(B, K, H, W, generator=g) * 2).to(dtype)
        x = logits.double()
    out = ops.pixel_loss(logits.cuda(), lab.cuda(), cabi.PIX_WEIGHTED_CE, want_grad=True, z=z.cuda(),
                         want_distill_mask=True, old_cl=old_cl, ukd=True, focal_head=head, lowres=lowres)
    assert out["variant"] == _pixel_variant(name, T)
    acc = out["acc"].cpu()

    z64 = z.double()
    up = up_ac64(z64, s)                                       # [B,T,H,W]
    zabs = up_ac64(z64.abs(), s).max(1)[0]                     # largest absolute-term sum of an interpolated head
    zmax = up.max(1)[0]
    valid = lab != 255
    bg = lab == 0
    # distill mask: label 0 and max_t sigma(up(z_t)) > 0.5, i.e. max_t up(z_t) > 0.  Band: the kernel's fp32
    # interpolation (3 roundings of zabs) and its approximate sigmoid (~2 ulp at 0.5, i.e. 5e-7 in z) can put a
    # pixel with |zmax| below 2^-21 (1 + zabs) on either side; every other pixel must match exactly.
    band = zmax.abs() <= 2.0 ** -21 * (1 + zabs)
    want_m = bg & (zmax > 0)
    got_m = out["distill_mask"].cpu().bool()
    assert int(((got_m != want_m) & ~band).sum()) == 0
    assert int(acc[cabi.ACC_DISTILL_PIX]) == int(got_m.sum())

    # weighted CE with the seen weight (1 - s)^2, s = sigmoid(zmax) set to 1 above 0.5 (ukd on)
    lse = torch.logsumexp(x, 1)
    sig = torch.sigmoid(zmax)
    sgt = torch.where(sig > 0.5, torch.ones_like(sig), sig)
    mod = (1 - sgt) ** 2
    lse_fg = torch.logsumexp(x[:, 1:], 1)
    lse_old = torch.logsumexp(x[:, :old_cl], 1)
    y = lab.clamp(max=K - 1)
    xy = x.gather(1, y.unsqueeze(1)).squeeze(1)
    l1 = torch.where(bg, mod * (lse - x[:, 0]), torch.where(valid, lse - lse_fg, torch.zeros_like(lse)))
    l2 = torch.where(lab < old_cl, lse - lse_old, torch.where(valid, lse - xy, torch.zeros_like(lse)))
    # per pixel: 1e-5 relative, + the fast log's absolute error (2^-21 per __logf, four of them), + the seen weight's
    # error (sigmoid ~2^-22, zmax 2^-22 zabs, through d mod / d s <= 2), + in the band either seen weight
    e = RTOL * (l1.abs() + l2.abs()) + 2.0 ** -19 + 2 * (2.0 ** -22 * (1 + zabs)) * (lse - x[:, 0]).abs() * bg
    e = e + torch.where(band & bg, (0.25 - mod).abs() * (lse - x[:, 0]).abs(), torch.zeros_like(e))
    loss64 = float((l1 + l2).sum())
    assert abs(float(acc[cabi.ACC_LOSS]) - loss64) <= float(e.sum()), (float(acc[cabi.ACC_LOSS]), loss64)

    # focal term of head `head`: target = foreground, ignore dropped; gz = d(sum of terms) / d z[:, head]
    term, dterm = focal64(up[:, head], (~bg).double())
    term, dterm = term * valid, dterm * valid
    # per pixel: 1e-5 relative, + the intrinsics' absolute error and the fp32 interpolation of z (2^-20 (1 + zabs))
    floor = 2.0 ** -20 * (1 + zabs) * valid
    focal_bound = float((RTOL * term.abs() + floor).sum())
    assert abs(float(acc[cabi.ACC_FOCAL]) - float(term.sum())) <= focal_bound
    gz64 = _scatter_up(dterm, B, T, h, w, s)
    gz_bound = _scatter_up(RTOL * dterm.abs() + floor, B, T, h, w, s)
    err = (out["gz"].cpu().double() - gz64).abs()
    bad = err > gz_bound
    assert not bool(bad.any()), "gz: %d of %d cells out of bounds (worst ratio %.3g)" % (
        int(bad.sum()), bad.numel(), float((err / gz_bound).max()))
    assert int(acc[cabi.ACC_KEPT]) == int(valid.sum()) and int(acc[cabi.ACC_BG]) == int(bg.sum())


def test_pixel_loss_refuses_focal_head_out_of_range(ops, cabi):
    g = torch.Generator().manual_seed(1)
    T, h, w = 3, 2, 3
    z = torch.randn(1, T, h, w, generator=g).cuda()
    logits = torch.randn(1, 30, 32, 48, generator=g).cuda()
    lab = torch.randint(0, 30, (1, 32, 48), generator=g).cuda()
    with pytest.raises(cabi.BacsError):
        ops.pixel_loss(logits, lab, cabi.PIX_WEIGHTED_CE, want_grad=True, z=z, old_cl=15, focal_head=T)
    out = ops.pixel_loss(logits, lab, cabi.PIX_WEIGHTED_CE, want_grad=True, z=z, old_cl=15, focal_head=T - 1)
    assert out["gz"] is not None
