"""The integer kernels -- bacs_label_hist, bacs_label_remap (presence, then apply), bacs_label_downsample_task,
bacs_confmat_accumulate (vector, shared-memory, opt-in and global paths, int64 and fp32 predictions),
bacs_confmat_metrics and bacs_der_cut -- at every path the host code selects, against exact references on the host:

  label_hist             numpy.bincount with one bin for labels outside [0, 256)
  label_remap            oracle.sequential_remap / transform_label, image by image
  label_downsample_task  oracle.downsample_labels + the lut, then the raster rank and n_bt in numpy
  confmat_accumulate     oracle.confusion_matrix (int32 casts included) and a numpy count of oob
  confmat_metrics        oracle.iou_metrics
  der_cut                oracle.der_transplant_cut

Integer outputs must match bit for bit.  Metrics rows 0-4 are one fp32 division of fp32-rounded int64 sums on both
sides, so they must be bit-identical too; the broadcast mIoU (row 5) may differ by the summation order, at most
K * 2^-23 relative.

Every op is called through the C ABI with outputs owned here: each is pre-filled with a sentinel (or, for the
accumulating ops, with non-zero start values) and has a guard band before and after it.  Every entry must be
written as the reference says and every guard must stay untouched.  Every remap case runs with its input and output
16-byte aligned and 8 bytes off (and with only the output off), so the vector and scalar paths are compared on the
same data; integral confusion-matrix data goes through the int64 and the fp32 prediction paths alike.

NaN predictions are left out: the reference's own .int() turns NaN into different values on the CPU and on CUDA.

The host copies of the dispatch (hist_plan, remap_plan, ds_plan, cm_plan) follow labels.cu and misc.cu; the coverage
test prints what the case tables reach and the profiler test checks the confusion-matrix and down-sample plans by
the names of the kernels launched.  The refusal rows return before any launch and also run without a device."""
import json
import os
import re
import subprocess
import sys
from dataclasses import dataclass
from typing import Tuple

import numpy as np
import pytest
import torch

from oracle import bacs_oracle as O

gpu = pytest.mark.gpu
CPU_SMS = 148
GUARD = 64                            # elements of guard band before and after every output
GUARD_I = -(1 << 50) - 5
MAX_DOM, PRES_STRIDE = 1024, 1032     # labels.cu kMaxDom, kPresStride


def _on_gpu():
    return torch.cuda.is_available()


def sm_count():
    return torch.cuda.get_device_properties(0).multi_processor_count if _on_gpu() else CPU_SMS


def _dev():
    return "cuda" if _on_gpu() else "cpu"


def _lib():
    from bacs_b200 import _cabi
    return _cabi.load()


def _check(status, what):
    from bacs_b200 import _cabi
    _cabi.check(status, what)


def _stream():
    if not _on_gpu():
        return None
    from bacs_b200 import ops
    return ops._stream()


def _guarded(n, dtype, fill, guard, off=0):
    """[GUARD + off | n entries | GUARD] on the device; the entries hold `fill`, the rest `guard`.  `off` = 1 puts
    the entries 8 bytes (int64) off the 16-byte alignment of the allocation."""
    buf = torch.full((GUARD + off + n + GUARD,), guard, dtype=dtype, device=_dev())
    buf[GUARD + off:GUARD + off + n] = fill
    return buf


def _body(buf, n, off=0):
    return buf[GUARD + off:GUARD + off + n]


def _guards_intact(buf, n, guard, off=0):
    return bool((buf[:GUARD + off] == guard).all()) and bool((buf[GUARD + off + n:] == guard).all())


def _at_offset(x, off):
    """a device copy of x whose data pointer is `off` elements past a 16-byte boundary; two spare elements follow,
    so that even an empty x has a non-null pointer"""
    flat = x.reshape(-1)
    buf = torch.zeros(flat.numel() + off + 2, dtype=x.dtype, device=_dev())
    buf[off:off + flat.numel()] = flat.to(_dev())
    return buf[off:]


# --------------------------------------------------------------------------------------
# bacs_label_hist
# --------------------------------------------------------------------------------------
def hist_plan(n, sms):
    nchunk = (n + 7) >> 3
    blocks = (nchunk + 255) // 256
    return {"blocks": min(blocks, 8 * sms), "capped": blocks > 8 * sms, "tail": n % 8 != 0}


@dataclass(frozen=True)
class Hist:
    name: str
    n: int
    data: str          # "rand", "runs" (runs crossing 8-label chunks) or "edges" (runs + out-of-range labels)
    accumulate: bool = False

    def reached(self, sms):
        p, r = hist_plan(self.n, sms), set()
        r.add("tail chunk" if p["tail"] else "only full chunks")
        if self.n < 8:
            r.add("n < 8")
        if p["capped"]:
            r.add("grid capped at 8 SMs")
        if self.accumulate:
            r.add("accumulate into a non-zero hist")
        lab = hist_inputs(self)
        r |= {k for k, v in (("label < 0", (lab < 0).any()), ("label 256", (lab == 256).any()),
                             ("label >= 2^40", (lab >= 1 << 40).any())) if v}
        if self.n > 8 and (lab[7:-1:8] == lab[8::8]).any():
            r.add("runs across chunks")
        return r


def hist_cases(sms):
    cap_n = 8 * 2048 * sms + 8 * 37 + 3
    return [Hist("n1", 1, "rand"), Hist("n7", 7, "edges"), Hist("full-8000", 8000, "rand"),
            Hist("runs-32768", 32768, "runs", True), Hist("edges-2405", 2405, "edges"),
            Hist("capped-%d" % cap_n, cap_n, "edges", True), Hist("capped-even", 8 * 2048 * sms + 8 * 512, "runs")]


HIST_WANT = {"only full chunks", "tail chunk", "n < 8", "grid capped at 8 SMs", "accumulate into a non-zero hist",
             "label < 0", "label 256", "label >= 2^40", "runs across chunks"}


def hist_inputs(c):
    rng = np.random.RandomState(c.n % 100003)
    if c.data == "rand":
        return rng.randint(0, 256, c.n).astype(np.int64)
    vals = rng.randint(0, 256, c.n // 5 + 2).astype(np.int64)
    lab = np.repeat(vals, rng.randint(1, 10, vals.size))[:c.n]
    lab = np.concatenate([lab, rng.randint(0, 256, c.n - lab.size)]).astype(np.int64)
    if c.data == "edges":
        special = np.array([-1, -(1 << 40), 256, 1 << 40, (1 << 40) + 3, 255, 0, 257, -256], dtype=np.int64)
        idx = rng.randint(0, c.n, max(1, c.n // 50))
        lab[idx] = special[rng.randint(0, special.size, idx.size)]
        lab[0] = special[0]
    return lab


def hist_reference(lab):
    inside = (lab >= 0) & (lab < 256)
    return np.bincount(np.where(inside, lab, 256), minlength=257).astype(np.int64)


# --------------------------------------------------------------------------------------
# bacs_label_remap
# --------------------------------------------------------------------------------------
def remap_plan(n_images, ppi, in_off, out_off, sms):
    """grid and path of both remap kernels; in_off / out_off: the pointers are that many int64 past 16 bytes"""
    bx = min((ppi + 2047) // 2048, max(1, 8 * sms // n_images))
    bx = max(bx, 1)
    even = ppi % 2 == 0
    if not even:
        pres = "scalar, odd ppi"
    elif in_off % 2:
        pres = "scalar, 8-byte offset input"
    else:
        pres = "vector, exact tiling" if (ppi // 2) % (4 * bx * 256) == 0 else "vector, padding lanes"
    if even and in_off % 2 == 0 and out_off % 2 == 0:
        app = "vector"
    elif even and in_off % 2 == 0:
        app = "scalar, in aligned, out unaligned"
    else:
        app = "scalar"
    return {"bx": bx, "presence": pres, "apply": app}


@dataclass(frozen=True)
class Rm:
    name: str
    n_images: int
    ppi: int
    lo: int
    n_dom: int
    data: str           # "rand", "chain" (v -> v+1 over the whole domain), "shuffled" (a random-order chain),
                        # "every" (every domain value in every image), "pad-lo" (the padding-lane trap)
    masking1: str = "lo"        # "lo" or "top"
    two_pass: bool = False
    inplace: bool = False
    two_d: bool = False         # also through ops.label_remap with a 2-D [H, W] input

    def runs(self):
        """(in_off, out_off) of every call; out_off None = in place"""
        if self.inplace:
            return [(0, None), (1, None)]
        return [(0, 0), (1, 1), (0, 1)]

    def reached(self, sms):
        r = set()
        for in_off, out_off in self.runs():
            p = remap_plan(self.n_images, self.ppi, in_off, in_off if out_off is None else out_off, sms)
            r |= {"presence: " + p["presence"], "apply: " + p["apply"]}
            if p["bx"] == 1 and self.n_images > 8 * sms:
                r.add("n_images > 8 SMs (bx 1)")
        r.add("two passes" if self.two_pass else "one pass")
        if self.inplace:
            r.add("in place")
        r.add("2-D input" if self.two_d else ("several images" if self.n_images > 1 else "one image"))
        r.add("n_dom %d" % self.n_dom)
        r.add("lo < 0" if self.lo < 0 else "lo > 0" if self.lo > 0 else "lo 0")
        lab, m1, k1, _, _ = remap_inputs(self)
        if (lab < self.lo).any():
            r.add("below the domain")
        if (lab >= self.lo + self.n_dom).any():
            r.add("above the domain")
        r.add("masking1 == lo" if k1 == self.lo else "masking1 at the top" if k1 == self.lo + self.n_dom - 1 else "")
        if self.data in ("chain", "shuffled") and self.n_dom >= 257:
            r.add("chain as long as the domain (%s)" % self.data)
        if all(len(np.unique(lab[b][(lab[b] >= self.lo) & (lab[b] < self.lo + self.n_dom)])) == self.n_dom
               for b in range(self.n_images)):
            r.add("every domain value present")
        return r - {""}


def remap_cases(sms):
    many = 8 * sms + 5
    return [
        Rm("pad-lo-1000", 3, 1000, 0, 8, "pad-lo"),
        Rm("rand-1000-top", 3, 1000, -1, 257, "rand", "top", True),
        Rm("exact-512sq", 2, 512 * 512, -1, 257, "rand", "lo", True),
        Rm("odd-37x53", 3, 37 * 53, -1, 257, "rand", "top"),
        Rm("big-1024x2048x2", 2, 1024 * 2048, -1, 257, "rand", "lo", True),
        Rm("many-images", many, 64, 3, 40, "rand", "lo", True),
        Rm("inplace-2pass", 4, 3000, -1, 257, "rand", "top", True, True),
        Rm("inplace-odd", 2, 999, 10, 100, "rand", "lo", False, True),
        Rm("two-d", 1, 20 * 50, -1, 257, "rand", "lo", True, False, True),
        Rm("dom1-lo5", 3, 1000, 5, 1, "rand"),
        Rm("dom1-neg", 2, 777, -9, 1, "rand", "lo", True),
        Rm("chain-1024", 2, 2048, -300, 1024, "chain", "top"),
        Rm("chain-1024-2pass", 2, 4100, 7, 1024, "chain", "lo", True),
        Rm("shuffled-1024", 2, 3001, -512, 1024, "shuffled", "lo", True),
        Rm("shuffled-257", 3, 1200, -1, 257, "shuffled", "top"),
        Rm("every-257", 2, 1024, -1, 257, "every", "lo", True),
        Rm("every-1024-inplace", 2, 1030, 20, 1024, "every", "top", False, True),
    ]


REMAP_WANT = {"presence: vector, padding lanes", "presence: vector, exact tiling", "presence: scalar, odd ppi",
              "presence: scalar, 8-byte offset input", "apply: vector", "apply: scalar",
              "apply: scalar, in aligned, out unaligned", "one pass", "two passes", "in place", "2-D input",
              "several images", "n_images > 8 SMs (bx 1)", "n_dom 1", "n_dom 257", "n_dom 1024", "lo < 0", "lo > 0",
              "below the domain", "above the domain", "masking1 == lo", "masking1 at the top",
              "chain as long as the domain (chain)", "chain as long as the domain (shuffled)",
              "every domain value present"}


def remap_inputs(c):
    """(labels int64 [n_images, ppi], map1 int32 [n_dom], masking1, map2 or None, masking2)"""
    rng = np.random.RandomState(sum(map(ord, c.name)))
    lo, nd, hi = c.lo, c.n_dom, c.lo + c.n_dom
    k1 = lo if c.masking1 == "lo" else hi - 1
    if c.data == "pad-lo":        # lo = 0 maps to 7; one pixel below the domain goes to masking1 = lo = 0
        lab = np.full((c.n_images, c.ppi), lo + 3, dtype=np.int64)
        lab[0, 0] = lo - 4
        m1 = np.arange(lo, hi, dtype=np.int32)
        m1[0] = hi - 1
        return lab, m1, lo, None, 0
    if c.data == "chain":
        m1 = np.arange(lo + 1, hi + 1, dtype=np.int32)
        m1[-1] = lo
    elif c.data == "shuffled":
        order = rng.permutation(nd) + lo
        m1 = np.empty(nd, dtype=np.int32)
        m1[order - lo] = np.roll(order, -1)
    else:
        m1 = rng.randint(lo, hi, nd).astype(np.int32)
        m1[rng.rand(nd) < 0.3] = k1                      # unmapped entries hold the masking value
    if c.data in ("chain", "shuffled", "every"):
        lab = np.stack([np.concatenate([rng.permutation(nd) + lo, rng.randint(lo, hi, c.ppi - nd)])
                        for _ in range(c.n_images)]).astype(np.int64)
    else:
        # a few present values per image, in runs, like a segmentation map
        lab = np.empty((c.n_images, c.ppi), dtype=np.int64)
        for b in range(c.n_images):
            vals = rng.choice(nd, size=min(nd, 12), replace=False) + lo
            lab[b] = np.repeat(vals, c.ppi // vals.size + 1)[:c.ppi]
            rng.shuffle(lab[b].reshape(-1)[: (c.ppi // 16) * 16].reshape(-1, 16))
    if c.data != "every":
        out = np.array([lo - 1, lo - 2, lo - (1 << 40), hi, hi + 5, 1 << 40], dtype=np.int64)
        mask = rng.rand(*lab.shape) < 0.02
        lab[mask] = out[rng.randint(0, out.size, int(mask.sum()))]
        lab[:, -1] = out[rng.randint(0, out.size, c.n_images)]
    m2, k2 = None, 0
    if c.two_pass:
        k2 = int(rng.randint(lo, hi))
        m2 = rng.randint(lo, hi, nd).astype(np.int32)
        m2[rng.rand(nd) < 0.3] = k2
    return lab, m1, k1, m2, k2


def remap_reference(lab, lo, m1, k1, m2, k2):
    d1 = {lo + i: int(v) for i, v in enumerate(m1)}
    d2 = None if m2 is None else {lo + i: int(v) for i, v in enumerate(m2)}
    return np.stack([O.transform_label(img, d1, k1, d2, k2) for img in lab])


def run_remap(lab, lo, m1, k1, m2, k2, in_off, out_off):
    """C ABI call; out_off None = in place.  Returns (output, guard band intact)."""
    n_img, ppi = lab.shape
    n = lab.size
    dev = _dev()
    m1d = torch.from_numpy(m1).to(dev)
    m2d = None if m2 is None else torch.from_numpy(m2).to(dev)
    lib = _lib()
    ws = torch.full((lib.bacs_label_remap_workspace_bytes(n_img) // 4,), 7, dtype=torch.int32, device=dev)
    if out_off is None:
        buf = _guarded(n, torch.int64, 0, GUARD_I, in_off)
        _body(buf, n, in_off).copy_(torch.from_numpy(lab.reshape(-1)))
        src = dst = _body(buf, n, in_off)
        off = in_off
    else:
        src = _at_offset(torch.from_numpy(lab), in_off)
        buf = _guarded(n, torch.int64, (1 << 50) + 3, GUARD_I, out_off)
        dst = _body(buf, n, out_off)
        off = out_off
    _check(lib.bacs_label_remap(src.data_ptr(), dst.data_ptr(), n_img, ppi, lo, m1.size, m1d.data_ptr(), k1,
                                None if m2d is None else m2d.data_ptr(), k2, ws.data_ptr(), _stream()),
           "bacs_label_remap")
    return dst.cpu().numpy().reshape(n_img, ppi), _guards_intact(buf, n, GUARD_I, off)


# --------------------------------------------------------------------------------------
# bacs_label_downsample_task
# --------------------------------------------------------------------------------------
def ds_plan(T):
    return {"kmax": 32 if T <= 32 else 128}


@dataclass(frozen=True)
class Ds:
    name: str
    B: int
    H: int
    W: int
    h: int
    w: int
    T: int
    down: bool          # labels_down given
    data: str           # "rand", "blocky" (large regions) or "lanes" (label = column mod 32)

    def reached(self):
        r = {"KMAX %d" % ds_plan(self.T)["kmax"], "T %d" % self.T, "labels_down given" if self.down else
             "labels_down NULL"}
        hw = self.h * self.w
        r.add("hw < 1024" if hw < 1024 else "hw 1024" if hw == 1024 else
              "hw multiple of 1024" if hw % 1024 == 0 else "chunks with a partial last one")
        if (self.H, self.h) in ((513, 33), (500, 32)):
            r.add("ratio %d->%d" % (self.H, self.h))
        if self.h == self.H:
            r.add("h = H")
        lab, lut = ds_inputs(self)
        down, task, _, _ = ds_reference(self, lab, lut)
        r |= {k for k, v in (("labels < 0", (down < 0).any()), ("labels >= 256", (down >= 256).any()),
                             ("label 255", (down == 255).any())) if v}
        inr = (down >= 0) & (down < 256)
        raw = lut[np.clip(down, 0, 255)]
        r |= {k for k, v in (("lut -1", (inr & (raw == -1)).any()), ("lut >= T", (inr & (raw >= self.T)).any())) if v}
        for b in range(self.B):
            flat = task[b].reshape(-1)
            for q0 in range(0, flat.size - 31, 32):   # whole warps (chunks of 1024 start at multiples of 32)
                lanes = flat[q0:q0 + 32]
                if lanes[0] >= 0 and (lanes == lanes[0]).all():
                    r.add("warp in one task")
                if np.unique(lanes[lanes >= 0]).size == 32:
                    r.add("warp in 32 tasks")
        return r


DS_CASES = [
    Ds("t1-24px", 2, 64, 96, 4, 6, 1, False, "rand"),
    Ds("t32-lanes-1024", 2, 32, 32, 32, 32, 32, True, "lanes"),
    Ds("t33-2048", 1, 256, 256, 32, 64, 33, False, "rand"),
    Ds("t128-513to33", 3, 513, 513, 33, 33, 128, True, "rand"),
    Ds("t128-500to32", 2, 500, 500, 32, 32, 128, False, "blocky"),
    Ds("t128-lanes-chunks", 2, 97, 1000, 97, 61, 128, True, "lanes"),
    Ds("t20-blocky", 2, 512, 1024, 32, 64, 20, True, "blocky"),
    Ds("t33-lanes-h=H", 1, 40, 96, 40, 96, 33, False, "lanes"),
]
DS_WANT = {"KMAX 32", "KMAX 128", "T 1", "T 32", "T 33", "T 128", "hw < 1024", "hw 1024", "hw multiple of 1024",
           "chunks with a partial last one", "labels_down NULL", "labels_down given", "labels < 0", "labels >= 256",
           "label 255", "lut -1", "lut >= T", "warp in one task", "warp in 32 tasks", "ratio 513->33",
           "ratio 500->32", "h = H"}


def ds_inputs(c):
    rng = np.random.RandomState(sum(map(ord, c.name)))
    if c.data == "lanes":
        lab = np.broadcast_to(np.arange(c.W) % 32 + 64, (c.B, c.H, c.W)).astype(np.int64).copy()
    elif c.data == "blocky":
        blocks = rng.randint(0, 256, (c.B, c.H // 128 + 1, c.W // 512 + 1))
        lab = np.repeat(np.repeat(blocks, 128, 1), 512, 2)[:, :c.H, :c.W].astype(np.int64)
    else:
        lab = rng.randint(0, 256, (c.B, c.H, c.W)).astype(np.int64)
    special = np.array([-1, -7, 256, (1 << 33) + 3, 255, -(1 << 33)], dtype=np.int64)
    mask = rng.rand(*lab.shape) < 0.03
    lab[mask] = special[rng.randint(0, special.size, int(mask.sum()))]
    lab[:, 0, 0], lab[:, -1, -1] = -1, 255
    if c.data == "lanes":
        lut = (np.arange(256) % c.T).astype(np.int32)         # 32 columns -> 32 tasks when T >= 32
    else:
        lut = rng.randint(-1, c.T + 4, 256).astype(np.int32)  # entries -1 and >= T included
    lut[255], lut[0] = -1, c.T + 2
    return lab, lut


def ds_reference(c, lab, lut):
    down = O.downsample_labels(torch.from_numpy(lab), c.h, c.w).numpy()
    inr = (down >= 0) & (down < 256)
    task = np.where(inr, lut[np.clip(down, 0, 255)], -1)
    task[task >= c.T] = -1
    rank = np.zeros(task.shape, dtype=np.int32)
    n_bt = np.zeros((c.B, c.T), dtype=np.int32)
    for b in range(c.B):
        flat, rk = task[b].reshape(-1), rank[b].reshape(-1)
        for t in np.unique(flat[flat >= 0]):
            sel = np.flatnonzero(flat == t)
            rk[sel] = np.arange(sel.size)
            n_bt[b, t] = sel.size
    return down, task.astype(np.int8), rank, n_bt


# --------------------------------------------------------------------------------------
# bacs_confmat_accumulate
# --------------------------------------------------------------------------------------
def cm_plan(n, K, is_float, p_off, t_off):
    """the launches of bacs_confmat_accumulate: a list of (kernel, pred type, shared-memory flag)"""
    smem = 4 * K * K
    if n == 0:
        return []
    if not is_float and smem <= 48 * 1024 and n >= 2 and p_off % 2 == 0 and t_off % 2 == 0:
        return [("vec", "long", None)] + ([("scalar", "long", False)] if n % 2 else [])
    pt = "float" if is_float else "long"
    return [("scalar", pt, smem <= 96 * 1024)]


def cm_path(n, K, is_float, p_off, t_off):
    plan = cm_plan(n, K, is_float, p_off, t_off)
    if not plan:
        return "none"
    if plan[0][0] == "vec":
        return "vec + tail" if len(plan) == 2 else "vec"
    kind = "smem" if 4 * K * K <= 48 * 1024 else "smem opt-in" if plan[0][2] else "global"
    return ("float " if is_float else "int64 ") + kind


@dataclass(frozen=True)
class Cm:
    name: str
    n: int
    K: int
    data: str                 # "blocky" or "rand"
    is_float: bool = False
    p_off: int = 0
    t_off: int = 0
    oob: bool = True          # oob pointer given
    calls: int = 1
    special: Tuple[str, ...] = ()   # "wrap", "negt", "oobp", "frac", "big"

    def path(self):
        return cm_path(self.n, self.K, self.is_float, self.p_off, self.t_off)

    def reached(self):
        r = {"path " + self.path(), "oob given" if self.oob else "oob NULL"}
        if self.n in (0, 1):
            r.add("n %d" % self.n)
        if self.K in (110, 111, 156, 157, 4096):
            r.add("K %d" % self.K)
        if self.calls == 2:
            r.add("two calls")
        p, t = cm_inputs(self)
        t32 = t.astype(np.int32)
        kept = (t32 >= 0) & (t32 < self.K)
        if not self.is_float:
            p32 = p.astype(np.int32)
            r |= {k for k, v in (("wrap +2^32", ((p >= 1 << 32) & (p32 >= 0) & (p32 < self.K)).any()),
                                 ("wrap -2^32", ((t < -(1 << 31)) & kept).any())) if v}
        else:
            fin = np.isfinite(p)
            r |= {k for k, v in (("float fractional", (fin & (p != np.trunc(p)) & (p > 0)).any()),
                                 ("float -0.5", (p == -0.5).any()), ("float >= 2^31", (fin & (p >= 2.0 ** 31)).any()),
                                 ("float +inf", (p == np.inf).any()), ("float -inf", (p == -np.inf).any())) if v}
        _, oob = cm_reference(self, p, t)
        if (t32 < 0).any():
            r.add("negative targets")
        if oob:
            r.add("oob preds")
        if self.path().startswith("vec"):
            r.add("vec " + self.data)
        return r


CM_CASES = [
    Cm("vec-even-k21", 100000, 21, "blocky", calls=2, special=("wrap", "negt", "oobp")),
    Cm("vec-odd-k21", 100001, 21, "rand", special=("negt", "oobp")),
    Cm("vec-odd-k110", 4001, 110, "blocky", oob=False, special=("wrap", "oobp")),
    Cm("vec-n2", 2, 5, "rand"),
    Cm("n0", 0, 5, "rand"),
    Cm("n1", 1, 5, "rand"),
    Cm("smem-p-off-k110", 30001, 110, "blocky", p_off=1, special=("wrap", "negt", "oobp")),
    Cm("smem-t-off-k19", 20000, 19, "rand", t_off=1, oob=False, calls=2, special=("oobp",)),
    Cm("optin-k111", 40000, 111, "blocky", special=("wrap", "negt", "oobp")),
    Cm("optin-k156", 40001, 156, "rand", calls=2, special=("oobp",)),
    Cm("global-k157", 40000, 157, "blocky", special=("wrap", "negt", "oobp")),
    Cm("global-k4096", 200001, 4096, "rand", oob=False, special=("negt", "oobp")),
    Cm("float-smem-k21", 50001, 21, "blocky", True, special=("frac", "big", "negt")),
    Cm("float-smem-k110-off", 9000, 110, "rand", True, 1, 1, calls=2, special=("frac", "big")),
    Cm("float-optin-k111", 30000, 111, "rand", True, special=("frac", "big", "negt")),
    Cm("float-global-k157", 30000, 157, "blocky", True, oob=False, special=("frac", "big")),
    Cm("float-global-k300", 20001, 300, "rand", True, special=("frac", "big")),
    Cm("float-n1", 1, 3, "rand", True),
]
CM_WANT = {"path vec", "path vec + tail", "path int64 smem", "path int64 smem opt-in", "path int64 global",
           "path float smem", "path float smem opt-in", "path float global", "path none", "n 0", "n 1",
           "K 110", "K 111", "K 156", "K 157", "K 4096", "oob NULL", "oob given", "two calls",
           "wrap +2^32", "wrap -2^32", "negative targets", "oob preds", "vec blocky", "vec rand",
           "float fractional", "float -0.5", "float >= 2^31", "float +inf", "float -inf"}


def cm_inputs(c):
    """(preds int64 or float32 [n], target int64 [n])"""
    rng = np.random.RandomState(sum(map(ord, c.name)))
    n, K = c.n, c.K
    t = rng.randint(0, K, n).astype(np.int64)
    p = rng.randint(0, K, n).astype(np.int64)
    if c.data == "blocky":                      # long runs; preds mostly agree with the target
        t = t[np.arange(n) // 97 * 97]
        p = np.where(rng.rand(n) < 0.9, t, p)
    t[rng.rand(n) < 0.05] = 255 if K <= 255 else K
    if "negt" in c.special:
        t[rng.rand(n) < 0.02] = -1
        t[rng.rand(n) < 0.01] = -(1 << 32) + 2       # wraps to 2
    if "oobp" in c.special:
        bad = np.array([-1, K, K + 7, -(1 << 40), 1 << 31], dtype=np.int64)
        m = rng.rand(n) < 0.02
        p[m] = bad[rng.randint(0, bad.size, int(m.sum()))]
    if "wrap" in c.special:
        m = rng.rand(n) < 0.02
        p[m] = (1 << 32) + rng.randint(0, K, int(m.sum()))
        m = rng.rand(n) < 0.01
        t[m] = -(1 << 32) + rng.randint(0, K, int(m.sum()))
    if n:                                       # the last pixel (the separate launch of an odd n) counts
        t[-1], p[-1] = min(1, K - 1), min(2, K - 1)
    if not c.is_float:
        return p, t
    pf = p.astype(np.float32)
    if "frac" in c.special:
        m = rng.rand(n) < 0.1
        pf[m] += rng.rand(int(m.sum())).astype(np.float32) * 0.98
        pf[rng.rand(n) < 0.02] = -0.5
        pf[rng.rand(n) < 0.01] = -0.999
    if "big" in c.special:
        big = np.array([2.0 ** 31, 3e9, np.inf, -np.inf, -3e9, -2.0 ** 31, 1e30], dtype=np.float32)
        m = rng.rand(n) < 0.02
        pf[m] = big[rng.randint(0, big.size, int(m.sum()))]
    return pf, t


def cm_reference(c, p, t):
    """(confmat int64 [K, K], oob count); a float prediction is truncated toward zero, out-of-range ones are oob"""
    K = c.K
    if c.is_float:
        ok = np.isfinite(p) & (np.abs(p) < 2.0 ** 31)
        pi = np.where(ok, np.trunc(np.where(ok, p, 0)).astype(np.int64), -1)
    else:
        pi = p
    t32, p32 = t.astype(np.int32), pi.astype(np.int32)
    kept = (t32 >= 0) & (t32 < K)
    bad = kept & ((p32 < 0) | (p32 >= K))
    return O.confusion_matrix(p32[~bad], t[~bad], K).astype(np.int64), int(bad.sum())


def run_confmat(c, p, t, init, oob_init):
    """C ABI calls (c.calls of them) accumulating into a guarded confmat that starts at `init`"""
    KK = c.K * c.K
    pd = _at_offset(torch.from_numpy(p), c.p_off)
    td = _at_offset(torch.from_numpy(t), c.t_off)
    cm = _guarded(KK, torch.int64, 0, GUARD_I)
    _body(cm, KK).copy_(torch.from_numpy(init.reshape(-1)))
    ob = _guarded(1, torch.int64, oob_init, GUARD_I)
    lib = _lib()
    for _ in range(c.calls):
        _check(lib.bacs_confmat_accumulate(pd.data_ptr(), int(c.is_float), td.data_ptr(), c.n, c.K,
                                           _body(cm, KK).data_ptr(), _body(ob, 1).data_ptr() if c.oob else None,
                                           _stream()), "bacs_confmat_accumulate")
    assert _guards_intact(cm, KK, GUARD_I), "confmat guard band written"
    assert _guards_intact(ob, 1, GUARD_I), "oob guard band written"
    return _body(cm, KK).cpu().numpy().reshape(c.K, c.K), int(_body(ob, 1).cpu())


# --------------------------------------------------------------------------------------
# bacs_confmat_metrics
# --------------------------------------------------------------------------------------
MET_CASES = [(1, "rand"), (1, "absent"), (2, "rand"), (21, "absent"), (21, "diag"), (150, "big"), (256, "absent"),
             (256, "big"), (4096, "rand"), (4096, "absent")]


def met_reached():
    r = set()
    for K, data in MET_CASES:
        cm = met_inputs(K, data)
        r.add("K %d" % K)
        union = cm.sum(0) + cm.sum(1) - np.diag(cm)
        if (union == 0).any():
            r.add("absent class")
        if cm.sum() == 0 or (np.diag(cm) + cm.sum(1) - np.diag(cm) == 0).any():
            r.add("0/0")
        if (cm > 1 << 24).any():
            r.add("counts > 2^24")
        if (cm == np.diag(np.diag(cm))).all():
            r.add("diagonal only")
    return r


MET_WANT = {"K 1", "K 2", "K 21", "K 150", "K 256", "K 4096", "absent class", "0/0", "counts > 2^24", "diagonal only"}


def met_inputs(K, data):
    rng = np.random.RandomState(K * 7 + len(data))
    if data == "big":
        cm = rng.randint(0, 1 << 31, (K, K)).astype(np.int64) * rng.randint(0, 2, (K, K))
        cm[np.arange(K), np.arange(K)] += 1 << 33
    elif data == "diag":
        cm = np.diag(rng.randint(0, 1000, K)).astype(np.int64)
    else:
        cm = rng.randint(0, 50, (K, K)).astype(np.int64) * (rng.rand(K, K) < 0.3)
        cm[np.arange(K), np.arange(K)] += rng.randint(0, 500, K)
        if data == "absent":
            gone = rng.rand(K) < 0.3
            gone[0] = True
            cm[gone] = 0
            cm[:, gone] = 0
    return cm


def run_metrics(cm):
    K = cm.shape[0]
    cmd = torch.from_numpy(np.ascontiguousarray(cm)).to(_dev())
    out = _guarded(6 * K, torch.float32, float("nan"), -1234.5)
    _check(_lib().bacs_confmat_metrics(cmd.data_ptr(), K, _body(out, 6 * K).data_ptr(), _stream()),
           "bacs_confmat_metrics")
    assert _guards_intact(out, 6 * K, -1234.5), "metrics guard band written"
    return _body(out, 6 * K).cpu().numpy().reshape(6, K)


# --------------------------------------------------------------------------------------
# bacs_der_cut
# --------------------------------------------------------------------------------------
DC_CASES = [(1, 21, "rand"), (5, 21, "rand"), (5, 1, "equal"), (1024, 1024, "distinct"), (1024, 21, "equal"),
            (1025, 1023, "rand"), (4000, 1, "rand"), (4000, 21, "distinct"), (4000, 1023, "edges"),
            (1025, 1024, "edges")]


def dc_inputs(Br, K, data):
    rng = np.random.RandomState(Br * 3 + K)
    if data == "equal":
        return np.full(Br, min(K, 1023) if Br == 1024 else 0, dtype=np.int64)
    if data == "distinct":
        return np.resize(rng.permutation(1024), Br).astype(np.int64)
    n = rng.randint(0, 1024, Br).astype(np.int64)
    if data == "edges":
        n[rng.rand(Br) < 0.3] = 0
        n[rng.rand(Br) < 0.3] = 1023
    return n


def dc_reached():
    r = set()
    for Br, K, data in DC_CASES:
        n = dc_inputs(Br, K, data)
        r |= {"Br %d" % Br, "K %d" % K}
        r |= {k for k, v in (("all equal", np.unique(n).size == 1), ("1024 distinct", np.unique(n).size == 1024),
                             ("value >= K", (n >= K).any()), ("value 0", (n == 0).any()),
                             ("value 1023", (n == 1023).any())) if v}
    return r


DC_WANT = {"Br 1", "Br 5", "Br 1024", "Br 1025", "Br 4000", "K 1", "K 21", "K 1023", "K 1024", "all equal",
           "1024 distinct", "value >= K", "value 0", "value 1023"}


# --------------------------------------------------------------------------------------
# coverage of the plans
# --------------------------------------------------------------------------------------
def test_label_family_coverage():
    """the case tables reach every plan item of every op on this device's SM count"""
    sms = sm_count()
    if _on_gpu():
        assert _lib().bacs_device_sm_count() == sms
    tables = [("label_hist", HIST_WANT, lambda: set().union(*(c.reached(sms) for c in hist_cases(sms)))),
              ("label_remap", REMAP_WANT, lambda: set().union(*(c.reached(sms) for c in remap_cases(sms)))),
              ("label_downsample_task", DS_WANT, lambda: set().union(*(c.reached() for c in DS_CASES))),
              ("confmat_accumulate", CM_WANT, lambda: set().union(*(c.reached() for c in CM_CASES))),
              ("confmat_metrics", MET_WANT, met_reached),
              ("der_cut", DC_WANT, dc_reached)]
    print()
    for name, want, reach in tables:
        got = reach()
        print("%s: reached %d of %d plan items (%d SMs)" % (name, len(got & want), len(want), sms))
        assert got >= want, "%s not reached: %s" % (name, sorted(want - got))


def test_plan_boundaries():
    """the shared-memory boundaries of the confusion-matrix plan and the tiling of the remap presence sweep"""
    assert cm_path(10, 110, False, 0, 0) == "vec" and cm_path(10, 111, False, 0, 0) == "int64 smem opt-in"
    assert cm_path(10, 156, False, 0, 0) == "int64 smem opt-in" and cm_path(10, 157, False, 0, 0) == "int64 global"
    assert cm_path(1, 21, False, 0, 0) == "int64 smem" and cm_path(3, 21, False, 0, 0) == "vec + tail"
    assert cm_path(10, 21, True, 0, 0) == "float smem"
    assert remap_plan(2, 512 * 512, 0, 0, 148)["presence"] == "vector, exact tiling"
    assert remap_plan(1, 1024 * 2048, 0, 0, 148)["presence"] == "vector, exact tiling"
    assert remap_plan(2, 1024 * 2048, 0, 0, 148)["presence"] == "vector, padding lanes"
    assert remap_plan(3, 1000, 0, 0, 148)["presence"] == "vector, padding lanes"


# --------------------------------------------------------------------------------------
# label_hist
# --------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("c", hist_cases(sm_count()), ids=lambda c: c.name)
def test_label_hist_exact(c):
    lab = hist_inputs(c)
    want = hist_reference(lab)
    start = np.arange(257, dtype=np.int64) * 1000 + 17 if c.accumulate else np.zeros(257, dtype=np.int64)
    ld = torch.from_numpy(lab).cuda()
    h = _guarded(257, torch.int64, 0, GUARD_I)
    _body(h, 257).copy_(torch.from_numpy(start))
    _check(_lib().bacs_label_hist(ld.data_ptr(), c.n, _body(h, 257).data_ptr(), _stream()), "bacs_label_hist")
    assert _guards_intact(h, 257, GUARD_I), "hist guard band written"
    got = _body(h, 257).cpu().numpy()
    assert np.array_equal(got, start + want), np.flatnonzero(got != start + want)[:10]


# --------------------------------------------------------------------------------------
# label_remap
# --------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("c", remap_cases(sm_count()), ids=lambda c: c.name)
def test_label_remap_exact(c):
    lab, m1, k1, m2, k2 = remap_inputs(c)
    want = remap_reference(lab, c.lo, m1, k1, m2, k2)
    outs = {}
    for in_off, out_off in c.runs():
        got, intact = run_remap(lab, c.lo, m1, k1, m2, k2, in_off, out_off)
        p = remap_plan(c.n_images, c.ppi, in_off, in_off if out_off is None else out_off, sm_count())
        where = "in +%d, out %s (%s / %s)" % (in_off, "in place" if out_off is None else "+%d" % out_off,
                                              p["presence"], p["apply"])
        assert intact, "guard band written: " + where
        bad = np.argwhere(got != want)
        assert bad.size == 0, "%s: %d pixels differ, first %s: got %d want %d" % (
            where, len(bad), tuple(bad[0]), got[tuple(bad[0])], want[tuple(bad[0])])
        outs[where] = got
    if c.two_d:
        # through ops: a 2-D [H, W] input is one image; out= an 8-byte offset view
        from bacs_b200 import ops
        x = torch.from_numpy(lab.reshape(20, 50)).cuda()
        buf = _guarded(lab.size, torch.int64, (1 << 50) + 3, GUARD_I, 1)
        o = _body(buf, lab.size, 1).view(20, 50)
        ops.label_remap(x, torch.from_numpy(m1).cuda(), k1, None if m2 is None else torch.from_numpy(m2).cuda(), k2,
                        lo=c.lo, out=o)
        assert _guards_intact(buf, lab.size, GUARD_I, 1)
        assert np.array_equal(o.cpu().numpy().reshape(1, -1), want)


@gpu
def test_label_remap_padding_lanes_do_not_mark_lo():
    """lo = 0 maps to 7 and is absent from every image; a pixel below the domain goes to masking1 = 0 and stays 0.
    With 1000-pixel images the presence sweep pads its last loads: the padded lanes must not mark 0 as present."""
    from bacs_b200 import ops
    m1 = torch.tensor([7, 1, 2, 3, 4, 5, 6, 7], dtype=torch.int32)
    lab = torch.full((2, 20, 50), 3, dtype=torch.int64)
    lab[0, 0, 0] = -4
    want = np.stack([O.sequential_remap(img, {i: int(v) for i, v in enumerate(m1)}, 0) for img in lab.numpy()])
    assert want[0, 0, 0] == 0
    for shape in ((2, 20, 50), (2, 1, 1000), (2, 1, 999)):
        x = torch.full((2, int(np.prod(shape[1:]))), 3, dtype=torch.int64)
        x[0, 0] = -4
        got = ops.label_remap(x.view(shape).cuda(), m1.cuda(), 0, lo=0).cpu().view(2, -1)
        assert int(got[0, 0]) == 0, shape
        assert bool((got.view(-1)[1:] == 3).all()), shape


@gpu
def test_transform_label_padding_lanes():
    """TransformLabel: one 20x50 image of 2s; the first pass maps -1 -> 5 (-1 is absent), the second 2 -> 5 -> 9
    only if 5 was present after the first pass -- it was not, so every pixel is 5"""
    from bacs_b200 import labels as L
    d1 = {i: i for i in range(10)}
    d1[-1] = 5
    inv = {2: 5, 5: 9, 255: 255}
    lbl = np.full((20, 50), 2, dtype=np.int64)
    want = O.transform_label(lbl, d1, 255, inv, 0)
    assert (want == 5).all()
    tl = L.TransformLabel(d1, 255, inv, 0)
    assert np.array_equal(tl(torch.from_numpy(lbl).cuda()).cpu().numpy(), want)
    assert np.array_equal(tl(torch.from_numpy(np.stack([lbl, lbl])).cuda()).cpu().numpy(), np.stack([want, want]))


# --------------------------------------------------------------------------------------
# label_downsample_task
# --------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("c", DS_CASES, ids=lambda c: c.name)
def test_label_downsample_task_exact(c):
    lab, lut = ds_inputs(c)
    down, task, rank, n_bt = ds_reference(c, lab, lut)
    n, nb = c.B * c.h * c.w, c.B * c.T
    ld, lutd = torch.from_numpy(lab).cuda(), torch.from_numpy(lut).cuda()
    bd = _guarded(n, torch.int64, (1 << 61) + 1, GUARD_I) if c.down else None
    bt = _guarded(n, torch.int8, -128, 77)
    br = _guarded(n, torch.int32, -3, -77)
    bn = _guarded(nb, torch.int32, -3, -77)
    _check(_lib().bacs_label_downsample_task(ld.data_ptr(), c.B, c.H, c.W, c.h, c.w, lutd.data_ptr(), c.T,
                                             _body(bd, n).data_ptr() if c.down else None, _body(bt, n).data_ptr(),
                                             _body(br, n).data_ptr(), _body(bn, nb).data_ptr(), _stream()),
           "bacs_label_downsample_task")
    assert _guards_intact(bt, n, 77) and _guards_intact(br, n, -77) and _guards_intact(bn, nb, -77)
    if c.down:
        assert _guards_intact(bd, n, GUARD_I)
        assert np.array_equal(_body(bd, n).cpu().numpy(), down.reshape(-1)), "labels_down"
    assert np.array_equal(_body(bt, n).cpu().numpy(), task.reshape(-1)), "task"
    assert np.array_equal(_body(br, n).cpu().numpy(), rank.reshape(-1)), "rank"
    assert np.array_equal(_body(bn, nb).cpu().numpy(), n_bt.reshape(-1)), "n_bt"


# --------------------------------------------------------------------------------------
# confmat_accumulate and confmat_metrics
# --------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("c", CM_CASES, ids=lambda c: c.name)
def test_confmat_accumulate_exact(c):
    p, t = cm_inputs(c)
    want, oob = cm_reference(c, p, t)
    init = np.random.RandomState(c.K).randint(0, 1 << 40, (c.K, c.K)).astype(np.int64)
    got, got_oob = run_confmat(c, p, t, init, 5)
    assert np.array_equal(got - init, c.calls * want), "%d entries differ" % int((got - init != c.calls * want).sum())
    assert got_oob == 5 + (c.calls * oob if c.oob else 0)
    if not c.is_float:
        # the fp32-prediction path on the same integral data (predictions that fp32 cannot hold are made K + 3)
        p2 = np.where(np.abs(p) < 1 << 24, p, c.K + 3)
        cf = Cm(c.name, c.n, c.K, c.data, True, c.p_off, c.t_off, c.oob, c.calls)
        got_i, oob_i = run_confmat(c, p2, t, init, 5) if (p2 != p).any() else (got, got_oob)
        got_f, oob_f = run_confmat(cf, p2.astype(np.float32), t, init, 5)
        assert np.array_equal(got_f, got_i) and oob_f == oob_i, "fp32 preds (%s) disagree with int64" % cf.path()


@gpu
@pytest.mark.parametrize("K,data", MET_CASES, ids=["k%d-%s" % kd for kd in MET_CASES])
def test_confmat_metrics_exact(K, data):
    cm = met_inputs(K, data)
    got = run_metrics(cm)
    ref = O.iou_metrics(cm)
    for row, key in enumerate(["iou_per_class", "accuracy", "precision", "recall", "specificity"]):
        w = np.asarray(ref[key], dtype=np.float32)
        assert np.array_equal(got[row].view(np.int32), w.view(np.int32)), (key, np.flatnonzero(got[row] != w)[:8])
    miou = np.float32(ref["miou"])
    assert (got[5] == got[5][0]).all()
    assert abs(float(got[5][0]) - float(miou)) <= K * 2.0 ** -23 * abs(float(miou)), (got[5][0], miou)


# --------------------------------------------------------------------------------------
# der_cut
# --------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("Br,K,data", DC_CASES, ids=["br%d-k%d-%s" % c for c in DC_CASES])
def test_der_cut_exact(Br, K, data):
    n = dc_inputs(Br, K, data)
    want = O.der_transplant_cut(n, K)
    nd = torch.from_numpy(n).cuda()
    cut = _guarded(Br, torch.int32, -9, -77)
    _check(_lib().bacs_der_cut(nd.data_ptr(), Br, K, _body(cut, Br).data_ptr(), _stream()), "bacs_der_cut")
    assert _guards_intact(cut, Br, -77), "cut guard band written"
    got = _body(cut, Br).cpu().numpy()
    assert np.array_equal(got, want), np.flatnonzero(got != want)[:8]


# --------------------------------------------------------------------------------------
# kernel names
# --------------------------------------------------------------------------------------
def _cm_kernel_key(name):
    if "confmat_vec_kernel" in name:
        return ("vec", "long", None)
    m = re.search(r"confmat_kernel<\s*(long|float)\s*,\s*(true|false)\s*>", name)
    assert m, name
    return ("scalar", m.group(1), m.group(2) == "true")


def _cm_name_cases():
    first = {}
    for c in CM_CASES:
        if c.n:
            first.setdefault(c.path(), c)
    return first


DS_NAME_T = (1, 32, 33, 128)


def launched_kernel_names():
    """{case: names of the kernels it launched}: one profiled call per confusion-matrix path and per down-sample
    task count, each after an unprofiled warm-up call"""
    from torch.profiler import ProfilerActivity, profile
    from bacs_b200 import ops
    got = {}
    for path, c in sorted(_cm_name_cases().items()):
        p, t = cm_inputs(c)
        init = np.zeros((c.K, c.K), dtype=np.int64)
        run_confmat(c, p, t, init, 0)
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            run_confmat(c, p, t, init, 0)
        got[path] = [e.key for e in prof.key_averages() if "confmat" in e.key]
    lab = torch.zeros(2, 64, 64, dtype=torch.int64, device="cuda")
    lut = torch.zeros(256, dtype=torch.int32, device="cuda")
    for T in DS_NAME_T:
        ops.label_downsample_task(lab, 32, 32, lut, T)
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            ops.label_downsample_task(lab, 32, 32, lut, T)
            torch.cuda.synchronize()
        got["T %d" % T] = [e.key for e in prof.key_averages() if "downsample_task_kernel" in e.key]
    return got


@gpu
def test_plans_match_kernel_names():
    """the kernels launched are the ones the host plan names, the separate odd-pixel launch included.  The profile
    is taken in a fresh process: late in a long pytest process the profiler has been seen to record no event for the
    down-sample kernel (a programmatic-dependent launch) although the kernel ran."""
    here = os.path.dirname(os.path.abspath(__file__))
    env = dict(os.environ)
    env["PYTHONPATH"] = os.pathsep.join(p for p in (os.path.dirname(here), here, env.get("PYTHONPATH")) if p)
    code = "import json, test_gpu_label_family as t; print(json.dumps(t.launched_kernel_names()))"
    r = subprocess.run([sys.executable] + ["-s"] * sys.flags.no_user_site + ["-c", code], env=env, cwd=here,
                       capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-3000:]
    got = json.loads(r.stdout.strip().splitlines()[-1])
    first = _cm_name_cases()
    assert len(first) == 8, sorted(first)
    for path, c in first.items():
        keys = sorted(_cm_kernel_key(nm) for nm in got[path])
        assert keys == sorted(cm_plan(c.n, c.K, c.is_float, c.p_off, c.t_off)), (path, got[path])
    for T in DS_NAME_T:
        names = got["T %d" % T]
        assert len(names) == 1 and re.search(r"downsample_task_kernel<\s*%d\s*>" % ds_plan(T)["kmax"], names[0]), \
            (T, names)


# --------------------------------------------------------------------------------------
# refusals (no device needed)
# --------------------------------------------------------------------------------------
def _refuse_remap(over):
    a = dict(n_images=2, ppi=16, lo=-1, n_dom=257, masking1=0, masking2=0, map2=True)
    a.update(over)
    lab = torch.zeros(32, dtype=torch.int64, device=_dev())
    m = torch.zeros(1025, dtype=torch.int32, device=_dev())
    out = _guarded(32, torch.int64, 3, GUARD_I)
    ws = torch.full((PRES_STRIDE * 2,), 7, dtype=torch.int32, device=_dev())
    st = _lib().bacs_label_remap(lab.data_ptr(), _body(out, 32).data_ptr(), a["n_images"], a["ppi"], a["lo"],
                                 a["n_dom"], m.data_ptr(), a["masking1"], m.data_ptr() if a["map2"] else None,
                                 a["masking2"], ws.data_ptr(), _stream())
    return st, [(out, 32, 3, GUARD_I), (ws, PRES_STRIDE * 2, None, None)]


def _refuse_ds(over):
    a = dict(B=2, H=8, W=8, h=4, w=4, T=3)
    a.update(over)
    lab = torch.zeros(128, dtype=torch.int64, device=_dev())
    lut = torch.zeros(256, dtype=torch.int32, device=_dev())
    bd, bt = _guarded(32, torch.int64, 5, GUARD_I), _guarded(32, torch.int8, -128, 77)
    br, bn = _guarded(32, torch.int32, -3, -77), _guarded(260, torch.int32, -3, -77)
    st = _lib().bacs_label_downsample_task(lab.data_ptr(), a["B"], a["H"], a["W"], a["h"], a["w"], lut.data_ptr(),
                                           a["T"], _body(bd, 32).data_ptr(), _body(bt, 32).data_ptr(),
                                           _body(br, 32).data_ptr(), _body(bn, 260).data_ptr(), _stream())
    return st, [(bd, 32, 5, GUARD_I), (bt, 32, -128, 77), (br, 32, -3, -77), (bn, 260, -3, -77)]


def _refuse_hist(over):
    lab = torch.zeros(34, dtype=torch.int64, device=_dev())
    h = _guarded(257, torch.int64, 11, GUARD_I)
    st = _lib().bacs_label_hist(lab[1:].data_ptr(), 32, _body(h, 257).data_ptr(), _stream())
    return st, [(h, 257, 11, GUARD_I)]


def _refuse_cm(over):
    a = dict(K=4, n=16)
    a.update(over)
    p = torch.zeros(16, dtype=torch.int64, device=_dev())
    cm = _guarded(16, torch.int64, 9, GUARD_I)
    ob = _guarded(1, torch.int64, 9, GUARD_I)
    st = _lib().bacs_confmat_accumulate(p.data_ptr(), 0, p.data_ptr(), a["n"], a["K"], _body(cm, 16).data_ptr(),
                                        _body(ob, 1).data_ptr(), _stream())
    return st, [(cm, 16, 9, GUARD_I), (ob, 1, 9, GUARD_I)]


def _refuse_dc(over):
    a = dict(Br=4, K=21)
    a.update(over)
    n = torch.zeros(4, dtype=torch.int64, device=_dev())
    cut = _guarded(4, torch.int32, -9, -77)
    st = _lib().bacs_der_cut(n.data_ptr(), a["Br"], a["K"], _body(cut, 4).data_ptr(), _stream())
    return st, [(cut, 4, -9, -77)]


REFUSALS = [
    ("remap-ndom-0", _refuse_remap, dict(n_dom=0), "domain size 0"),
    ("remap-ndom-1025", _refuse_remap, dict(n_dom=1025), "domain size 1025"),
    ("remap-masking1-below", _refuse_remap, dict(masking1=-2), "masking values"),
    ("remap-masking1-above", _refuse_remap, dict(masking1=256), "masking values"),
    ("remap-masking2-above", _refuse_remap, dict(masking2=256), "masking values"),
    ("remap-images-65536", _refuse_remap, dict(n_images=65536), "bad sizes"),
    ("ds-T0", _refuse_ds, dict(T=0), "T=0 not in [1,128]"),
    ("ds-T129", _refuse_ds, dict(T=129), "T=129 not in [1,128]"),
    ("ds-B0", _refuse_ds, dict(B=0), "bad shape"),
    ("ds-H0", _refuse_ds, dict(H=0), "bad shape"),
    ("ds-W-1", _refuse_ds, dict(W=-1), "bad shape"),
    ("ds-h0", _refuse_ds, dict(h=0), "bad shape"),
    ("ds-w0", _refuse_ds, dict(w=0), "bad shape"),
    ("hist-unaligned", _refuse_hist, {}, "16-byte aligned"),
    ("cm-K0", _refuse_cm, dict(K=0), "bad K or n"),
    ("cm-K4097", _refuse_cm, dict(K=4097), "bad K or n"),
    ("cm-n-1", _refuse_cm, dict(n=-1), "bad K or n"),
    ("dc-Br0", _refuse_dc, dict(Br=0), "bad arguments"),
    ("dc-K0", _refuse_dc, dict(K=0), "bad arguments"),
]


@pytest.mark.parametrize("row", REFUSALS, ids=[r[0] for r in REFUSALS])
def test_label_family_refusals(row):
    """refused with a message before any launch; the outputs (and the remap workspace) stay untouched"""
    from bacs_b200 import _cabi
    _, fn, over, msg = row
    st, bufs = fn(over)
    assert st != 0 and msg in _cabi.last_error(), (st, _cabi.last_error())
    if _on_gpu():
        torch.cuda.synchronize()
    for buf, n, fill, guard in bufs:
        if fill is None:
            assert bool((buf == 7).all())
        else:
            assert _guards_intact(buf, n, guard) and bool((_body(buf, n) == fill).all())
