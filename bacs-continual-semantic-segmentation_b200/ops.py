"""Tensor-level wrappers over the C ABI: argument validation, output / workspace
allocation through PyTorch's caching allocator, and stream plumbing.  Every op is
asynchronous on the current CUDA stream and never synchronises with the host.

PyTorch is plumbing here (device memory, streams); the arithmetic is in csrc/*.cu.
There is deliberately no CPU implementation: a CPU tensor raises."""
from __future__ import annotations

import ctypes as C
from typing import Optional, Sequence, Tuple

import numpy as np
import torch

from . import _cabi
from ._cabi import PixelArgs, check

_DTYPES = {torch.float32: _cabi.F32, torch.bfloat16: _cabi.BF16, torch.float16: _cabi.F16}


def _lib():
    return _cabi.load()


def _dt(t: torch.Tensor) -> int:
    try:
        return _DTYPES[t.dtype]
    except KeyError:
        raise TypeError("bacs_b200: unsupported feature dtype %s (fp32, bf16, fp16 only)" % t.dtype)


def _cuda(t: torch.Tensor, name: str, dtype=None) -> torch.Tensor:
    if not isinstance(t, torch.Tensor) or not t.is_cuda:
        raise RuntimeError("bacs_b200.%s: expected a CUDA tensor (there is no CPU path)" % name)
    if dtype is not None and t.dtype != dtype:
        raise TypeError("bacs_b200.%s: expected dtype %s, got %s" % (name, dtype, t.dtype))
    return t if t.is_contiguous() else t.contiguous()


def _ptr(t: Optional[torch.Tensor]):
    return None if t is None else t.data_ptr()


_raw_stream = getattr(torch._C, "_cuda_getCurrentRawStream", None)


def _stream() -> int:
    """Raw handle of the current stream of the current device (the fast private accessor when this torch has
    it: torch.cuda.current_stream() builds a Stream object and costs ~10 us, nine times per step)."""
    if _raw_stream is not None:
        return _raw_stream(torch.cuda.current_device())
    return torch.cuda.current_stream().cuda_stream


def _ws(nbytes: int, device) -> torch.Tensor:
    return torch.empty(max(int(nbytes), 16), dtype=torch.uint8, device=device)


MAX_TASKS = 128   # BACS_MAX_TASKS: the int8 task map holds task ids 0..127


def check_task_count(T: int, name: str) -> None:
    """Raises BacsError unless 1 <= T <= MAX_TASKS (before any launch)."""
    if not 1 <= T <= MAX_TASKS:
        raise _cabi.BacsError("bacs_b200.%s: %d tasks; the task count must lie in [1, %d] (int8 task map)"
                              % (name, T, MAX_TASKS))


# --------------------------------------------------------------------------------------
# labels
# --------------------------------------------------------------------------------------
def label_hist(labels: torch.Tensor, out: Optional[torch.Tensor] = None) -> torch.Tensor:
    labels = _cuda(labels, "label_hist", torch.int64)
    if labels.data_ptr() % 16:       # a view such as big[1:]: the kernel reads labels in 16-byte pairs
        labels = labels.clone()
    if out is None:
        out = torch.zeros(257, dtype=torch.int64, device=labels.device)
    check(_lib().bacs_label_hist(labels.data_ptr(), labels.numel(), out.data_ptr(), _stream()), "bacs_label_hist")
    return out


def label_remap(labels: torch.Tensor, map1: torch.Tensor, masking1: int, map2: Optional[torch.Tensor] = None,
                masking2: int = 0, lo: int = -1, out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """labels int64 [N, ...] (remapped per leading-dim image); map1/map2 int32 [n_dom]."""
    labels = _cuda(labels, "label_remap", torch.int64)
    map1 = _cuda(map1, "label_remap", torch.int32)
    if map2 is not None:
        map2 = _cuda(map2, "label_remap", torch.int32)
        if map2.numel() != map1.numel():
            raise ValueError("label_remap: map1 and map2 must cover the same domain")
    n_images = labels.shape[0] if labels.dim() > 2 else 1
    ppi = labels.numel() // max(n_images, 1)
    if out is None:
        out = torch.empty_like(labels)
    lib = _lib()
    ws = _ws(lib.bacs_label_remap_workspace_bytes(n_images), labels.device)
    check(lib.bacs_label_remap(labels.data_ptr(), out.data_ptr(), n_images, ppi, lo, map1.numel(), map1.data_ptr(),
                               masking1, _ptr(map2), masking2, ws.data_ptr(), _stream()), "bacs_label_remap")
    return out


def label_downsample_task(labels: torch.Tensor, h: int, w: int, task_lut: torch.Tensor, T: int,
                          want_labels_down: bool = False):
    check_task_count(T, "label_downsample_task")
    labels = _cuda(labels, "label_downsample_task", torch.int64)
    task_lut = _cuda(task_lut, "label_downsample_task", torch.int32)
    B, H, W = labels.shape
    dev = labels.device
    task = torch.empty((B, h, w), dtype=torch.int8, device=dev)
    rank = torch.empty((B, h, w), dtype=torch.int32, device=dev)
    n_bt = torch.empty((B, T), dtype=torch.int32, device=dev)
    down = torch.empty((B, h, w), dtype=torch.int64, device=dev) if want_labels_down else None
    check(_lib().bacs_label_downsample_task(labels.data_ptr(), B, H, W, h, w, task_lut.data_ptr(), T, _ptr(down),
                                            task.data_ptr(), rank.data_ptr(), n_bt.data_ptr(), _stream()),
          "bacs_label_downsample_task")
    return task, rank, n_bt, down


# --------------------------------------------------------------------------------------
# prototypes
# --------------------------------------------------------------------------------------
def proto_accumulate(features: torch.Tensor, task: torch.Tensor, rank: torch.Tensor, n_bt: torch.Tensor, T: int,
                     mode: int = 0, out: Optional[torch.Tensor] = None) -> Tuple[torch.Tensor, torch.Tensor]:
    """Returns (sums fp64 [T,D], counts fp64 [T]) as two views of ONE packed fp64 buffer
    [T*D + T] so that a single all-reduce moves both."""
    check_task_count(T, "proto_accumulate")
    features = _cuda(features, "proto_accumulate")
    B, D, h, w = features.shape
    dev = features.device
    packed = out if out is not None else torch.empty(T * D + T, dtype=torch.float64, device=dev)
    sums, counts = packed[:T * D].view(T, D), packed[T * D:T * D + T]
    lib = _lib()
    ws = _ws(lib.bacs_proto_workspace_bytes(B, D, T), dev)
    check(lib.bacs_proto_accumulate(features.data_ptr(), _dt(features), B, D, h, w, task.data_ptr(), rank.data_ptr(),
                                    n_bt.data_ptr(), T, mode, sums.data_ptr(), counts.data_ptr(), ws.data_ptr(),
                                    ws.numel(), _stream()), "bacs_proto_accumulate")
    return sums, counts


def proto_accumulate_update(features: torch.Tensor, task: torch.Tensor, rank: torch.Tensor, n_bt: torch.Tensor, mode: int,
                            proto: torch.Tensor, count: torch.Tensor,
                            ready: Optional[torch.Tensor] = None) -> Tuple[torch.Tensor, torch.Tensor, torch.Tensor]:
    """proto_accumulate + proto_update without a launch of its own for the update (single-process step).
    Returns (sums, counts, ready)."""
    check_task_count(proto.shape[0], "proto_accumulate_update")
    features = _cuda(features, "proto_accumulate_update")
    proto = _cuda(proto, "proto_accumulate_update", torch.float32)
    if not proto.is_contiguous() or not count.is_contiguous():
        raise ValueError("proto_accumulate_update works in place: proto and count must be contiguous")
    if count.dtype not in (torch.int64, torch.float32):
        raise TypeError("proto_accumulate_update: count must be int64 or float32 (reference Q3)")
    B, D, h, w = features.shape
    T = proto.shape[0]
    dev = features.device
    packed = torch.empty(T * D + T, dtype=torch.float64, device=dev)
    sums, counts = packed[:T * D].view(T, D), packed[T * D:T * D + T]
    if ready is None:
        ready = torch.empty(1, dtype=torch.int32, device=dev)
    lib = _lib()
    ws = _ws(lib.bacs_proto_workspace_bytes(B, D, T), dev)
    check(lib.bacs_proto_accumulate_update(features.data_ptr(), _dt(features), B, D, h, w, task.data_ptr(), rank.data_ptr(),
                                           n_bt.data_ptr(), T, mode, sums.data_ptr(), counts.data_ptr(), ws.data_ptr(),
                                           ws.numel(), proto.data_ptr(), count.data_ptr(), int(count.dtype == torch.int64),
                                           ready.data_ptr(), _stream()), "bacs_proto_accumulate_update")
    return sums, counts, ready


def proto_accumulate_view(features: torch.Tensor, task: torch.Tensor, rank: torch.Tensor, n_bt: torch.Tensor, T: int,
                          view_pre: torch.Tensor, view_n: torch.Tensor,
                          out: Optional[torch.Tensor] = None) -> Tuple[torch.Tensor, torch.Tensor]:
    """proto_accumulate in the exact mode over the global view of a data-parallel batch: ``view_pre`` / ``view_n``
    (int64 [T], from distributed.exchange_task_counts) count each task's masked pixels in the images of the lower ranks
    / of all ranks.  The sums over the ranks equal the exact sums of the concatenated batch; the counts stay local."""
    check_task_count(T, "proto_accumulate_view")
    features = _cuda(features, "proto_accumulate_view")
    view_pre = _cuda(view_pre, "proto_accumulate_view", torch.int64)
    view_n = _cuda(view_n, "proto_accumulate_view", torch.int64)
    if view_pre.numel() != T or view_n.numel() != T:
        raise ValueError("proto_accumulate_view: the view needs %d entries per array" % T)
    B, D, h, w = features.shape
    dev = features.device
    packed = out if out is not None else torch.empty(T * D + T, dtype=torch.float64, device=dev)
    sums, counts = packed[:T * D].view(T, D), packed[T * D:T * D + T]
    lib = _lib()
    ws = _ws(lib.bacs_proto_workspace_bytes(B, D, T), dev)
    check(lib.bacs_proto_accumulate_view(features.data_ptr(), _dt(features), B, D, h, w, task.data_ptr(), rank.data_ptr(),
                                         n_bt.data_ptr(), T, 0, view_pre.data_ptr(), view_n.data_ptr(), sums.data_ptr(),
                                         counts.data_ptr(), ws.data_ptr(), ws.numel(), _stream()),
          "bacs_proto_accumulate_view")
    return sums, counts


def proto_task_totals(n_bt: torch.Tensor) -> torch.Tensor:
    """int64 [T]: every task's masked pixels over the images of ``n_bt`` [B, T]."""
    n_bt = _cuda(n_bt, "proto_task_totals", torch.int32)
    B, T = n_bt.shape
    check_task_count(T, "proto_task_totals")
    totals = torch.empty(T, dtype=torch.int64, device=n_bt.device)
    check(_lib().bacs_proto_task_totals(n_bt.data_ptr(), B, T, totals.data_ptr(), _stream()), "bacs_proto_task_totals")
    return totals


def proto_count_view(table: torch.Tensor, rank: int) -> Tuple[torch.Tensor, torch.Tensor]:
    """(view_pre, view_n) int64 [T] of rank ``rank`` from the gathered task totals ``table`` [world, T]."""
    table = _cuda(table, "proto_count_view", torch.int64)
    world, T = table.shape
    check_task_count(T, "proto_count_view")
    view_pre = torch.empty(T, dtype=torch.int64, device=table.device)
    view_n = torch.empty(T, dtype=torch.int64, device=table.device)
    check(_lib().bacs_proto_count_view(table.data_ptr(), world, int(rank), T, view_pre.data_ptr(), view_n.data_ptr(),
                                       _stream()), "bacs_proto_count_view")
    return view_pre, view_n


def proto_update(proto: torch.Tensor, count: torch.Tensor, sums: torch.Tensor, counts: torch.Tensor,
                 ready: Optional[torch.Tensor] = None) -> torch.Tensor:
    check_task_count(proto.shape[0], "proto_update")
    proto = _cuda(proto, "proto_update", torch.float32)
    if not proto.is_contiguous() or not count.is_contiguous():
        raise ValueError("proto_update works in place: proto and count must be contiguous")
    if count.dtype not in (torch.int64, torch.float32):
        raise TypeError("proto_update: count must be int64 or float32 (reference Q3)")
    T, D = proto.shape
    if ready is None:
        ready = torch.empty(1, dtype=torch.int32, device=proto.device)
    check(_lib().bacs_proto_update(proto.data_ptr(), count.data_ptr(), int(count.dtype == torch.int64),
                                   sums.data_ptr(), counts.data_ptr(), T, D, ready.data_ptr(), _stream()),
          "bacs_proto_update")
    return ready


# --------------------------------------------------------------------------------------
# seen / unseen heads
# --------------------------------------------------------------------------------------
def seen_logits(features: torch.Tensor, proto: torch.Tensor, weight: torch.Tensor, bias: torch.Tensor) -> torch.Tensor:
    features = _cuda(features, "seen_logits")
    proto = _cuda(proto.float(), "seen_logits")
    weight = _cuda(weight.float(), "seen_logits")
    bias = _cuda(bias.float(), "seen_logits")
    B, D, h, w = features.shape
    T = proto.shape[0]
    z = torch.empty((B, T, h, w), dtype=torch.float32, device=features.device)
    check(_lib().bacs_seen_logits(features.data_ptr(), _dt(features), B, D, h, w, proto.data_ptr(), weight.data_ptr(),
                                  bias.data_ptr(), T, z.data_ptr(), _stream()), "bacs_seen_logits")
    return z


def seen_logits_heads(features: torch.Tensor, proto: torch.Tensor, weights: Sequence[torch.Tensor],
                      biases: Sequence[torch.Tensor], zero_out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """seen_logits with the heads' own parameter tensors (fp32, contiguous: ``conv.weight`` [1,D,1,1] and ``conv.bias``
    [1] of every head) instead of a stacked copy; ``zero_out`` fp32 [B,h,w] is cleared by the same launch."""
    features = _cuda(features, "seen_logits_heads")
    proto = _cuda(proto.float(), "seen_logits_heads")
    B, D, h, w = features.shape
    T = len(weights)
    if T != len(biases) or T > proto.shape[0]:
        raise ValueError("seen_logits_heads: %d weights, %d biases, %d prototypes" % (T, len(biases), proto.shape[0]))
    for t in list(weights) + list(biases):
        if t.dtype != torch.float32 or not t.is_cuda or not t.is_contiguous():
            raise TypeError("seen_logits_heads: head parameters must be contiguous fp32 CUDA tensors")
    if any(wt.numel() != D for wt in weights):
        raise ValueError("seen_logits_heads: a head weight does not have D=%d entries" % D)
    if zero_out is not None and (zero_out.dtype != torch.float32 or tuple(zero_out.shape) != (B, h, w)
                                 or not zero_out.is_contiguous()):
        raise ValueError("seen_logits_heads: zero_out must be a contiguous fp32 [B,h,w] tensor")
    wp = (C.c_void_p * T)(*[wt.data_ptr() for wt in weights])
    bp = (C.c_void_p * T)(*[bt.data_ptr() for bt in biases])
    z = torch.empty((B, T, h, w), dtype=torch.float32, device=features.device)
    check(_lib().bacs_seen_logits_heads(features.data_ptr(), _dt(features), B, D, h, w, proto.data_ptr(), wp, bp, T,
                                        z.data_ptr(), _ptr(zero_out), _stream()), "bacs_seen_logits_heads")
    return z


def seen_logits_many(features: torch.Tensor, proto: torch.Tensor, weight, bias,
                     zero_out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """seen_logits for any head count up to MAX_TASKS (seen_logits / seen_logits_heads take at most 32).  ``weight`` /
    ``bias`` are either the stacked fp32 [T,D] / [T] tensors of seen_logits or the per-head sequences of
    seen_logits_heads; ``zero_out`` as in seen_logits_heads."""
    stacked = isinstance(weight, torch.Tensor)
    T = weight.shape[0] if stacked else len(weight)
    check_task_count(T, "seen_logits_many")
    features = _cuda(features, "seen_logits_many")
    proto = _cuda(proto.float(), "seen_logits_many")
    B, D, h, w = features.shape
    if stacked:
        weight = _cuda(weight.float(), "seen_logits_many")
        bias = _cuda(bias.float(), "seen_logits_many")
        if tuple(weight.shape) != (T, D) or bias.numel() != T:
            raise ValueError("seen_logits_many: weight must be [T,D=%d] and bias [T]" % D)
    else:
        if T != len(bias):
            raise ValueError("seen_logits_many: %d weights, %d biases" % (T, len(bias)))
        for t in list(weight) + list(bias):
            if t.dtype != torch.float32 or not t.is_cuda or not t.is_contiguous():
                raise TypeError("seen_logits_many: head parameters must be contiguous fp32 CUDA tensors")
        if any(wt.numel() != D for wt in weight):
            raise ValueError("seen_logits_many: a head weight does not have D=%d entries" % D)
    if T > proto.shape[0]:
        raise ValueError("seen_logits_many: %d heads, %d prototypes" % (T, proto.shape[0]))
    if zero_out is not None and (zero_out.dtype != torch.float32 or tuple(zero_out.shape) != (B, h, w)
                                 or not zero_out.is_contiguous()):
        raise ValueError("seen_logits_many: zero_out must be a contiguous fp32 [B,h,w] tensor")
    if stacked:
        wp = bp = None
        wd, bd = weight.data_ptr(), bias.data_ptr()
    else:
        wp = (C.c_void_p * T)(*[wt.data_ptr() for wt in weight])
        bp = (C.c_void_p * T)(*[bt.data_ptr() for bt in bias])
        wd = bd = None
    z = torch.empty((B, T, h, w), dtype=torch.float32, device=features.device)
    check(_lib().bacs_seen_logits_many(features.data_ptr(), _dt(features), B, D, h, w, proto.data_ptr(), wd, bd, wp, bp,
                                       T, z.data_ptr(), _ptr(zero_out), _stream()), "bacs_seen_logits_many")
    return z


def seen_upsample(z: torch.Tensor, scale: int = 16, apply_sigmoid: bool = False) -> torch.Tensor:
    z = _cuda(z, "seen_upsample", torch.float32)
    B, T, h, w = z.shape
    out = torch.empty((B, T, h * scale, w * scale), dtype=torch.float32, device=z.device)
    check(_lib().bacs_seen_upsample(z.data_ptr(), B, T, h, w, scale, int(apply_sigmoid), out.data_ptr(), _stream()),
          "bacs_seen_upsample")
    return out


def seen_head_backward(features: torch.Tensor, proto_t: torch.Tensor, weight_t: torch.Tensor, gz: torch.Tensor,
                       scale_dev: Optional[torch.Tensor], want_dfeatures: bool, stream: Optional[int] = None):
    """``stream``: raw handle of the stream to launch on (default: the current stream).  The outputs are allocated on
    the current stream either way; a caller that passes another stream orders it against the current one itself."""
    features = _cuda(features, "seen_head_backward")
    B, D, h, w = features.shape
    dev = features.device
    dweight = torch.empty(D, dtype=torch.float32, device=dev)
    dbias = torch.empty(1, dtype=torch.float32, device=dev)
    dfeat = torch.empty_like(features) if want_dfeatures else None
    check(_lib().bacs_seen_head_backward(features.data_ptr(), _dt(features), B, D, h, w, proto_t.data_ptr(),
                                         weight_t.data_ptr(), gz.data_ptr(), _ptr(scale_dev), dweight.data_ptr(),
                                         dbias.data_ptr(), _ptr(dfeat), _stream() if stream is None else stream),
          "bacs_seen_head_backward")
    return dweight, dbias, dfeat


def focal_scale(acc: torch.Tensor, ready: Optional[torch.Tensor], weight: float):
    """-> (scale fp32 [1], out2 fp64 [2] = {scale, scale * focal sum})"""
    dev = acc.device
    scale = torch.empty(1, dtype=torch.float32, device=dev)
    out2 = torch.empty(2, dtype=torch.float64, device=dev)
    check(_lib().bacs_focal_scale(acc.data_ptr(), _ptr(ready), float(weight), scale.data_ptr(), out2.data_ptr(),
                                  _stream()), "bacs_focal_scale")
    return scale, out2


def focal_scale_loss(acc: torch.Tensor, ready: Optional[torch.Tensor], weight: float, main_coef: float,
                     main_over_wsum: bool):
    """-> (focal scale fp32 [1], loss fp32 [1] = main_coef * acc[LOSS] (/ acc[WSUM]) + scale * acc[FOCAL])"""
    dev = acc.device
    scale = torch.empty(1, dtype=torch.float32, device=dev)
    loss = torch.empty(1, dtype=torch.float32, device=dev)
    check(_lib().bacs_focal_scale_loss(acc.data_ptr(), _ptr(ready), float(weight), float(main_coef),
                                       int(bool(main_over_wsum)), scale.data_ptr(), loss.data_ptr(), _stream()),
          "bacs_focal_scale_loss")
    return scale, loss


# --------------------------------------------------------------------------------------
# fused per-pixel kernel
# --------------------------------------------------------------------------------------
def pixel_loss(logits: torch.Tensor, labels: torch.Tensor, mode: int, *, want_grad: bool, want_preds: bool = True,
               z: Optional[torch.Tensor] = None, want_distill_mask: bool = False, focal_head: int = -1,
               class_w: Optional[torch.Tensor] = None, hist: Optional[torch.Tensor] = None, old_cl: int = 0,
               ukd: bool = True, gamma: float = 2.0, threshold: float = 0.5, focal_gamma: float = 2.0,
               focal_alpha: Optional[float] = None, lkd_threshold: float = 0.5, ignore_index: int = 255,
               grad_scale: float = 1.0, seen_scale: int = 16, want_score: bool = False,
               seen_max: Optional[torch.Tensor] = None, epilogue: Optional[dict] = None,
               lowres: bool = False, gz: Optional[torch.Tensor] = None) -> dict:
    """``epilogue`` = {"ready": int32 [1] tensor or None, "focal_weight": float, "loss_coef": float,
    "over_wsum": bool}: the reduction launch also writes out["focal_scale"] and out["loss"] (fp32 [1]).

    ``lowres=True``: ``logits`` are the network's low-res ``sem_logits`` [B,K,lh,lw] (``return_sem_logits=True``,
    networks/deeplab_v3.py:155-156); the x16 / x8 bilinear up-sample (align_corners=False, deeplab_v3.py:157-160) and
    its adjoint are evaluated inside the kernel, ``out["dlogits"]`` is d loss / d sem_logits.

    ``gz``: an already ZEROED fp32 [B,h,w] accumulator for the focal gradient (``seen_logits_heads(zero_out=...)`` clears
    it in its own launch); allocated and cleared here when absent."""
    logits = _cuda(logits, "pixel_loss")
    labels = _cuda(labels, "pixel_loss", torch.int64)
    B, K = logits.shape[0], logits.shape[1]
    if lowres:
        if labels.dim() != 3 or labels.shape[0] != B:
            raise ValueError("pixel_loss: labels %s do not match sem_logits %s" % (tuple(labels.shape), tuple(logits.shape)))
        H, W = labels.shape[1], labels.shape[2]
    else:
        H, W = logits.shape[2], logits.shape[3]
    if tuple(labels.shape) != (B, H, W):
        raise ValueError("pixel_loss: labels %s do not match logits %s" % (tuple(labels.shape), tuple(logits.shape)))
    dev = logits.device
    a = PixelArgs()
    out = {}
    a.logits, a.labels = logits.data_ptr(), labels.data_ptr()
    out["dlogits"] = torch.empty_like(logits) if want_grad else None
    out["preds"] = torch.empty((B, H, W), dtype=torch.int64, device=dev) if want_preds else None
    out["acc"] = torch.empty(_cabi.NACC, dtype=torch.float64, device=dev)
    out["distill_mask"] = torch.empty((B, H, W), dtype=torch.uint8, device=dev) if want_distill_mask else None
    out["gz"] = None
    out["score"] = torch.empty(B, dtype=torch.float64, device=dev) if want_score else None
    a.T = a.h = a.w = 0
    if z is not None:
        z = _cuda(z, "pixel_loss", torch.float32)
        a.T, a.h, a.w = z.shape[1], z.shape[2], z.shape[3]
        if focal_head >= 0:
            if gz is not None and (gz.dtype != torch.float32 or tuple(gz.shape) != (B, a.h, a.w) or not gz.is_contiguous()):
                raise ValueError("pixel_loss: gz must be a contiguous fp32 [B,h,w] tensor")
            out["gz"] = gz if gz is not None else torch.zeros((B, a.h, a.w), dtype=torch.float32, device=dev)
    if seen_max is not None:
        seen_max = _cuda(seen_max.float(), "pixel_loss")
        if tuple(seen_max.shape) != (B, H, W):
            raise ValueError("pixel_loss: seen_max must be [B,H,W]")
    a.seen_max = _ptr(seen_max)
    if class_w is not None:
        class_w = _cuda(class_w.float(), "pixel_loss")
        if class_w.numel() != K:
            raise ValueError("pixel_loss: class weights must have K=%d entries" % K)
    need_hist = want_grad and mode in (_cabi.PIX_CE, _cabi.PIX_UNBIASED_CE)
    if need_hist and hist is None:
        hist = label_hist(labels)
    a.dlogits, a.preds, a.z = _ptr(out["dlogits"]), _ptr(out["preds"]), _ptr(z)
    a.distill_mask, a.gz, a.class_w = _ptr(out["distill_mask"]), _ptr(out["gz"]), _ptr(class_w)
    a.hist, a.acc, a.score = _ptr(hist), out["acc"].data_ptr(), _ptr(out["score"])
    a.B, a.K, a.H, a.W = B, K, H, W
    a.dtype, a.mode = _dt(logits), mode
    a.old_cl, a.ukd, a.focal_head = int(old_cl), int(bool(ukd)), int(focal_head)
    a.ignore_index, a.seen_scale = int(ignore_index), int(seen_scale)
    a.gamma, a.threshold, a.focal_gamma = float(gamma), float(threshold), float(focal_gamma)
    a.focal_alpha = -1.0 if focal_alpha is None else float(focal_alpha)
    a.lkd_threshold, a.grad_scale = float(lkd_threshold), float(grad_scale)
    out["focal_scale"] = out["loss"] = None
    a.ready = a.focal_scale_out = a.loss_out = None
    a.focal_weight = a.loss_coef = 0.0
    a.loss_over_wsum = 0
    if epilogue is not None:
        out["focal_scale"] = torch.empty(1, dtype=torch.float32, device=dev)
        out["loss"] = torch.empty(1, dtype=torch.float32, device=dev)
        a.ready = _ptr(epilogue.get("ready"))
        a.focal_scale_out, a.loss_out = out["focal_scale"].data_ptr(), out["loss"].data_ptr()
        a.focal_weight, a.loss_coef = float(epilogue.get("focal_weight", 0.0)), float(epilogue["loss_coef"])
        a.loss_over_wsum = int(bool(epilogue.get("over_wsum", False)))
    lib = _lib()
    if lowres:
        lh, lw = int(logits.shape[2]), int(logits.shape[3])
        nbytes = lib.bacs_pixel_lowres_workspace_bytes(C.byref(a), lh, lw)
        if nbytes == 0:
            raise _cabi.BacsError("bacs_pixel_loss_lowres: unsupported geometry %s -> (%d, %d), K=%d"
                                  % (tuple(logits.shape), H, W, K))
        ws = _ws(nbytes, dev)
        check(lib.bacs_pixel_loss_lowres(C.byref(a), lh, lw, ws.data_ptr(), ws.numel(), _stream()),
              "bacs_pixel_loss_lowres")
        out["hist"] = hist
        out["variant"] = 3
        return out
    nbytes = lib.bacs_pixel_workspace_bytes(C.byref(a))
    if nbytes == 0:
        raise _cabi.BacsError("bacs_pixel_loss: no tile plan for K=%d" % K)
    ws = _ws(nbytes, dev)
    check(lib.bacs_pixel_loss(C.byref(a), ws.data_ptr(), ws.numel(), _stream()), "bacs_pixel_loss")
    out["hist"] = hist
    out["variant"] = lib.bacs_pixel_kernel_variant(C.byref(a))
    return out


def pseudo_label_inplace(labels: torch.Tensor, teacher_logits: torch.Tensor, lowres: bool = False) -> torch.Tensor:
    """labels[labels == 0] = teacher_logits.argmax(1)[labels == 0] in place (bacs_loss.py:205-210), in one launch and
    without a host synchronisation; ties go to the lowest channel, every other label keeps its value.  Returns
    ``labels`` (int64 [B,H,W]; a non-contiguous tensor is rewritten through a contiguous copy).

    ``teacher_logits``: [B,K_t,H,W], or with ``lowres=True`` the teacher's low-res ``sem_logits`` [B,K_t,lh,lw] whose
    bilinear up-sample (align_corners=False) is evaluated inside the arg-max -- then the pseudo labels equal the
    ``preds`` of ``pixel_loss(..., lowres=True)`` at the same sem_logits.  K_t may differ from the student's K."""
    work = _cuda(labels, "pseudo_label_inplace", torch.int64)
    teacher = _cuda(teacher_logits, "pseudo_label_inplace")
    if work.dim() != 3 or teacher.dim() != 4 or teacher.shape[0] != work.shape[0] \
            or (not lowres and tuple(teacher.shape[2:]) != tuple(work.shape[1:])):
        raise ValueError("pseudo_label_inplace: labels %s do not match teacher logits %s"
                         % (tuple(labels.shape), tuple(teacher_logits.shape)))
    B, H, W = work.shape
    Kt = teacher.shape[1]
    if lowres:
        check(_lib().bacs_pseudo_label_lowres(teacher.data_ptr(), _dt(teacher), B, Kt, teacher.shape[2], teacher.shape[3],
                                              H, W, work.data_ptr(), _stream()), "bacs_pseudo_label_lowres")
    else:
        check(_lib().bacs_pseudo_label(teacher.data_ptr(), _dt(teacher), B, Kt, H, W, work.data_ptr(), _stream()),
              "bacs_pseudo_label")
    if work is not labels:
        labels.copy_(work)
    return labels


# --------------------------------------------------------------------------------------
# teacher distillation / DER
# --------------------------------------------------------------------------------------
def teacher_distill(old_att: torch.Tensor, new_att: torch.Tensor, mask: Optional[torch.Tensor], out_hw,
                    grad_coef: float, want_grad: bool, want_scaled: bool = False, addend: Optional[torch.Tensor] = None):
    """-> (sum of row norms fp64 [1], grad_coef * d(sum)/d(new) or None[, grad_coef * sum as fp32 [1]])
    ``addend`` (fp32 scalar on the device, with ``want_scaled``): the scaled output is addend + grad_coef * sum."""
    old_att = _cuda(old_att, "teacher_distill")
    new_att = _cuda(new_att, "teacher_distill")
    if old_att.dtype != new_att.dtype:
        old_att = old_att.to(new_att.dtype)
    if old_att.shape != new_att.shape:
        raise ValueError("teacher_distill: attention shapes differ")
    B, A, h, w = new_att.shape
    H, W = out_hw
    if mask is not None:
        mask = _cuda(mask, "teacher_distill", torch.uint8)
    dev = new_att.device
    loss_sum = torch.empty(1, dtype=torch.float64, device=dev)
    loss_scaled = torch.empty(1, dtype=torch.float32, device=dev) if want_scaled else None
    dnew = torch.empty_like(new_att) if want_grad else None
    lib = _lib()
    ws = _ws(lib.bacs_distill_workspace_bytes(B, A, h, w, H, W), dev)
    if addend is not None:
        if not want_scaled or addend.dtype != torch.float32 or addend.numel() != 1 or not addend.is_cuda:
            raise ValueError("teacher_distill: addend must be a CUDA fp32 scalar and needs want_scaled")
        check(lib.bacs_teacher_distill_add(old_att.data_ptr(), new_att.data_ptr(), _dt(new_att), B, A, h, w, _ptr(mask), H,
                                           W, float(grad_coef), loss_sum.data_ptr(), loss_scaled.data_ptr(),
                                           addend.data_ptr(), _ptr(dnew), ws.data_ptr(), ws.numel(), _stream()),
              "bacs_teacher_distill_add")
    else:
        check(lib.bacs_teacher_distill(old_att.data_ptr(), new_att.data_ptr(), _dt(new_att), B, A, h, w, _ptr(mask), H, W,
                                       float(grad_coef), loss_sum.data_ptr(), _ptr(loss_scaled), _ptr(dnew), ws.data_ptr(),
                                       ws.numel(), _stream()), "bacs_teacher_distill")
    if want_scaled:
        return loss_sum, dnew, loss_scaled
    return loss_sum, dnew


def distill_set_mode(mode: int) -> None:
    """0: tensor-core kernel where it applies (default), 1: FMA kernel only, 2: tensor-core kernel or an error."""
    check(_lib().bacs_distill_set_mode(int(mode)), "bacs_distill_set_mode")


def distill_kernel_variant(att: torch.Tensor, out_hw) -> int:
    """1 when bacs_teacher_distill serves this shape on the tensor cores, 0 for the packed-fp32 kernel."""
    B, A, h, w = att.shape
    return int(_lib().bacs_distill_kernel_variant(_dt(att), B, A, h, w, int(out_hw[0]), int(out_hw[1])))


def der_transplant_cut(n_classes, K: int) -> np.ndarray:
    """Host restatement of the transplant index quirk (loss/bacs_loss.py:415-425): for i, n
    in enumerate(unique(n_classes)) the sample touched is inverse[i], not the samples whose
    class count is n.  n_classes is a tiny host array (it comes from the buffer loader)."""
    n_classes = np.asarray(n_classes).astype(np.int64).reshape(-1)
    uniq, inv = np.unique(n_classes, return_inverse=True)
    cut = np.full(n_classes.shape[0], K, dtype=np.int32)
    for i, n in enumerate(uniq.tolist()):
        j = int(inv[i])
        if n < K:
            cut[j] = min(int(cut[j]), int(n))
    return cut


def der_cut(n_classes: torch.Tensor, K: int) -> torch.Tensor:
    """Device version of der_transplant_cut (no host synchronisation)."""
    if not n_classes.is_cuda:
        raise RuntimeError("bacs_b200.der_cut: expected a CUDA tensor (there is no CPU path)")
    n = n_classes.reshape(-1).long().contiguous()
    cut = torch.empty(n.numel(), dtype=torch.int32, device=n.device)
    check(_lib().bacs_der_cut(n.data_ptr(), n.numel(), int(K), cut.data_ptr(), _stream()), "bacs_der_cut")
    return cut


def der_mse(sem_logits: torch.Tensor, memory_logits: torch.Tensor, cut: torch.Tensor, ignore_rep_bg: bool,
            truncate: bool, grad_coef: float, want_grad: bool):
    sem_logits = _cuda(sem_logits, "der_mse")
    memory_logits = _cuda(memory_logits, "der_mse")
    is_i64 = memory_logits.dtype == torch.int64
    if not is_i64 and memory_logits.dtype != torch.float32:
        memory_logits = memory_logits.float()
    cut = _cuda(cut, "der_mse", torch.int32)
    Br, K, h, w = sem_logits.shape
    if memory_logits.shape != sem_logits.shape:
        raise ValueError("der_mse: stored logits %s vs live %s (pad with change_data_size first)"
                         % (tuple(memory_logits.shape), tuple(sem_logits.shape)))
    dev = sem_logits.device
    loss_sum = torch.empty(1, dtype=torch.float64, device=dev)
    dsem = torch.empty_like(sem_logits) if want_grad else None
    lib = _lib()
    ws = _ws(lib.bacs_der_workspace_bytes(Br, K, h * w), dev)
    check(lib.bacs_der_mse(sem_logits.data_ptr(), _dt(sem_logits), memory_logits.data_ptr(), int(is_i64),
                           int(truncate), cut.data_ptr(), int(ignore_rep_bg), Br, K, h * w, float(grad_coef),
                           loss_sum.data_ptr(), _ptr(dsem), ws.data_ptr(), ws.numel(), _stream()), "bacs_der_mse")
    return loss_sum, dsem


def unbiased_kd(logits: torch.Tensor, old_logits: torch.Tensor, mask: Optional[torch.Tensor], alpha: float,
                grad_coef: float, want_grad: bool):
    logits = _cuda(logits, "unbiased_kd")
    old_logits = _cuda(old_logits.to(logits.dtype), "unbiased_kd")
    B, K, H, W = logits.shape
    Ko = old_logits.shape[1]
    if mask is not None:
        mask = _cuda(mask.to(torch.uint8), "unbiased_kd", torch.uint8)
    dev = logits.device
    loss_sum = torch.empty(1, dtype=torch.float64, device=dev)
    dx = torch.empty_like(logits) if want_grad else None
    lib = _lib()
    ws = _ws(lib.bacs_unbiased_kd_workspace_bytes(B * H * W), dev)
    check(lib.bacs_unbiased_kd(logits.data_ptr(), old_logits.data_ptr(), _dt(logits), B, K, Ko, H, W, float(alpha),
                               _ptr(mask), float(grad_coef), loss_sum.data_ptr(), _ptr(dx), ws.data_ptr(), ws.numel(),
                               _stream()), "bacs_unbiased_kd")
    return loss_sum, dx


# --------------------------------------------------------------------------------------
# confusion matrix
# --------------------------------------------------------------------------------------
def confmat_accumulate(preds: torch.Tensor, target: torch.Tensor, K: int, confmat: torch.Tensor,
                       oob: Optional[torch.Tensor] = None) -> torch.Tensor:
    target = _cuda(target, "confmat_accumulate", torch.int64)
    if not preds.is_cuda:
        raise RuntimeError("bacs_b200.confmat_accumulate: expected CUDA tensors (there is no CPU path)")
    if preds.dtype == torch.int64:
        is_float = 0
    else:
        preds = preds.float()
        is_float = 1
    preds = preds.contiguous()
    if preds.numel() != target.numel():
        raise ValueError("confmat_accumulate: preds and target sizes differ")
    if confmat.dtype != torch.int64 or confmat.numel() != K * K or not confmat.is_contiguous():
        raise ValueError("confmat_accumulate: confmat must be a contiguous int64 [K,K]")
    check(_lib().bacs_confmat_accumulate(preds.data_ptr(), is_float, target.data_ptr(), target.numel(), K,
                                         confmat.data_ptr(), _ptr(oob), _stream()), "bacs_confmat_accumulate")
    return confmat


def confmat_metrics(confmat: torch.Tensor) -> torch.Tensor:
    confmat = _cuda(confmat, "confmat_metrics", torch.int64)
    K = confmat.shape[0]
    out = torch.empty((6, K), dtype=torch.float32, device=confmat.device)
    check(_lib().bacs_confmat_metrics(confmat.data_ptr(), K, out.data_ptr(), _stream()), "bacs_confmat_metrics")
    return out


# --------------------------------------------------------------------------------------
# scalar helpers
# --------------------------------------------------------------------------------------
def class_distance(features: torch.Tensor, class_protos: torch.Tensor, want_nearest: bool = True):
    """Squared distance of every pixel feature to every class prototype on the tensor cores (bf16 operands, fp32
    accumulation): features [B,D,h,w], class_protos [Kc,D] -> (dist2 fp32 [B,Kc,h,w], nearest int64 [B,h,w] or None)."""
    features = _cuda(features, "class_distance")
    class_protos = _cuda(class_protos, "class_distance")
    if features.dtype != torch.bfloat16:
        features = features.to(torch.bfloat16)
    if class_protos.dtype != torch.bfloat16:
        class_protos = class_protos.to(torch.bfloat16)
    B, D, h, w = features.shape
    Kc = class_protos.shape[0]
    if class_protos.shape[1] != D:
        raise ValueError("class_distance: prototypes %s do not match features %s" % (tuple(class_protos.shape),
                                                                                     tuple(features.shape)))
    dev = features.device
    dist2 = torch.empty((B, Kc, h, w), dtype=torch.float32, device=dev)
    nearest = torch.empty((B, h, w), dtype=torch.int64, device=dev) if want_nearest else None
    lib = _lib()
    ws = _ws(lib.bacs_class_distance_workspace_bytes(B, Kc, D, h, w), dev)
    check(lib.bacs_class_distance(features.data_ptr(), _dt(features), B, D, h, w, class_protos.data_ptr(), Kc,
                                  dist2.data_ptr(), _ptr(nearest), ws.data_ptr(), ws.numel(), _stream()),
          "bacs_class_distance")
    return dist2, nearest


def class_sums(features: torch.Tensor, labels_down: torch.Tensor, K: int) -> Tuple[torch.Tensor, torch.Tensor]:
    """Per-class feature sums and pixel counts (the per-class prototype family, SURVEY 8f-4): features [B,D,h,w],
    labels_down int64 [B,h,w] class ids (ids outside [0,K), e.g. ignore-255, are skipped) ->
    (sums fp64 [K,D], counts int64 [K])."""
    features = _cuda(features, "class_sums")
    labels_down = _cuda(labels_down, "class_sums", torch.int64)
    B, D, h, w = features.shape
    if tuple(labels_down.shape) != (B, h, w):
        raise ValueError("class_sums: labels %s do not match features %s" % (tuple(labels_down.shape), tuple(features.shape)))
    if not 0 < K <= 256:
        raise ValueError("class_sums: K must be in (0, 256] (the label histogram has 256 bins)")
    dev = features.device
    sums = torch.empty((K, D), dtype=torch.float64, device=dev)
    lib = _lib()
    ws = _ws(lib.bacs_class_sums_workspace_bytes(B, D, K), dev)
    check(lib.bacs_class_sums(features.data_ptr(), _dt(features), B, D, h, w, labels_down.data_ptr(), K, sums.data_ptr(),
                              ws.data_ptr(), ws.numel(), _stream()), "bacs_class_sums")
    return sums, label_hist(labels_down)[:K]


def gather_rows(src: torch.Tensor, idx: torch.Tensor) -> torch.Tensor:
    """out[i] = src[idx[i]] along dim 0 (any dtype; rows are copied as bytes)."""
    src = _cuda(src, "gather_rows")
    idx = _cuda(idx, "gather_rows", torch.int64)
    n = int(idx.numel())
    out = torch.empty((n,) + tuple(src.shape[1:]), dtype=src.dtype, device=src.device)
    if n and src.shape[0]:
        row_bytes = src[0].numel() * src.element_size()
        if row_bytes:
            check(_lib().bacs_gather_rows(src.data_ptr(), src.shape[0], row_bytes, idx.data_ptr(), n, out.data_ptr(),
                                          _stream()), "bacs_gather_rows")
    return out


def scale_inplace(x: torch.Tensor, g: torch.Tensor) -> torch.Tensor:
    """x *= g for a device scalar g (fp32 [1] or 0-d); returns immediately on the device when g == 1."""
    if g.dtype != torch.float32:
        g = g.float()
    check(_lib().bacs_scale_inplace(x.data_ptr(), _dt(x), x.numel(), g.data_ptr(), _stream()), "bacs_scale_inplace")
    return x


def scale_inplace_multi(xs: Sequence[Optional[torch.Tensor]], g: torch.Tensor) -> None:
    """x *= g for every tensor of ``xs`` (None entries skipped) in one launch; g is a device scalar."""
    live = [x for x in xs if x is not None and x.numel() > 0]
    if not live:
        return
    for x in live:
        _cuda(x, "scale_inplace_multi")
        if not x.is_contiguous():
            raise ValueError("scale_inplace_multi works in place: tensors must be contiguous")
    g = _cuda(g.reshape(1).float(), "scale_inplace_multi")
    n = len(live)
    if n > 8:
        raise ValueError("scale_inplace_multi: at most 8 tensors")
    ptrs = (C.c_void_p * n)(*[x.data_ptr() for x in live])
    dts = (C.c_int * n)(*[_dt(x) for x in live])
    nums = (C.c_int64 * n)(*[x.numel() for x in live])
    check(_lib().bacs_scale_inplace_multi(n, ptrs, dts, nums, g.data_ptr(), _stream()), "bacs_scale_inplace_multi")


def combine_scalars(terms: Sequence[tuple], device) -> torch.Tensor:
    """terms: (src fp64 tensor, index, coef[, den fp64 tensor, den index]) -> fp32 [1]
    = sum coef * src[idx] / den[didx]."""
    n = len(terms)
    src = (C.c_void_p * n)()
    den = (C.c_void_p * n)()
    idx = (C.c_int * n)()
    didx = (C.c_int * n)()
    coef = (C.c_float * n)()
    for i, t in enumerate(terms):
        src[i], idx[i], coef[i] = t[0].data_ptr(), int(t[1]), float(t[2])
        if len(t) > 3 and t[3] is not None:
            den[i], didx[i] = t[3].data_ptr(), int(t[4])
        else:
            den[i], didx[i] = None, 0
    out = torch.empty(1, dtype=torch.float32, device=device)
    check(_lib().bacs_combine_scalars(n, src, idx, den, didx, coef, out.data_ptr(), _stream()),
          "bacs_combine_scalars")
    return out


def pack_state(sums: Optional[torch.Tensor], counts: Optional[torch.Tensor], confmat: Optional[torch.Tensor],
               device) -> torch.Tensor:
    T, D = (sums.shape if sums is not None else (0, 0))
    K = confmat.shape[0] if confmat is not None else 0
    packed = torch.empty(T * D + T + K * K, dtype=torch.float64, device=device)
    check(_lib().bacs_pack_state(_ptr(sums), _ptr(counts), T, D, _ptr(confmat), K, packed.data_ptr(), _stream()),
          "bacs_pack_state")
    return packed


def unpack_state(packed: torch.Tensor, sums: Optional[torch.Tensor], counts: Optional[torch.Tensor],
                 confmat: Optional[torch.Tensor]) -> None:
    T, D = (sums.shape if sums is not None else (0, 0))
    K = confmat.shape[0] if confmat is not None else 0
    check(_lib().bacs_unpack_state(packed.data_ptr(), T, D, _ptr(sums), _ptr(counts), _ptr(confmat), K, _stream()),
          "bacs_unpack_state")


# --------------------------------------------------------------------------------------
# BACS_NVTX=1: every op of this module runs inside an NVTX range named after it (timeline tools then show the step as
# bacs/label_downsample_task, bacs/proto_accumulate_update, bacs/seen_logits_heads, bacs/pixel_loss, bacs/teacher_distill
# ...).  Off by default: the ranges cost a few microseconds of host time per op.
# --------------------------------------------------------------------------------------
def _install_nvtx_ranges():
    import functools
    import os
    if os.environ.get("BACS_NVTX") != "1":
        return

    def wrap(fn):
        @functools.wraps(fn)
        def inner(*args, **kwargs):
            torch.cuda.nvtx.range_push("bacs/" + fn.__name__)
            try:
                return fn(*args, **kwargs)
            finally:
                torch.cuda.nvtx.range_pop()
        return inner
    skip = {"check", "der_transplant_cut"}
    for name, obj in list(globals().items()):
        if callable(obj) and getattr(obj, "__module__", None) == __name__ and not name.startswith("_") and name not in skip \
                and not isinstance(obj, type):
            globals()[name] = wrap(obj)


_install_nvtx_ranges()
