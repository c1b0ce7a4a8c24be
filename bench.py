#!/usr/bin/env python
"""bench.py -- BACS loss step throughput (pixels/s, forward + backward) on B200.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--config NAME] [--dump-outputs DIR]

One "step" = one pass of the whole BACS loss path (SURVEY 8a rows 3-12) over one batch of
synthetic network outputs: prototype update, seen-head logits, fused weighted-CE + focal +
arg-max + distill-mask kernel with d(loss)/d(logits), teacher-distill fwd+bwd, head
backward -- called through the reference-facing class interface
``BACSLoss.compute_loss(batch, network, train=True)`` followed by ``loss.backward()``.
The network itself is out of scope: a stand-in returns fixed tensors.

Workload at N = 1: BASELINE.json configs[1] -- VOC 15-1 overlap step, 512x512 crops, B=24,
K=21, T=6 prototypes, D=512, A=256, bf16 logits/features.  For N > 1 every rank runs the
same per-GPU workload (weak scaling) and the per-task prototype sums/counts travel in one
packed fp64 NCCL all-reduce per step.

Prints ONE JSON line (rank 0).  --impl reference times the reference's OWN code for the path
(oracle/_ref, staged by oracle/make_ref.py: the unmodified loss/bacs_loss.py step; the oracle
port only when that tree is absent) on the host cores, on a bounded sample of the same workload.

  --config cityscapes_eval   times only the integer rows (confusion matrix at the Cityscapes
                             1024x2048 evaluation shape, label remap, label down-sample) in GB/s."""
from __future__ import annotations

import argparse
import json
import os
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "BACS loss step pixels/sec (fwd+bwd)"
UNIT = "pixels/s"


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=None,
                    help="timed steps of every timed window (default: 200; 2 with --impl reference, whose step takes "
                         "seconds on the host; 20 with --config cityscapes_eval)")
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", default="voc15-1_b24")
    ap.add_argument("--dtype", default="bf16", choices=["bf16", "fp32", "fp16"])
    ap.add_argument("--cpu-sample-batch", type=int, default=2,
                    help="images per CPU step of the cpu_baseline block (default run: bounded to ~10-30 s)")
    ap.add_argument("--ref-sample-batch", type=int, default=8,
                    help="images per step of --impl reference (the reference materialises 2 x 0.27 GB per image)")
    ap.add_argument("--no-graph", action="store_true", help="do not also time the CUDA-graph replay of the step")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-fused-lowres", action="store_true",
                    help="skip the extra timing of BACSLoss(fused_logit_upsample=True) (low-res logits in, N=1 only)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last timed step returned (loss, arg-max, gradients, "
                         "updated prototypes and counts) as DIR/<name>.npy, to compare two builds output for output")
    args = ap.parse_args()
    if args.steps is None:
        args.steps = 2 if args.impl == "reference" else 20 if args.config == "cityscapes_eval" else 200
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl == "reference" or args.config == "cityscapes_eval"):
        ap.error("--dump-outputs writes what the BACS loss step on the GPU returns; --impl reference and "
                 "--config cityscapes_eval do not run that step")
    return args


DUMP_SAMPLE = 1 << 20


def host_sample(t):
    """-> a host numpy copy of ``t``: float64 stays float64, everything else becomes float32.  A tensor of more than
    DUMP_SAMPLE elements is replaced by its elements at DUMP_SAMPLE flat positions drawn from a generator with a fixed
    seed, so every run of every build keeps the same positions (at most 8 MB per array)."""
    import numpy as np
    import torch
    t = t.detach()
    if t.numel() > DUMP_SAMPLE:
        idx = np.sort(np.random.default_rng(0).integers(0, t.numel(), DUMP_SAMPLE))
        t = t.reshape(-1)[torch.from_numpy(idx).to(t.device)]
    return t.to(torch.float64 if t.dtype == torch.float64 else torch.float32).cpu().numpy()


def peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            p = json.load(f)
        return float(p["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler(threading.Thread):
    """Samples SM clock and throttle reasons through NVML while the timed regions run."""

    def __init__(self, index: int):
        super().__init__(daemon=True)
        self.index, self.samples, self.reasons, self.stop_flag = index, [], set(), False
        self.sm_max = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.sm_max = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nv = None

    def run(self):
        if self.nv is None:
            return
        nv = self.nv
        names = {nv.nvmlClocksThrottleReasonHwSlowdown: "hw_slowdown",
                 nv.nvmlClocksThrottleReasonHwThermalSlowdown: "hw_thermal_slowdown",
                 nv.nvmlClocksThrottleReasonSwThermalSlowdown: "sw_thermal_slowdown",
                 nv.nvmlClocksThrottleReasonSwPowerCap: "sw_power_cap"}
        while not self.stop_flag:
            try:
                util = nv.nvmlDeviceGetUtilizationRates(self.h).gpu
                clk = nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)
                mask = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                self.samples.append((clk, util))
                for bit, name in names.items():
                    if mask & bit:
                        self.reasons.add(name)
            except Exception:
                pass
            time.sleep(0.01)

    def summary(self):
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.sm_max, "reasons": [], "note": "NVML unavailable"}
        loaded = sorted(c for c, u in self.samples if u > 0) or sorted(c for c, _ in self.samples)
        return {"sm_mhz": loaded[len(loaded) // 2], "sm_max_mhz": self.sm_max, "reasons": sorted(self.reasons),
                "samples": len(self.samples)}


def cpu_step_time(cfg, batch, steps, warmup):
    """CPU baseline of the path: the reference's own BACSLoss.compute_loss + backward when its modules are staged
    (oracle/_ref, kind "reference"), else the oracle port (kind "port"); fp32, all host threads.
    -> (pixels/s, seconds per step, description, kind)"""
    import dataclasses
    import torch
    from bacs_b200 import synth
    small = dataclasses.replace(cfg, B=batch, Br=0)
    inp = synth.make_step_inputs(small, seed=0, dtype=torch.float32, with_replay=False)
    px = small.B * small.H * small.W
    from oracle import ref_step
    if ref_step.available():
        dt, _ = ref_step.time_step(small, inp, steps=steps, warmup=warmup)
        kind = "reference"
        what = "unmodified reference BACSLoss.compute_loss+backward (oracle/_ref)"
    else:
        from oracle import bacs_oracle as O

        def step():
            leaf = lambda t: t.clone().requires_grad_(True)
            lg, na, hw, hb = leaf(inp.logits), leaf(inp.new_att), leaf(inp.head_w), leaf(inp.head_b)
            out = O.bacs_step(lg, inp.pen, inp.old_att, na, inp.mask, inp.protos, inp.counts, hw, hb,
                              initial_classes=small.initial_classes, increment=small.increment, old_cl=small.old_cl,
                              task_num=small.T - 1, epoch=3, max_epochs=30)
            out["loss"].backward()
        for _ in range(warmup):
            step()
        t0 = time.perf_counter()
        for _ in range(steps):
            step()
        dt = (time.perf_counter() - t0) / steps
        kind = "port"
        what = "oracle port of the reference step (oracle/bacs_oracle.py)"
    return px / dt, dt, "%s, fp32, B=%d of the B=%d %dx%d K=%d D=%d A=%d step, %d timed steps" % (
        what, small.B, cfg.B, small.H, small.W, small.K, small.D, small.A, steps), kind


def run_reference(args):
    import torch
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from bacs_b200 import synth
    # torchrun exports OMP_NUM_THREADS=1: the reference arm uses every host core this process may run on
    try:
        ncores = len(os.sched_getaffinity(0))
    except AttributeError:
        ncores = os.cpu_count() or 1
    torch.set_num_threads(max(1, ncores))
    cfg = synth.CONFIGS[args.config]
    steps, warmup = args.steps, 0
    batch = max(1, min(args.ref_sample_batch, cfg.B))
    value, dt, sample, kind = cpu_step_time(cfg, batch, steps, warmup)
    cores = torch.get_num_threads()
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
            "steps": steps, "warmup": warmup, "ms_per_step": dt * 1e3, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": workload_name(cfg), "per_step_sample": sample,
                       "same_config": batch == cfg.B},
            "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": kind, "sample": sample},
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)


def workload_name(cfg):
    return ("%s: BACS step B=%d K=%d old_cl=%d T=%d %dx%d (features %dx%d) D=%d A=%d" %
            (cfg.name, cfg.B, cfg.K, cfg.old_cl, cfg.T, cfg.H, cfg.W, cfg.h, cfg.w, cfg.D, cfg.A))


def integer_rows(timed_fn, dev, peak, shape=(4, 1024, 2048), K=20, steps=20):
    """The integer rows of the path, each timed alone on inputs larger than L2 (SURVEY 8a rows 14, 0, 3):
    * confusion-matrix histogram at the Cityscapes evaluation shape (training/metrics.py:38-50): 16 B of int64
      predictions + targets per pixel; on uniformly random classes (every lane a different bin: the worst case for
      the shared-memory histogram) and on a blocky map with 10 % wrong pixels (what an evaluation pass looks like);
    * label remap (training/utils.py:225-261): the labels present decide the mapping (sequential aliasing, Q13), so
      the image is read twice (presence, remap) and written once: 24 B per pixel;
    * nearest label down-sample + class -> task + raster rank (loss/prototypes.py:177-205): only one pixel in 256 is
      read -- one 32-byte sector per low-res pixel -- so the row is latency-bound, not bandwidth-bound.
    -> list of {name, us, algorithmic_bytes, GB/s, frac_of_hbm_peak, limiter}."""
    import torch
    from bacs_b200 import ops
    g = torch.Generator(device=dev).manual_seed(5)
    B, H, W = shape
    px = B * H * W
    target = torch.randint(0, K, (B, H, W), device=dev, generator=g, dtype=torch.int64)
    target[:, :8] = 255                                                # ignored border
    preds = torch.randint(0, K, (B, H, W), device=dev, generator=g, dtype=torch.int64)
    blocky = torch.randint(0, K, (B, H // 64, W // 64), device=dev, generator=g, dtype=torch.int64)
    blocky = blocky.repeat_interleave(64, 1).repeat_interleave(64, 2).contiguous()
    noisy = torch.where(torch.rand(B, H, W, device=dev, generator=g) < 0.1, preds, blocky)
    confmat = torch.zeros(K, K, dtype=torch.int64, device=dev)
    lut = torch.arange(256, dtype=torch.int32, device=dev)
    lut[K:] = 0
    task_lut = torch.full((256,), -1, dtype=torch.int32, device=dev)
    task_lut[1:K] = torch.arange(K - 1, dtype=torch.int32, device=dev) % 4
    out = torch.empty_like(target)
    rows = []
    for name, fn, nbytes, limiter in (
            ("confmat_accumulate [%d,%d,%d] K=%d, random classes" % (B, H, W, K),
             lambda: ops.confmat_accumulate(preds, target, K, confmat), 16 * px,
             "HBM (one shared-memory atomic per distinct bin of a warp instruction: ballot aggregation)"),
            ("confmat_accumulate [%d,%d,%d] K=%d, blocky map with 10%% errors" % (B, H, W, K),
             lambda: ops.confmat_accumulate(noisy, blocky, K, confmat), 16 * px, "HBM"),
            ("label_remap [%d,%d,%d]" % (B, H, W), lambda: ops.label_remap(target, lut, 0, out=out), 24 * px,
             "HBM (two passes: the label set must be known before a pixel can be mapped)"),
            ("label_downsample_task [%d,%d,%d] -> /16" % (B, H, W),
             lambda: ops.label_downsample_task(target, H // 16, W // 16, task_lut, 4), (32 + 13) * (px // 256),
             "latency: one 32-byte sector per low-res pixel + block scan; 1/256 of the labels are read")):
        ms = timed_fn(fn, steps, 3)
        gbs = nbytes / (ms * 1e-3) / 1e9
        rows.append({"name": name, "us": ms * 1e3, "algorithmic_bytes": nbytes, "GB/s": gbs,
                     "frac_of_hbm_peak": gbs / peak, "limiter": limiter})
    # the optional per-class prototype family (SURVEY 8f-4) at the ADE20K shape: tensor-core distance, per-class sums
    Bc, Dc, hc, wc, Kc = 24, 512, 32, 32, 150
    f = torch.randn(Bc, Dc, hc, wc, device=dev, generator=g).to(torch.bfloat16)
    c = torch.randn(Kc, Dc, device=dev, generator=g).to(torch.bfloat16)
    lab = torch.randint(0, Kc + 1, (Bc, hc, wc), device=dev, generator=g, dtype=torch.int64)
    ms = timed_fn(lambda: ops.class_distance(f, c), steps, 3)
    flop = 2.0 * Bc * hc * wc * 160 * Dc
    rows.append({"name": "class_distance [%d,%d,%d,%d] x %d classes (tcgen05, bf16)" % (Bc, Dc, hc, wc, Kc), "us": ms * 1e3,
                 "algorithmic_bytes": int(f.numel() * 2 + Bc * Kc * hc * wc * 4), "TFLOP/s": flop / (ms * 1e-3) / 1e12,
                 "limiter": "prototype fill from L2 + 192 tiles on 148 SMs (a 4 GFLOP product)"})
    ms = timed_fn(lambda: ops.class_sums(f, lab, Kc + 1), steps, 3)
    rows.append({"name": "class_sums [%d,%d,%d,%d] into %d classes" % (Bc, Dc, hc, wc, Kc + 1), "us": ms * 1e3,
                 "algorithmic_bytes": int(f.numel() * 2), "GB/s": f.numel() * 2 / (ms * 1e-3) / 1e9,
                 "limiter": "shared-memory table update per pixel + per-class warp sums"})
    del f, c, lab
    # BASELINE.json configs[3]: the per-pixel loss at the ADE20K 100-50 shape (K = 151, B = 24, 512 x 512, bf16 logits)
    from bacs_b200 import _cabi, synth
    cfg = synth.CONFIGS["ade100-50"]
    logits = torch.randn(cfg.B, cfg.K, cfg.H, cfg.W, device=dev, generator=g).to(torch.bfloat16)
    mask = synth.make_labels(cfg, torch.Generator().manual_seed(1), classes=list(range(1, cfg.K))).to(dev)
    z = torch.randn(cfg.B, cfg.T, cfg.h, cfg.w, device=dev, generator=g)
    kw = dict(want_grad=True, z=z, want_distill_mask=True, old_cl=cfg.old_cl, focal_head=cfg.T - 1)
    variant = ops.pixel_loss(logits, mask, _cabi.PIX_WEIGHTED_CE, **kw)["variant"]
    ms = timed_fn(lambda: ops.pixel_loss(logits, mask, _cabi.PIX_WEIGHTED_CE, **kw), steps, 3)
    nbytes = cfg.B * cfg.H * cfg.W * (2 * cfg.K * 2 + 17)
    gbs = nbytes / (ms * 1e-3) / 1e9
    rows.append({"name": "pixel_loss ade100-50 [%d,%d,%d,%d] bf16 (variant %d: one pass, channel column in registers)"
                         % (cfg.B, cfg.K, cfg.H, cfg.W, variant), "us": ms * 1e3, "algorithmic_bytes": nbytes,
                 "GB/s": gbs, "frac_of_hbm_peak": gbs / peak,
                 "limiter": "instruction issue (about 40 instructions per channel and pixel pair, two ex2 per logit) "
                            "at 16 warps per SM; DRAM traffic equals the algorithmic bytes"})
    del logits, mask, z
    return rows


def run_integer_rows(args, dev, world, rank):
    """bench.py --config cityscapes_eval: the integer rows alone (BASELINE.json configs[4], SURVEY 8a rows 0, 3, 14)."""
    import torch

    def timed(fn, steps, warmup):
        for _ in range(warmup):
            fn()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            fn()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / steps
    peak, peak_src = peaks()
    rows = integer_rows(timed, dev, peak, shape=(8, 1024, 2048), K=20, steps=args.steps)
    cm = rows[1]                      # the evaluation-like input
    px = 8 * 1024 * 2048
    if rank == 0:
        print(json.dumps({"metric": "confusion-matrix pixels/sec (Cityscapes 1024x2048 evaluation)", "value": px / (cm["us"] * 1e-6),
                          "unit": UNIT, "n_gpus": 1, "steps": args.steps, "warmup": 3, "ms_per_step": cm["us"] * 1e-3,
                          "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "int64",
                          "data": "synthetic", "config": {"workload": "cityscapes_eval: " + cm["name"],
                                                          "l2_policy": "inputs larger than L2 (268 MB per launch)"},
                          "roofline": {"bound": "hbm", "kernel": "confmat_kernel", "achieved": cm["GB/s"], "peak": peak,
                                       "unit": "GB/s", "frac": cm["frac_of_hbm_peak"], "traffic": None,
                                       "peak_source": peak_src},
                          "other_kernels": rows, "gpu_launches": (args.steps + 3) * len(rows)}), flush=True)


def verify_ranks(loss_fn, leaves, batch, cfg, dev, world, rank):
    """One UN-TIMED training-step prototype exchange at N > 1, checked three ways (the reference never synchronises
    prototypes, loss/prototypes.py:157-163, so the added behaviour has to be proven): (i) this rank's prototypes and
    counts after the product path (NVLink peer exchange fused with the update, or the packed NCCL all-reduce) equal,
    bit for bit, the update applied to a plain NCCL all-reduce of the same per-rank sums; (ii) every rank holds the
    same bits; (iii) no peer exchange timed out.  Raises on any mismatch."""
    import torch
    import torch.distributed as dist
    from bacs_b200 import ops
    from bacs_b200.distributed import check_peer_errors, peer_reducer
    P = loss_fn._prototypes
    proto0, count0 = P._prototypes_tensors.clone(), P._count_features.clone()
    pen, mask = leaves["pen"].detach(), (batch["main"][1] if isinstance(batch, dict) else batch[1])
    T, D = proto0.shape
    drop = os.environ.get("BACS_BENCH_DROP_RANK")                   # fault injection: this rank skips the exchange
    if drop is None or int(drop) != rank:
        P.update_feats_prototypes(pen, mask)
    torch.cuda.synchronize()
    check_peer_errors()                                               # raises on a timed-out NVLink exchange
    got_p, got_c = P._prototypes_tensors.clone(), P._count_features.clone()
    # reference sum: per-rank sums (same kernels, per-channel mode) through ONE plain NCCL all-reduce
    lut = P._device_task_lut(dev, T)
    B, _, h, w = pen.shape
    task, rnk, n_bt, _ = ops.label_downsample_task(mask, h, w, lut, T)
    packed = torch.empty(T * D + T, dtype=torch.float64, device=dev)
    sums, counts = ops.proto_accumulate(pen, task, rnk, n_bt, T, 1, out=packed)
    dist.all_reduce(packed, op=dist.ReduceOp.SUM)
    want_p, want_c = proto0.clone(), count0.clone()
    ops.proto_update(want_p, want_c, sums, counts)
    torch.cuda.synchronize()
    ok = torch.equal(got_p, want_p) and torch.equal(got_c, want_c)
    gathered = [torch.empty_like(got_p) for _ in range(world)]
    dist.all_gather(gathered, got_p)
    same = all(torch.equal(g, gathered[0]) for g in gathered)
    flag = torch.tensor([int(ok), int(same)], device=dev)
    dist.all_reduce(flag, op=dist.ReduceOp.MIN)
    P._prototypes_tensors.copy_(proto0)
    P._count_features.copy_(count0)
    P.refresh_ready()
    if int(flag[0]) != 1 or int(flag[1]) != 1:
        raise SystemExit("bench.py: N=%d prototype exchange FAILED verification (matches NCCL sum: %s, identical "
                         "across ranks: %s)" % (world, bool(flag[0]), bool(flag[1])))
    red = peer_reducer(T * D + T, dev)
    return "peer_symm" if red is not None else "nccl_packed"


def main():
    args = parse()
    if args.impl == "reference":
        return run_reference(args)

    import numpy as np
    import torch
    import torch.distributed as dist
    from bacs_b200 import _cabi, ops, synth

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device (the BACS loss path has no CPU fallback; use --impl reference)")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    lib = _cabi.load()
    dtype = {"bf16": torch.bfloat16, "fp32": torch.float32, "fp16": torch.float16}[args.dtype]
    if args.config == "cityscapes_eval":
        return run_integer_rows(args, dev, world, rank)
    cfg = synth.CONFIGS[args.config]
    inp = synth.make_step_inputs(cfg, seed=rank, dtype=dtype)
    # multi-GPU runs use the decomposable per-channel prototype sums (SURVEY 8e)
    loss_fn, net, batch, leaves = synth.build_bacs_step(cfg, inp, device=dev, exact_prototypes=(world == 1))
    protos0 = loss_fn._prototypes._prototypes_tensors.clone()
    counts0 = loss_fn._prototypes._count_features.clone()
    pixels = cfg.B * cfg.H * cfg.W
    last = {}                         # the outputs of the latest step (the graph's own buffers once it is captured)

    def step():
        for v in leaves.values():
            v.grad = None
        loss, preds = loss_fn.compute_loss(batch, net, train=True)
        loss.backward()
        last["loss"], last["preds"] = loss.detach(), preds     # detached: the autograd graph must not outlive the step
        return loss, preds

    def snapshot():
        """host copies of what the latest step returned to its caller"""
        torch.cuda.synchronize()
        out = {"loss": last["loss"], "preds": last["preds"], "prototypes": loss_fn.prototypes,
               "prototype_counts": loss_fn._prototypes._count_features}
        out.update(("grad_" + k, v.grad) for k, v in leaves.items() if v.grad is not None)
        return {k: host_sample(v) for k, v in out.items()}

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps, warmup):
        for _ in range(warmup):
            fn()
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            fn()
        e1.record()
        barrier()
        ms = e0.elapsed_time(e1)
        if world > 1:
            t = torch.tensor([ms], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t)
        return ms / steps

    collective, nranks_checked = "none (single process)", 1
    if world > 1:
        # data-parallel replicas start from identical prototype state (the per-rank seed only varies the batch)
        dist.broadcast(loss_fn._prototypes._prototypes_tensors, 0)
        dist.broadcast(loss_fn._prototypes._count_features, 0)
        loss_fn._prototypes.refresh_ready()
        collective = verify_ranks(loss_fn, leaves, batch, cfg, dev, world, rank)
        nranks_checked = world

    sampler = ClockSampler(local_rank)
    sampler.start()

    # ---- the headline: K steps through the public class interface, inputs resident in HBM
    n0 = lib.bacs_launch_count()
    step()
    launches_per_step = int(lib.bacs_launch_count() - n0)
    ms_eager = timed(step, args.steps, max(args.warmup, 3))
    # taken after each timed window, before anything below runs the loss again and moves the prototypes on
    dumped = snapshot() if args.dump_outputs and rank == 0 else None

    # ---- the same step captured once in a CUDA graph (the step never synchronises with the host)
    ms_graph = None
    if not args.no_graph:
        try:
            side = torch.cuda.Stream()
            side.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(side):
                step()
            torch.cuda.current_stream().wait_stream(side)
            torch.cuda.synchronize()
            graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(graph):
                step()
            ms_graph = timed(graph.replay, args.steps, max(args.warmup, 3))
            if dumped is not None:
                dumped = snapshot()
        except Exception as exc:                                  # noqa: BLE001
            sys.stderr.write("bench.py: CUDA-graph replay unavailable: %r\n" % (exc,))
            ms_graph = None
    ms_step = ms_eager if ms_graph is None else min(ms_eager, ms_graph)
    value = world * pixels / (ms_step * 1e-3)
    if dumped is not None:
        os.makedirs(args.dump_outputs, exist_ok=True)
        for name, arr in dumped.items():
            np.save(os.path.join(args.dump_outputs, name + ".npy"), arr)

    # ---- dominant kernel (fused pixel kernel) timed alone, back to back, on its launch stream
    es = torch.finfo(dtype).bits // 8
    with torch.no_grad():
        P = loss_fn._prototypes
        w, b = loss_fn._stack_heads(net.seen_fg_network, cfg.T)
        z = ops.seen_logits(leaves["pen"].detach(), P._prototypes_tensors, w, b)
        lg, mk = leaves["logits"].detach(), batch["main"][1] if isinstance(batch, dict) else batch[1]

        variant = {}

        def pixel_only():
            variant["v"] = ops.pixel_loss(lg, mk, _cabi.PIX_WEIGHTED_CE, want_grad=True, z=z, want_distill_mask=True,
                                          focal_head=cfg.T - 1, old_cl=cfg.old_cl)["variant"]
        ms_pix = timed(pixel_only, args.steps, max(args.warmup, 3))
    kernel_name = {2: "pixel_wce_kernel", 1: "pixel_fast_kernel", 0: "pixel_loss_kernel (shared-memory tiles)",
                   4: "pixel_stream_stats_kernel + pixel_stream_grad_kernel"}.get(
        variant.get("v"), "pixel kernel")
    alg_bytes = pixels * (2 * cfg.K * es + 8 + 8 + 1) + z.numel() * 4
    peak, peak_src = peaks()
    achieved = alg_bytes / (ms_pix * 1e-3) / 1e9
    traffic = None
    tpath = os.path.join(ROOT, "profiles", "r01_pixel_wce_traffic.json")
    if os.path.exists(tpath) and args.config == "voc15-1_b24" and args.dtype == "bf16":
        with open(tpath) as f:
            traffic = json.load(f).get("traffic_bytes_per_launch")   # dram read + write of one launch (ncu --set full)
    roofline = {"bound": "hbm", "kernel": kernel_name + " (weighted CE + focal + argmax + distill mask + dlogits)",
                "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": traffic,
                "peak_source": peak_src, "algorithmic_bytes_per_launch": alg_bytes, "ms_per_launch": ms_pix,
                "share_of_step": ms_pix / ms_step}

    # ---- the other kernels of the step, each timed alone on the step's own inputs (time-dominant first)
    kernels = [{"name": kernel_name, "us": ms_pix * 1e3}]
    with torch.no_grad():
        dmask = ops.pixel_loss(lg, mk, _cabi.PIX_WEIGHTED_CE, want_grad=False, z=z, want_distill_mask=True,
                               focal_head=cfg.T - 1, old_cl=cfg.old_cl)["distill_mask"]
        old_att = loss_fn.prev_model(batch["main"][0] if isinstance(batch, dict) else batch[0],
                                     return_penultimate=True, return_attentions=True)[2][-1]
        new_att = leaves["new_att"].detach()
        coef = 0.25 / (cfg.B * cfg.A * cfg.H)
        tc = ops.distill_kernel_variant(new_att, (cfg.H, cfg.W))
        ms_dist = timed(lambda: ops.teacher_distill(old_att, new_att, dmask, (cfg.H, cfg.W), coef, True, want_scaled=True),
                        args.steps, 3)
        kernels.append({"name": "teacher_distill (%s)" % ("distill_tc_kernel: tcgen05 split-tf32 GEMM form + finish" if tc
                                                         else "distill_kernel: packed fp32"), "us": ms_dist * 1e3})
        pen_d = leaves["pen"].detach()
        lut = P._device_task_lut(dev, cfg.T)
        pr, ct = P._prototypes_tensors.clone(), P._count_features.clone()

        def proto_chain():
            task, rnk, n_bt, _ = ops.label_downsample_task(mk, cfg.h, cfg.w, lut, cfg.T)
            if world == 1:      # what Prototypes.update_feats_prototypes launches in a single process
                ops.proto_accumulate_update(pen_d, task, rnk, n_bt, 0, pr, ct)
            else:
                sums, counts = ops.proto_accumulate(pen_d, task, rnk, n_bt, cfg.T, 1)
                ops.proto_update(pr, ct, sums, counts)

        def graph_timed(fn):    # three small launches: replayed from a graph so that the host does not pace them
            try:
                fn()
                torch.cuda.synchronize()
                gk = torch.cuda.CUDAGraph()
                with torch.cuda.graph(gk):
                    fn()
                return timed(gk.replay, args.steps, 3)
            except Exception as exc:                              # noqa: BLE001
                sys.stderr.write("bench.py: graph timing of the prototype chain unavailable: %r\n" % (exc,))
                return timed(fn, args.steps, 3)
        ms_proto = graph_timed(proto_chain)
        kernels.append({"name": "prototype chain (label_downsample_task + proto_accumulate + finalize/update)",
                        "us": ms_proto * 1e3})
        ms_seen = timed(lambda: ops.seen_logits(pen_d, P._prototypes_tensors, w, b), args.steps, 3)
        kernels.append({"name": "seen_logits_kernel", "us": ms_seen * 1e3})
    for k in kernels:
        k["share_of_step"] = k["us"] / (ms_step * 1e3)
    kernels.sort(key=lambda k: -k["us"])
    # whole-step roofline, SURVEY 8d: 2 K s_l + 16 + (D s_f + 3 A s_f + 16 T) / 256 bytes per main-batch pixel
    step_bytes = pixels * (2 * cfg.K * es + 16 + (cfg.D * es + 3 * cfg.A * es + 16 * cfg.T) / 256.0)
    roofline["step"] = {"bytes": step_bytes, "bytes_per_pixel": step_bytes / pixels, "ms_per_step": ms_step,
                        "achieved": step_bytes / (ms_step * 1e-3) / 1e9, "frac": step_bytes / (ms_step * 1e-3) / 1e9 / peak,
                        "target_frac": 0.70}
    other = integer_rows(timed, dev, peak) if world == 1 else None

    # ---- end to end: host (pinned) inputs -> device -> step -> loss back on the host
    def run_e2e(lfn, nt, bt0, host, sem_key=None):
        """Every step's inputs cross PCIe inside the timed region (two device-side input sets: the copy stream uploads
        step i+1 while the compute stream runs step i) and the loss of every step is read back.  Labels travel as
        uint8, the way the data loader holds them, and are widened on the device by preprocess_batch
        (loss/base_loss.py:274-282 runs after Lightning's transfer as well)."""
        h2d = sum(t.numel() * t.element_size() for t in host.values())
        img = bt0["main"][0] if isinstance(bt0, dict) else bt0[0]
        loss_host = torch.empty((), dtype=torch.float32).pin_memory()
        copy_stream = torch.cuda.Stream()
        dbuf = [{k: torch.empty_like(t, device=dev) for k, t in host.items()} for _ in range(2)]
        uploaded = [torch.cuda.Event() for _ in range(2)]
        consumed = [torch.cuda.Event() for _ in range(2)]
        state = {"i": 0, "primed": False}

        def upload(slot):
            with torch.cuda.stream(copy_stream):
                copy_stream.wait_event(consumed[slot])            # the step that last used this slot is done
                for k, t in host.items():
                    dbuf[slot][k].copy_(t, non_blocking=True)
                uploaded[slot].record(copy_stream)

        def e2e_step():
            cur = torch.cuda.current_stream()
            slot = state["i"] & 1
            if not state["primed"]:
                upload(slot)
                state["primed"] = True
            upload(slot ^ 1)                                       # next step's inputs, overlapping this step
            cur.wait_event(uploaded[slot])
            d = dbuf[slot]
            nat = d["new_att"].detach().requires_grad_(True)
            if sem_key is None:
                lgt = d["logits"].detach().requires_grad_(True)
                nt.register(img, lgt, d["pen"], [nat])
                lfn.prev_model.register(img, d["logits"], d["pen"], [d["old_att"]])
            else:
                sem = d[sem_key].detach().requires_grad_(True)
                nt.register(img, sem, d["pen"], [nat])
                nt.register_sem(img, sem)
                lfn.prev_model.register(img, sem.detach(), d["pen"], [d["old_att"]])
            bt = lfn.preprocess_batch([img, d["mask"]])            # uint8 -> int64 on the device
            if isinstance(bt0, dict):
                bt = dict(bt0, main=bt)
            loss, _ = lfn.compute_loss(bt, nt, train=True)
            loss.backward()
            loss_host.copy_(loss.detach(), non_blocking=True)
            consumed[slot].record(cur)
            state["i"] += 1
            if state["i"] >= 2:
                consumed[slot ^ 1].synchronize()                   # bound the queue: at most two steps in flight
        for ev in consumed:
            ev.record(torch.cuda.current_stream())
        ms = timed(e2e_step, max(3, min(args.steps, 20)), 3)
        torch.cuda.synchronize()
        return {"value": world * pixels / (ms * 1e-3), "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": 4,
                "ms_per_step": ms, "labels": "uint8 on the wire, widened to int64 on the device"}

    e2e = None
    if not args.no_e2e:
        host = {k: getattr(inp, k).pin_memory() for k in ("logits", "pen", "old_att", "new_att")}
        host["mask"] = inp.mask.to(torch.uint8).pin_memory()
        e2e = run_e2e(loss_fn, net, batch, host)
        img0 = batch["main"][0] if isinstance(batch, dict) else batch[0]
        net.register(img0, leaves["logits"], leaves["pen"], [leaves["new_att"]])
        loss_fn.prev_model.register(img0, inp.logits.to(dev), inp.pen.to(dev), [inp.old_att.to(dev)])

    # ---- extra (not the headline): the opt-in fused path -- the network hands over its low-res sem_logits and the
    # x16 bilinear up-sample, the loss and the adjoint of the up-sample run in one kernel (SURVEY 8f-1)
    fused = None
    if world == 1 and not args.no_fused_lowres:
        try:
            loss2, net2, batch2, leaves2 = synth.build_bacs_step(cfg, inp, device=dev, fused_logit_upsample=True)
            gen = torch.Generator().manual_seed(7)
            sems = []
            for key, nb in (("main", cfg.B), ("buffer", cfg.Br)):
                if isinstance(batch2, dict) and key in batch2 or key == "main":
                    im = batch2[key][0] if isinstance(batch2, dict) else batch2[0]
                    sem = torch.randn(nb, cfg.K, cfg.h, cfg.w, generator=gen).to(dtype).to(dev).requires_grad_(True)
                    net2.register_sem(im, sem)
                    sems.append(sem)

            def step2():
                for v in list(leaves2.values()) + sems:
                    v.grad = None
                loss, preds = loss2.compute_loss(batch2, net2, train=True)
                loss.backward()
            ms2 = timed(step2, args.steps, max(args.warmup, 3))
            side = torch.cuda.Stream()
            side.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(side):
                step2()
            torch.cuda.current_stream().wait_stream(side)
            torch.cuda.synchronize()
            graph2 = torch.cuda.CUDAGraph()
            with torch.cuda.graph(graph2):
                step2()
            ms2g = timed(graph2.replay, args.steps, max(args.warmup, 3))
            fused = {"what": "BACSLoss(fused_logit_upsample=True): sem_logits [B,K,H/16,W/16] in, up-sample + loss + "
                             "adjoint in one kernel; no [B,K,H,W] logits or gradient exist",
                     "ms_per_step_eager": ms2, "ms_per_step_graph": ms2g,
                     "value": pixels / (min(ms2, ms2g) * 1e-3), "unit": UNIT,
                     "logit_bytes_per_step": int(sems[0].numel() * es * 2)}
            graph2 = None
            if not args.no_e2e and not isinstance(batch2, dict):
                # end to end with the low-res logits on the wire: 2 MB of sem_logits instead of 264 MB of logits
                host2 = {k: getattr(inp, k).pin_memory() for k in ("pen", "old_att", "new_att")}
                host2["sem"] = sems[0].detach().cpu().pin_memory()
                host2["mask"] = inp.mask.to(torch.uint8).pin_memory()
                fused["e2e_lowres"] = run_e2e(loss2, net2, batch2, host2, sem_key="sem")
        except Exception as exc:                                  # noqa: BLE001
            sys.stderr.write("bench.py: fused low-res timing unavailable: %r\n" % (exc,))

    sampler.stop_flag = True
    sampler.join(timeout=2)
    clocks = sampler.summary()

    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        try:
            torch.set_num_threads(max(1, len(os.sched_getaffinity(0))))
        except AttributeError:
            pass
        v, dt, sample, kind = cpu_step_time(cfg, args.cpu_sample_batch, 2, 0)
        cpu = {"value": v, "unit": UNIT, "cores": torch.get_num_threads(), "kind": kind, "sample": sample,
               "ms_per_step": dt * 1e3}

    if rank == 0:
        line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
                "warmup": max(args.warmup, 3), "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak",
                "vs_baseline": None, "dtype": args.dtype, "data": "synthetic",
                "config": {"workload": workload_name(cfg), "global_batch": world * cfg.B,
                           "parallelism": "dp%d" % world, "collective": collective,
                           "l2_policy": "inputs larger than L2 (logits %.0f MB per step, L2 126 MB)"
                                        % (cfg.B * cfg.K * cfg.H * cfg.W * es / 1e6),
                           "timed_path": "cuda-graph replay of BACSLoss.compute_loss+backward" if ms_step == ms_graph
                                         else "BACSLoss.compute_loss+backward (eager)"},
                "ms_per_step_eager": ms_eager, "ms_per_step_graph": ms_graph,
                "gpu_launches": launches_per_step * args.steps, "gpu_launches_per_step": launches_per_step,
                "nranks_checked": nranks_checked, "roofline": roofline, "kernels": kernels, "other_kernels": other,
                "cpu_baseline": cpu, "e2e": e2e, "clocks": clocks, "fused_lowres": fused}
        print(json.dumps(line), flush=True)
    if world > 1:
        # A captured graph that holds NCCL kernels must be gone before the communicator is torn down; the
        # teardown itself is skipped (it can block on a communicator that was used under capture) and the
        # ranks leave together after a final barrier.
        graph = None
        torch.cuda.synchronize()
        dist.barrier()
        torch.cuda.synchronize()
        sys.stdout.flush()
        sys.stderr.flush()
        os._exit(0)


if __name__ == "__main__":
    main()
