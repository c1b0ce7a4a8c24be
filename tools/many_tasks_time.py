"""Times the BACS loss step and its task-count-dependent kernels at T = 6, 32, 33, 64 and 128 tasks.

  * the whole compute_loss + backward step replayed from a CUDA graph, at the VOC headline shape (B=24, 512x512,
    D=512, A=256, bf16 features, bg_weighted_ce on).  A run with T tasks has K = 15 + T classes (16 base classes and
    one per later step), so the pixel loss grows with T as well: K = 21 at T = 6 is bench.py's headline;
  * the seen heads alone: seen_logits_heads (T <= 32, what the step runs there) and seen_logits_many (every T) on the
    step's [24,512,32,32] bf16 features;
  * the prototype chain alone: label_downsample_task + proto_accumulate_update (exact mode), one-hot GEMM path.

The kernel-alone numbers are L2-warm: the calls run back to back on the same 25 MB of features, which stay in the
126 MB L2, so every read -- the first 32-head chunk's included -- is served from L2.

CUDA events around back-to-back calls after a warm-up; each number is the median of --repeats windows of --iters
calls, and the spread (min..max) is printed beside it.  The card's name and power limit are printed with the numbers.

    python tools/many_tasks_time.py [--iters N] [--repeats R] [--tasks 6,32,33,64,128]"""
import argparse
import json
import os
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from bacs_b200 import ops, synth  # noqa: E402


def card():
    name = torch.cuda.get_device_name()
    try:
        limit = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i",
                                str(torch.cuda.current_device())], capture_output=True, text=True,
                               timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        limit = "unknown"
    return name, limit or "unknown"


def timeit(fn, iters, repeats, warmup=3):
    """-> (median, min, max) microseconds per call over `repeats` windows of `iters` calls"""
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    out = []
    for _ in range(repeats):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(iters):
            fn()
        e1.record()
        torch.cuda.synchronize()
        out.append(e0.elapsed_time(e1) / iters * 1000.0)
    out.sort()
    return out[len(out) // 2], out[0], out[-1]


def config(T):
    return synth.StepConfig("voc_shape_T%d" % T, B=24, K=15 + T, old_cl=14 + T, T=T, H=512, W=512, D=512, A=256,
                            initial_classes=16, increment=1)


def time_step(T, iters, repeats):
    cfg = config(T)
    inp = synth.make_step_inputs(cfg, seed=T, dtype=torch.bfloat16)
    loss_fn, net, batch, leaves = synth.build_bacs_step(cfg, inp, device="cuda")
    protos0 = loss_fn._prototypes._prototypes_tensors.clone()

    def step():
        for v in leaves.values():
            v.grad = None
        loss, _ = loss_fn.compute_loss(batch, net, train=True)
        loss.backward()

    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        step()
    torch.cuda.current_stream().wait_stream(side)
    torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        step()
    t = timeit(graph.replay, iters, repeats)
    loss_fn._prototypes._prototypes_tensors.copy_(protos0)

    # the kernels alone, on the step's own tensors
    pen = leaves["pen"].detach()
    protos = loss_fn._prototypes._prototypes_tensors
    heads = list(net.seen_fg_network.seen_not_seen_clf)
    ws = [h.conv.weight.detach() for h in heads]
    bs = [h.conv.bias.detach() for h in heads]
    gz = torch.empty(cfg.B, cfg.h, cfg.w, device="cuda")
    seen = {}
    with torch.no_grad():
        if T <= 32:
            seen["seen_logits_heads"] = timeit(lambda: ops.seen_logits_heads(pen, protos, ws, bs, zero_out=gz),
                                               iters, repeats)
        seen["seen_logits_many"] = timeit(lambda: ops.seen_logits_many(pen, protos, ws, bs, zero_out=gz), iters,
                                          repeats)
        P = loss_fn._prototypes
        mask = batch[1] if isinstance(batch, (list, tuple)) else batch["main"][1]
        lut = P._device_task_lut(pen.device, T)
        count = P._count_features.clone()
        proto = protos.clone()

        def chain():
            task, rank, n_bt, _ = ops.label_downsample_task(mask, cfg.h, cfg.w, lut, T)
            ops.proto_accumulate_update(pen, task, rank, n_bt, 0, proto, count)
        seen["prototype_chain"] = timeit(chain, iters, repeats)
    del loss_fn, net, batch, leaves, graph
    torch.cuda.empty_cache()
    return t, seen


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=50)
    ap.add_argument("--repeats", type=int, default=5)
    ap.add_argument("--tasks", default="6,32,33,64,128")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("many_tasks_time.py: needs a CUDA device")
    name, limit = card()
    print("device: %s, power limit %s" % (name, limit))
    rows = []
    for T in [int(x) for x in args.tasks.split(",")]:
        step, parts = time_step(T, args.iters, args.repeats)
        row = {"T": T, "K": 15 + T, "step_graph_us": step}
        row.update({k + "_us": v for k, v in parts.items()})
        rows.append(row)
        print("T=%3d K=%3d  step (graph) %8.1f us [%.1f..%.1f]" % (T, 15 + T, *step))
        for k, v in parts.items():
            print("        %-18s %8.1f us [%.1f..%.1f]" % (k, *v))
        sys.stdout.flush()
    print(json.dumps({"device": name, "power_limit": limit, "rows": rows}))


if __name__ == "__main__":
    main()
