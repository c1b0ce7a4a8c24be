"""Times the cost of exact-mode prototypes across data-parallel ranks (exact_prototypes_across_ranks=True) against the
default per-channel sums of runs with N > 1, at bench.py's VOC headline shape (B = 24 per GPU, 512 x 512, D = 512 bf16
features, T = 6).  Run with N >= 2 GPUs:

  python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 tools/proto_global_view_time.py

Two things are timed, with the option off and on, alternating window by window in the same process:
  * the prototype chain alone: task down-sample + Prototypes.update_feats_prototypes (off: per-channel accumulate and
    the sums exchange; on: count exchange, global-view accumulate and the sums exchange);
  * the whole compute_loss + backward step, replayed from a CUDA graph.
CUDA events around back-to-back calls after a warm-up; each number is the median of --repeats windows of --iters calls,
with the spread (min..max) beside it.  Rank 0 prints the card's name and power limit with the numbers."""
import argparse
import json
import os
import subprocess
import sys

import torch
import torch.distributed as dist

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from bacs_b200 import synth  # noqa: E402


def card():
    name = torch.cuda.get_device_name()
    try:
        limit = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i",
                                str(torch.cuda.current_device())], capture_output=True, text=True,
                               timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        limit = "unknown"
    return name, limit or "unknown"


def window(fn, iters):
    dist.barrier()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / iters * 1000.0


def build(rank, on):
    cfg = synth.CONFIGS["voc15-1_b24"]
    inp = synth.make_step_inputs(cfg, seed=rank, dtype=torch.bfloat16)
    loss_fn, net, batch, leaves = synth.build_bacs_step(cfg, inp, device="cuda", exact_prototypes=on,
                                                        exact_prototypes_across_ranks=on)
    P = loss_fn._prototypes
    mask = batch[1] if isinstance(batch, (list, tuple)) else batch["main"][1]
    pen = leaves["pen"].detach()

    def chain():
        P.update_feats_prototypes(pen, mask)

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
    return {"chain": chain, "step_graph": graph.replay, "keep": (loss_fn, net, batch, leaves, graph)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=50)
    ap.add_argument("--repeats", type=int, default=7)
    args = ap.parse_args()
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if world < 2 or not torch.cuda.is_available():
        sys.exit("proto_global_view_time.py: needs >= 2 GPUs under torch.distributed.run")
    rank, local = int(os.environ["RANK"]), int(os.environ["LOCAL_RANK"])
    torch.cuda.set_device(local)
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    runs = {False: build(rank, False), True: build(rank, True)}
    res = {(on, k): [] for on in runs for k in ("chain", "step_graph")}
    for k in ("chain", "step_graph"):
        for on in runs:
            for _ in range(3):
                runs[on][k]()
        for _ in range(args.repeats):
            for on in runs:
                res[(on, k)].append(window(runs[on][k], args.iters))
    from bacs_b200.distributed import check_peer_errors
    check_peer_errors()
    if rank == 0:
        name, limit = card()
        print("device: %s, power limit %s, N = %d" % (name, limit, world))
        rows = []
        for (on, k), v in res.items():
            v.sort()
            rows.append({"exact_across_ranks": on, "what": k, "median_us": v[len(v) // 2], "min_us": v[0],
                         "max_us": v[-1]})
            print("%-10s exact_across_ranks=%-5s %8.1f us [%.1f..%.1f]" % (k, on, v[len(v) // 2], v[0], v[-1]))
        print(json.dumps({"device": name, "power_limit": limit, "world": world, "rows": rows}))
    sys.stdout.flush()
    dist.barrier()
    os._exit(0)


if __name__ == "__main__":
    main()
