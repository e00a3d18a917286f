#!/usr/bin/env python
"""Where does the time of ONE captured phase-1 step go?  The step is a single CUDA graph (four streams + the NCCL comm
stream), so it cannot be timed call by call; with A3D_TIMELINE=1 the schedule enqueues `a3d_stamp` marks (one-thread
kernels storing %globaltimer) at its segment boundaries on every stream.  This tool replays the graph, averages the marks
over the replays and prints a table; with --out DIR it also writes a Chrome trace per rank
(DIR/step_timeline_r02_n<N>[_rank<r>].json, as kept under profiles/).

    python tools/step_timeline.py [--out DIR]                     # 1 GPU
    torchrun --nproc-per-node 8 tools/step_timeline.py            # data parallel
"""
import argparse
import json
import os
import sys

os.environ["A3D_TIMELINE"] = "1"
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch  # noqa: E402
import bench  # noqa: E402
from ann3depth_b200 import models, ops  # noqa: E402
from ann3depth_b200.init import glorot_params  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", metavar="DIR", help="directory for the Chrome trace JSON (none written without it)")
    args = ap.parse_args()
    rank, world = int(os.environ.get("RANK", 0)), int(os.environ.get("WORLD_SIZE", 1))
    local = int(os.environ.get("LOCAL_RANK", 0))
    torch.cuda.set_device(local)
    dev = torch.device(f"cuda:{local}")
    ctx = models.get_context(local)
    comm = None
    if world > 1:
        import torch.distributed as dist
        from ann3depth_b200.dp import DataParallel
        dist.init_process_group("gloo")
        saved = os.dup(1); os.dup2(2, 1)
        ids = [ops.comm_unique_id() if rank == 0 else None]
        dist.broadcast_object_list(ids, src=0)
        comm = DataParallel(ctx, rank, world, ids[0])
        sys.stdout.flush(); os.dup2(saved, 1)
    images, depths = bench.synthetic_batch(rank, torch)
    op = models.msdn(images.to(dev), depths.to(dev), train=True, comm=comm)
    op.net.load_params(glorot_params(seed=1))
    for _ in range(5):
        op.run()
    step_ms = None
    if True:
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        e0.record()
        for _ in range(50):
            op.run()
        op.net.flush()
        e1.record()
        torch.cuda.synchronize()
        step_ms = e0.elapsed_time(e1) / 50
    reps, acc = 20, None
    for _ in range(reps):
        if world > 1:
            dist.barrier()
        op.run()
        marks = ctx.timeline.read()
        if acc is None:
            acc = [[lab, st, 0.0] for lab, st, _ in marks]
        for a, (_, _, us) in zip(acc, marks):
            a[2] += us / reps
    streams = {}
    for a in acc:
        streams.setdefault(a[1], len(streams))
    rows = sorted(acc, key=lambda a: a[2])
    text = [f"rank {rank}/{world}: {step_ms:.4f} ms/step over 50 back-to-back replays (stamps included); marks: mean over {reps} "
            f"graph replays (us since the first mark; stream index)"]
    for lab, st, us in rows:
        text.append(f"  {us:8.1f}  s{streams[st]}  {lab}")
    print("\n".join(text), flush=True)
    events = [{"name": lab, "ph": "i", "s": "t", "pid": rank, "tid": streams[st], "ts": us} for lab, st, us in acc]
    # segments: consecutive marks on the same stream
    by_stream = {}
    for lab, st, us in acc:
        by_stream.setdefault(st, []).append((us, lab))
    for st, lst in by_stream.items():
        lst.sort()
        for (t0, l0), (t1, l1) in zip(lst, lst[1:]):
            events.append({"name": f"{l0} -> {l1}", "ph": "X", "pid": rank, "tid": streams[st], "ts": t0, "dur": t1 - t0})
    out = {"traceEvents": events, "displayTimeUnit": "us", "marks": [{"label": l, "stream": streams[s], "us": u} for l, s, u in rows]}
    name = f"step_timeline_r02_n{world}" + (f"_rank{rank}" if world > 1 else "") + ".json"
    if args.out and rank in (0, world - 1):
        os.makedirs(args.out, exist_ok=True)
        with open(os.path.join(args.out, name), "w") as f:
            json.dump(out, f, indent=1)
    if world > 1:
        dist.barrier()
        sys.stdout.flush()
        os._exit(0)


if __name__ == "__main__":
    main()
