#!/usr/bin/env python
"""What the host can feed: N ranks copy the bench's per-step input (118.5 MB of float32 pixels, pinned) to their GPUs at the
same time -- the ceiling of bench.py's `e2e` (which moves exactly these bytes per step) at N GPUs.  With and without
binding each rank to the CPUs / memory node next to its GPU.

    torchrun --nproc-per-node 8 tools/h2d_ceiling.py [--out DIR]   -> JSON line (+ DIR/h2d_ceiling_r02_n8.json)
"""
import argparse
import json
import os
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch  # noqa: E402
import torch.distributed as dist  # noqa: E402
import bench  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", metavar="DIR", help="directory for the JSON report (none written without it)")
    args = ap.parse_args()
    rank, world = int(os.environ.get("RANK", 0)), int(os.environ.get("WORLD_SIZE", 1))
    local = int(os.environ.get("LOCAL_RANK", 0))
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("gloo")
    out = {}
    for bind in (False, True):
        cpus = bench.bind_to_gpu_numa(local) if bind else None
        host = torch.empty(bench.H2D_BYTES // 4, dtype=torch.float32).pin_memory()
        host.uniform_()                                  # first touch on the (possibly re-bound) node
        dev = torch.empty_like(host, device="cuda")
        for _ in range(3):
            dev.copy_(host, non_blocking=True)
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        n = 30
        t0 = time.perf_counter()
        for _ in range(n):
            dev.copy_(host, non_blocking=True)
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        gbs = torch.tensor([bench.H2D_BYTES * n / dt / 1e9])
        if world > 1:
            all_ = [torch.zeros(1) for _ in range(world)]
            dist.all_gather(all_, gbs)
            per = [float(x) for x in all_]
        else:
            per = [float(gbs)]
        out["numa_bound" if bind else "unbound"] = {
            "per_rank_GBps": [round(x, 2) for x in per], "aggregate_GBps": round(sum(per), 1),
            "images_per_s_ceiling": round(sum(per) * 1e9 / bench.H2D_BYTES * bench.BATCH),
            "cpus_rank0": (cpus[:8] if cpus else None)}
        del host, dev
    if rank == 0:
        out["n_gpus"] = world
        out["bytes_per_step_per_gpu"] = bench.H2D_BYTES
        print(json.dumps(out), flush=True)
        if args.out:
            os.makedirs(args.out, exist_ok=True)
            with open(os.path.join(args.out, f"h2d_ceiling_r02_n{world}.json"), "w") as f:
                json.dump(out, f, indent=1)
    if world > 1:
        dist.barrier()


if __name__ == "__main__":
    main()
