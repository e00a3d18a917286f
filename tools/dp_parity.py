#!/usr/bin/env python
"""Multi-GPU parity (torchrun, one rank per GPU): n ranks x batch 32 under the data-parallel step must equal ONE
replica x batch 32n in the CPU oracle (SURVEY.md 8e; the reference's asynchronous parameter servers,
src/ann3depth.py:78-92, are replaced by synchronous data parallelism).

One general-Adam (beta2 = 0.999) phase-1 step through the default DP schedule (CUDA graph, activation-gather dense
update, conv exchange), then on rank 0:
  * TF-Adam first-moment slots m = 0.1 * (mean gradient over all 32n samples) against the float64 oracle evaluated at the
    BF16 storage points -- per-parameter cosine >= 0.999 (the oracle's big-batch gradient is the mean of the per-rank
    batch gradients: the loss is a batch mean, src/models.py:272, and no op couples samples);
  * after `gather_master`, i.e. also for the row/slice-sharded optimizer state other ranks own;
  * every rank holds bit-identical bf16 weight mirrors AND bit-identical f32 biases (the kernels read biases from the f32
    master), before and after a second step.
Prints a JSON summary; with --out DIR it also writes DIR/dp_parity_r02_n<N>.json (as kept under profiles/).
Run: torchrun --nproc-per-node N tools/dp_parity.py [--out DIR]
"""
import argparse
import json
import os
import sys

import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench  # noqa: E402
from ann3depth_b200 import models, ops  # noqa: E402
from ann3depth_b200.dp import DataParallel  # noqa: E402


def all_equal(t, world):
    """True when every rank holds the same tensor bits."""
    mine = t.detach().cpu().contiguous()
    if mine.dtype in (torch.int16, torch.bfloat16):      # gloo has no 16-bit types
        mine = mine.view(torch.int16).to(torch.int32)
    ref = mine.clone()
    dist.broadcast(ref, src=0)
    flags = [None] * world
    dist.all_gather_object(flags, bool(torch.equal(mine, ref)))
    return all(flags)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", metavar="DIR", help="directory for the full JSON report (none written without it)")
    args = ap.parse_args()
    rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
    torch.cuda.set_device(local)
    dev = torch.device(f"cuda:{local}")
    dist.init_process_group("gloo")
    ctx = models.get_context(local)
    saved = os.dup(1); os.dup2(2, 1)
    ids = [ops.comm_unique_id() if rank == 0 else None]
    dist.broadcast_object_list(ids, src=0)
    comm = DataParallel(ctx, rank, world, ids[0])
    sys.stdout.flush(); os.dup2(saved, 1)

    from oracle import msdn as OM                        # checker only (this is a test tool, not the product path)
    B = bench.BATCH
    images, depths = bench.synthetic_batch(rank, torch)
    mask = (torch.rand(B, 4096, generator=torch.Generator().manual_seed(2 + rank)) < 0.5).float()
    p = OM.init_params(1, torch.float32, bias_range=0.05)
    p["coarse/dense/dense_1/bias"] += 1.0
    p["fine/third/bias"] += 1.0

    op = models.msdn(images.to(dev), depths.to(dev), train=True, comm=comm, beta2=0.999)
    net = op.net
    net.load_params(p)
    net.set_dropout_mask(mask.to(dev))
    op.run()                                             # graph path, as bench.py runs it
    net.flush()                                          # rows updated by peers are otherwise fetched by the next step
    torch.cuda.synchronize()
    report = {"n_gpus": world, "batch_per_gpu": B}
    report["identical_bf16_weights_after_step_1"] = all_equal(net.arena.wb.view(torch.int16), world)
    bias_ok = True
    for s in net.arena.specs.values():
        if s.kind == "bias":
            bias_ok &= all_equal(net.arena.w[s.offset:s.offset + s.numel], world)
    report["identical_f32_biases_after_step_1"] = bias_ok
    with torch.cuda.stream(comm.stream):
        comm.gather_master(net)
    torch.cuda.synchronize()
    report["identical_f32_master_after_gather"] = all_equal(net.arena.w, world)
    got_m = net.arena.export_tf(net.arena.m)
    loss_c = torch.tensor([float(op.losses["loss/coarse_loss"])], dtype=torch.float64)
    dist.all_reduce(loss_c)                              # sum of rank losses -> mean below

    # oracle at batch 32n = mean over the ranks' batches (rank 0 computes all of them)
    if rank == 0:
        p64 = {k: v.double() for k, v in p.items()}
        acc, loss_ref = None, 0.0
        for r in range(world):
            im, dp = bench.synthetic_batch(r, torch)
            mk = (torch.rand(B, 4096, generator=torch.Generator().manual_seed(2 + r)) < 0.5).double()
            g, out = OM.grads(p64, im.double(), dp.double(), mk, "coarse", q=OM.bf16_round)
            loss_ref += float(out["loss_coarse"]) / world
            acc = g if acc is None else {k: acc[k] + g[k] for k in g}
        worst, rows = 1.0, {}
        for name, g in acc.items():
            g = g / world
            a, b = got_m[name].double().reshape(-1), (0.1 * g).reshape(-1)
            c = float(a @ b / (a.norm() * b.norm() + 1e-300))
            rows[name] = {"cos": c, "norm_ratio": float(a.norm() / (b.norm() + 1e-300))}
            worst = min(worst, c)
        report["m_vs_oracle_batch_%d" % (B * world)] = rows
        report["worst_cosine"] = worst
        report["loss_coarse_mean_over_ranks"] = float(loss_c) / world
        report["loss_coarse_oracle_big_batch"] = loss_ref
    # a second step: replicas must stay in lock-step
    op.run()
    net.flush()
    torch.cuda.synchronize()
    report["identical_bf16_weights_after_step_2"] = all_equal(net.arena.wb.view(torch.int16), world)
    bias_ok = True
    for s in net.arena.specs.values():
        if s.kind == "bias":
            bias_ok &= all_equal(net.arena.w[s.offset:s.offset + s.numel], world)
    report["identical_f32_biases_after_step_2"] = bias_ok
    ok = True
    if rank == 0:
        ok = (report["worst_cosine"] >= 0.999 and all(v for k, v in report.items() if k.startswith("identical_"))
              and abs(report["loss_coarse_mean_over_ranks"] - report["loss_coarse_oracle_big_batch"])
              <= 1e-2 * abs(report["loss_coarse_oracle_big_batch"]))
        report["pass"] = ok
        if args.out:
            os.makedirs(args.out, exist_ok=True)
            with open(os.path.join(args.out, f"dp_parity_r02_n{world}.json"), "w") as f:
                json.dump(report, f, indent=1)
        print(json.dumps({k: v for k, v in report.items() if not k.startswith("m_vs_")}), flush=True)
    dist.barrier()
    sys.stdout.flush()
    os._exit(0 if ok else 1)


if __name__ == "__main__":
    main()
