"""Cost of the scale-and-shift-invariant loss against the reference's scale-invariant log loss.

  kernel: one a3d_ssi_loss / a3d_silog_loss call (the loss kernel + the batch mean) on [B, 4070] float32 maps with the
          bf16 gradient at row stride 4096, as the MSDN step calls them, at B = 1, 32 and 512.  The two losses alternate
          over --rounds rounds; each round is CUDA events around --iters launches; "us" is the median round.
  step:   the captured phase-1 MSDN training step (four streams, one CUDA graph) at B = 32, one net built with
          loss="silog" and one with loss="ssi", alternating rounds of --replays replays.

The card's name, power limit and maximum SM clock are read in the same run.
Usage: python tools/ssi_loss_bench.py [--out profiles/ssi_loss_bench_r06.json]
"""
import argparse
import json
import os
import statistics
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch

from ann3depth_b200 import models
from ann3depth_b200.init import glorot_params

H, W = 55, 74


def card():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return {"torch_name": torch.cuda.get_device_name(), "nvidia_smi": r.stdout.strip().splitlines()[:1]}


def time_ms(fn, iters):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    fn()
    torch.cuda.synchronize()
    e0.record()
    for _ in range(iters):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / iters


def kernel_case(ctx, B, iters, rounds):
    g = torch.Generator(device="cuda").manual_seed(B)
    p = torch.rand(B, H * W, device="cuda", generator=g) + 0.5
    t = torch.rand(B, H * W, device="cuda", generator=g) + 0.05
    lps, loss = torch.empty(B, device="cuda"), torch.empty(1, device="cuda")
    d = torch.empty(B, 4096, dtype=torch.bfloat16, device="cuda")
    kw = dict(want_grad=False, loss_ps=lps, loss=loss, dout_bf16=d, dout_ld=4096)
    calls = {"silog": lambda: ctx.silog_loss(p, t, 0.5 / (H * W), **kw),
             "ssi": lambda: ctx.ssi_loss(p, t, H, W, 0.5, 4, **kw)}
    us = {k: [] for k in calls}
    for _ in range(rounds):
        for k, fn in calls.items():
            us[k].append(1e3 * time_ms(fn, iters))
    res = {"B": B, **{k: {"us": statistics.median(v), "us_rounds": v} for k, v in us.items()}}
    res["ssi_over_silog"] = res["ssi"]["us"] / res["silog"]["us"]
    return res


def step_case(B, replays, rounds):
    g = torch.Generator().manual_seed(0)
    images = torch.rand(B, 480, 640, 3, generator=g).cuda()
    depths = (torch.rand(B, 55, 73, 1, generator=g) + 0.05).cuda()
    ops = {}
    for loss in ("silog", "ssi"):
        op = models.msdn(images, depths, train=True, loss=loss)
        op.net.load_params(glorot_params(1))
        for _ in range(3):
            op.run()                                    # capture + warm replays
        ops[loss] = op
    ms = {k: [] for k in ops}
    for _ in range(rounds):
        for k, op in ops.items():
            ms[k].append(time_ms(op.run, replays))
    res = {"B": B, "replays_per_round": replays, **{k: {"ms": statistics.median(v), "ms_rounds": v} for k, v in ms.items()}}
    res["ssi_over_silog"] = res["ssi"]["ms"] / res["silog"]["ms"]
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join("profiles", "ssi_loss_bench_r06.json"))
    ap.add_argument("--iters", type=int, default=200)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--replays", type=int, default=30)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("ssi_loss_bench needs a CUDA device")
    ctx = models.get_context(0)
    res = {"card": card(), "kernel": [], "iters": args.iters, "rounds": args.rounds}
    for B in (1, 32, 512):
        r = kernel_case(ctx, B, args.iters, args.rounds)
        print(json.dumps(r), flush=True)
        res["kernel"].append(r)
    res["step_phase1"] = step_case(32, args.replays, args.rounds)
    print(json.dumps(res["step_phase1"]), flush=True)
    print(json.dumps(res["card"]), flush=True)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
