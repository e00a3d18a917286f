"""Cost of evaluation: a3d_depth_metrics alone (CUDA events over many launches, both scale modes) at the shapes the two
models evaluate, and evaluation throughput with device-resident batches against inference alone.

  MSDN: B = 32, prediction 55x74 into 480x640 ground truth;  DCNF: B = 16, 240x320 into 480x640.

Algorithmic bytes = one read of the ground truth and of the prediction plus the sums written (the kernel reads the ground
truth 1x without and 4x with median scaling; repeated reads of one image come from L2).  The ground truth rotates over
enough copies (> 126 MB of L2) that every launch reads its image from HBM the first time.  The card's name, power limit
and maximum SM clock are read in the same run.  Usage: python tools/eval_bench.py [--out PATH]
"""
import argparse
import json
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch

from ann3depth_b200 import models
from ann3depth_b200.evaluate import DepthMetrics
from ann3depth_b200.init import glorot_params

HBM_TBS = 7.7                # HGX B200 data sheet, one GPU


def card():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return {"torch_name": torch.cuda.get_device_name(), "nvidia_smi": r.stdout.strip().splitlines()[:1]}


def time_ms(fn, iters):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    fn(0)
    torch.cuda.synchronize()
    e0.record()
    for i in range(iters):
        fn(i)
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / iters


def kernel_case(ctx, B, ph, pw, gh, gw, median, iters):
    g = torch.Generator(device="cuda").manual_seed(0)
    copies = max(2, -(-160 * 2 ** 20 // (B * gh * gw * 4)))
    gts = [torch.randint(1, 256, (B, gh, gw), device="cuda", generator=g).float() / 255.0 for _ in range(copies)]
    pred = torch.rand(B, ph, pw, device="cuda", generator=g)
    sums = torch.empty(B, 11, dtype=torch.float64, device="cuda")
    scale = torch.empty(B, device="cuda")
    ms = time_ms(lambda i: ctx.depth_metrics(pred, gts[i % copies], 1e-3, 1.0, median=median, sums=sums, scale=scale),
                 iters)
    nbytes = B * (gh * gw + ph * pw) * 4 + sums.numel() * 8
    return {"B": B, "pred": [ph, pw], "gt": [gh, gw], "scale": "median" if median else "none", "us": ms * 1e3,
            "algorithmic_bytes": nbytes, "GB_per_s": nbytes / ms / 1e6, "share_of_hbm": nbytes / ms / 1e9 / HBM_TBS,
            "gt_copies_rotated": copies}


def throughput(model, B, iters):
    g = torch.Generator(device="cuda").manual_seed(1)
    images = torch.rand(B, 480, 640, 3, device="cuda", generator=g)
    depths = torch.randint(0, 256, (B, 480, 640, 1), device="cuda", generator=g).float() / 255.0
    op = getattr(models, model)(images, depths, train=False)
    op.net.load_params(glorot_params(seed=1, model=model))
    outs = {"fine": op.outputs, "coarse": op.coarse} if model == "msdn" else {"output": op.outputs}
    res = {"B": B, "outputs": list(outs)}
    res["infer_ms"] = time_ms(lambda i: op.run(), iters)
    for scale in ("none", "median"):
        meters = {k: DepthMetrics(op.net.ctx, scale=scale) for k in outs}

        def step(i):
            op.run()
            for k, m in meters.items():
                m.update(outs[k], depths, B)
        ms = time_ms(step, iters)
        res[f"eval_ms_{scale}"] = ms
        res[f"eval_images_per_s_{scale}"] = B / ms * 1e3
        res[f"metrics_share_{scale}"] = (ms - res["infer_ms"]) / ms
    res["infer_images_per_s"] = B / res["infer_ms"] * 1e3
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default="")
    ap.add_argument("--iters", type=int, default=200)
    args = ap.parse_args()
    ctx = models.get_context()
    res = {"card": card(), "kernel": [], "throughput": {}}
    for B, ph, pw in ((32, 55, 74), (16, 240, 320), (1, 55, 74)):
        for median in (False, True):
            r = kernel_case(ctx, B, ph, pw, 480, 640, median, args.iters)
            res["kernel"].append(r)
            print(json.dumps(r), flush=True)
    for model, B in (("msdn", 32), ("dcnf", 16)):
        res["throughput"][model] = throughput(model, B, max(args.iters // 10, 10))
        print(model, json.dumps(res["throughput"][model]), flush=True)
    print(json.dumps(res["card"]))
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
