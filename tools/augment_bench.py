"""Cost of training-time augmentation: the augmented resizes against the plain ones (CUDA events over many launches), and
the batch-32 MSDN phase-1 graph step with and without augmentation, alternated in one process.

  MSDN: B = 32, image 480x640x3 (float32 and uint8) -> 228x304 space-to-depth(4) bf16; target 55x73 -> 55x74.
  DCNF: B = 16, image 480x640x3 and depth 480x640 -> 240x320 float32.

Sources rotate over enough copies to exceed the 126 MB L2, so every launch reads its batch from HBM.  Algorithmic bytes =
one read of the source and one write of the output.  The card's name, power limit and maximum SM clock are read in the
same run.  Usage: python tools/augment_bench.py [--out PATH] [--iters N]
"""
import argparse
import json
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch

from ann3depth_b200 import models
from ann3depth_b200.augment import Augment
from ann3depth_b200.init import glorot_params

HBM_TBS = 7.7                # HGX B200 data sheet, one GPU
L2_BYTES = 126 * 2 ** 20


def card():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return {"torch_name": torch.cuda.get_device_name(), "nvidia_smi": r.stdout.strip().splitlines()[:1]}


def time_us(fn, iters, warmup=20):
    for i in range(warmup):
        fn(i)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(iters):
        fn(i)
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / iters * 1e3


def copies_of(make, nbytes):
    n = max(2, -(-2 * L2_BYTES // nbytes))
    return [make() for _ in range(n)]


def kernel_pairs(ctx, iters):
    g = torch.Generator(device="cuda").manual_seed(0)
    aug = Augment.eigen_nyu()
    res = []

    def params(B):
        p = torch.zeros(B, 16, device="cuda")
        ctx.augment_draw(aug.desc(), p, 1, torch.tensor([7], dtype=torch.int64, device="cuda"))
        return p

    def record(name, B, src_bytes, out_bytes, plain, augm, n_copies):
        tp, ta = time_us(plain, iters), time_us(augm, iters)
        nb = src_bytes + out_bytes
        res.append({"case": name, "B": B, "plain_us": tp, "augmented_us": ta, "ratio": ta / tp,
                    "algorithmic_bytes": nb, "plain_share_of_hbm": nb / (tp * 1e-6) / 1e12 / HBM_TBS,
                    "augmented_share_of_hbm": nb / (ta * 1e-6) / 1e12 / HBM_TBS, "source_copies": n_copies})

    B = 32
    p32 = params(B)
    out = torch.empty(B, 57, 76, 64, dtype=torch.bfloat16, device="cuda")
    for dt, nbytes in ((torch.float32, 4), (torch.uint8, 1)):
        sb = B * 480 * 640 * 3 * nbytes
        if dt == torch.float32:
            srcs = copies_of(lambda: torch.rand(B, 480, 640, 3, device="cuda", generator=g), sb)
        else:
            srcs = copies_of(lambda: torch.randint(0, 256, (B, 480, 640, 3), device="cuda", generator=g,
                                                   dtype=torch.uint8), sb)
        n = len(srcs)
        record(f"msdn image {'f32' if nbytes == 4 else 'u8'} -> s2d bf16", B, sb, out.numel() * 2,
               lambda i: ctx.resize_bilinear_tf1_s2d(srcs[i % n], 228, 304, 4, out=out),
               lambda i: ctx.resize_affine_tf1_s2d(srcs[i % n], 228, 304, 4, p32, out=out), n)
        del srcs
    sb = B * 55 * 73 * 4
    deps = copies_of(lambda: torch.rand(B, 55, 73, 1, device="cuda", generator=g), sb)
    tar = torch.empty(B, 55, 74, 1, device="cuda")
    n = len(deps)
    record("msdn target 55x73 -> 55x74", B, sb, tar.numel() * 4,
           lambda i: ctx.resize_bilinear_tf1(deps[i % n], 55, 74, out=tar),
           lambda i: ctx.resize_affine_tf1(deps[i % n], 55, 74, p32, depth=True, out=tar), n)
    del deps
    B = 16
    p16 = params(B)
    for ch, depth in ((3, False), (1, True)):
        sb = B * 480 * 640 * ch * 4
        srcs = copies_of(lambda: torch.rand(B, 480, 640, ch, device="cuda", generator=g), sb)
        o = torch.empty(B, 240, 320, ch, device="cuda")
        n = len(srcs)
        record(f"dcnf {'depth' if depth else 'image'} 480x640x{ch} -> 240x320", B, sb, o.numel() * 4,
               lambda i: ctx.resize_bilinear_tf1(srcs[i % n], 240, 320, out=o),
               lambda i: ctx.resize_affine_tf1(srcs[i % n], 240, 320, p16, depth=depth, out=o), n)
        del srcs
    draw_us = time_us(lambda i: ctx.augment_draw(aug.desc(), p32, 1, None), iters)
    return res, draw_us


def step_pair(rounds, steps):
    B = 32
    g = torch.Generator(device="cuda").manual_seed(1)
    images = torch.rand(B, 480, 640, 3, device="cuda", generator=g)
    depths = torch.rand(B, 55, 73, 1, device="cuda", generator=g) * 9 + 0.5
    ops = {"plain": models.msdn(images, depths, train=True),
           "augmented": models.msdn(images, depths, train=True, augment=Augment.eigen_nyu())}
    for op in ops.values():
        op.net.load_params(glorot_params(seed=1, model="msdn"))
        for _ in range(3):
            op.run()
    torch.cuda.synchronize()
    times = {k: [] for k in ops}
    for _ in range(rounds):
        for k, op in ops.items():
            times[k].append(time_us(lambda i: op.run(), steps, warmup=2) / 1e3)
    med = {k: sorted(v)[len(v) // 2] for k, v in times.items()}
    return {"B": B, "phase": 1, "steps_per_window": steps, "rounds": rounds, "ms_per_step": times,
            "median_ms": med, "ratio": med["augmented"] / med["plain"]}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default="augment_bench.json")
    ap.add_argument("--iters", type=int, default=400)
    ap.add_argument("--rounds", type=int, default=7)
    ap.add_argument("--steps", type=int, default=30)
    a = ap.parse_args()
    ctx = models.get_context(0)
    res = {"card": card(), "iters": a.iters}
    res["kernels"], res["draw_us"] = kernel_pairs(ctx, a.iters)
    torch.cuda.empty_cache()
    res["msdn_phase1_step"] = step_pair(a.rounds, a.steps)
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res, indent=1))


if __name__ == "__main__":
    main()
