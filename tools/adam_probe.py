#!/usr/bin/env python
"""Times a3d_dense_wgrad_adam (fused dense weight gradient + TF-Adam) alone on MSDN's dense_0 shape and
reports the achieved HBM bandwidth (26 B/parameter); the separate wgrad + Adam kernels for comparison."""
import json
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from ann3depth_b200 import models  # noqa: E402


def main():
    ctx = models.get_context(0)
    dev = torch.device("cuda:0")
    M, N, K = 32, 4096, 12288
    x = (torch.rand(M, K, device=dev) - 0.5).bfloat16()
    dy = (torch.rand(M, N, device=dev) - 0.5).bfloat16()
    w = torch.rand(N, K, device=dev)
    m = torch.zeros(N, K, device=dev)
    v = torch.zeros(N, K, device=dev)
    wb = torch.zeros(N, K, dtype=torch.bfloat16, device=dev)
    db = torch.zeros(N, device=dev)
    g = torch.zeros(N, K, device=dev)
    flush = torch.empty(64 << 20, device=dev)

    def timed(fn, reps=5):
        best = 1e9
        for _ in range(reps):
            flush.fill_(0.0)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(); fn(); e1.record()
            torch.cuda.synchronize()
            best = min(best, e0.elapsed_time(e1))
        return best * 1e3

    fused = lambda: ctx.dense_wgrad_adam(x, dy, db, w, m, v, wb, 0.1, 0.9, 0.999, 1e-8, 1)
    fused(); torch.cuda.synchronize()
    tf = timed(fused)
    sep_w = lambda: ctx.dense_wgrad(x, dy, dw=g, db=db)
    sep_a = lambda: ctx.adam_tf(w.view(-1), g.view(-1), m.view(-1), v.view(-1), wb.view(-1), 0.1, 0.9, 0.999, 1e-8, 1)
    sep_w(); sep_a(); torch.cuda.synchronize()
    tw, ta = timed(sep_w), timed(sep_a)
    print(json.dumps({"fused_us": tf, "fused_GBs": 26.0 * N * K / tf / 1e3, "wgrad_us": tw, "adam_us": ta,
                      "adam_GBs": 30.0 * N * K / ta / 1e3}), flush=True)


if __name__ == "__main__":
    main()
