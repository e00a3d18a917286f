"""FP8 against bf16 inference of MSDN on one GPU: captured-graph forward latency and images/s at batch 1, 32 and 512
(the two modes measured alternately, several rounds, warm autotuned shapes, glorot weights as tools/infer_sweep.py),
per-call CUDA-event times of one un-graphed forward in each mode, and the FP8 maps' relative L2 error against the bf16
maps of the same net and inputs.  The card's name, power limit and max SM clock are read in the same run.

    python tools/fp8_infer_bench.py [--out profiles/fp8_infer_bench_r05.json] [--batches 1,32,512] [--rounds 5]
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

FWD_FLOP = 4.110e9          # MSDN forward FLOP per image (tools/infer_sweep.py)


def card():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    name, power, clock = [x.strip() for x in r.stdout.strip().splitlines()[0].split(",")]
    return {"name": name, "power_limit": power, "max_sm_clock": clock, "torch_name": torch.cuda.get_device_name()}


class Timed:
    """Stands in for the net's ops.Context: every liba3d call of the forward is bracketed by CUDA events."""

    def __init__(self, ctx):
        self._ctx, self.calls = ctx, []

    def __getattr__(self, name):
        f = getattr(self._ctx, name)
        if not callable(f) or name.startswith("_") or name in ("workspace", "stamp", "conv_ws"):
            return f

        def wrapped(*a, **k):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            r = f(*a, **k)
            e1.record()
            shape = next((tuple(x.shape) for x in a if torch.is_tensor(x)), ())
            self.calls.append((f"{len(self.calls):02d} {name} {shape}", e0, e1))
            return r
        return wrapped

    def __setattr__(self, name, value):
        if name in ("_ctx", "calls"):
            object.__setattr__(self, name, value)
        else:
            setattr(self._ctx, name, value)


def per_call(net):
    real = net.ctx
    net.ctx = Timed(real)
    try:
        net.forward()
        torch.cuda.synchronize()
        return [{"call": lab, "us": e0.elapsed_time(e1) * 1e3} for lab, e0, e1 in net.ctx.calls]
    finally:
        net.ctx = real


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default="profiles/fp8_infer_bench_r05.json")
    ap.add_argument("--batches", default="1,32,512")
    ap.add_argument("--rounds", type=int, default=5)
    args = ap.parse_args()
    res = {"card": card(), "rounds": args.rounds, "batches": []}
    print(res["card"], flush=True)
    p = glorot_params(1)
    for bs in (int(b) for b in args.batches.split(",")):
        g = torch.Generator().manual_seed(bs)
        images = torch.rand(bs, 480, 640, 3, generator=g).cuda()
        depths = torch.rand(bs, 55, 73, 1, generator=g).cuda() + 0.05
        ops, graphs = {}, {}
        for mode in ("bf16", "fp8"):
            op = models.msdn(images, depths, train=False, dtype=mode)
            op.net.load_params(p)
            for _ in range(3):
                op.net.forward()
            torch.cuda.synchronize()
            gr = torch.cuda.CUDAGraph()
            with torch.cuda.graph(gr):
                op.net.forward()
            gr.replay()
            torch.cuda.synchronize()
            ops[mode], graphs[mode] = op, gr
        err = {k: float((getattr(ops["fp8"], k).double() - getattr(ops["bf16"], k).double()).norm() /
                        getattr(ops["bf16"], k).double().norm()) for k in ("outputs", "coarse")}
        reps = max(10, int(200 / bs))
        times = {"bf16": [], "fp8": []}
        for _ in range(args.rounds):
            for mode in ("bf16", "fp8"):
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                for _ in range(reps):
                    graphs[mode].replay()
                e1.record()
                torch.cuda.synchronize()
                times[mode].append(e0.elapsed_time(e1) / reps)
        row = {"batch": bs, "reps_per_round": reps, "rel_l2_fp8_vs_bf16": {"fine": err["outputs"], "coarse": err["coarse"]}}
        for mode in ("bf16", "fp8"):
            ms = statistics.median(times[mode])
            row[mode] = {"latency_ms_median": ms, "latency_ms_rounds": times[mode], "images_per_s": bs / ms * 1e3,
                         "tflops": FWD_FLOP * bs / ms / 1e9, "per_call_us": per_call(ops[mode].net)}
        row["speedup_fp8"] = row["bf16"]["latency_ms_median"] / row["fp8"]["latency_ms_median"]
        print({k: v for k, v in row.items() if k not in ("bf16", "fp8")},
              {m: round(row[m]["latency_ms_median"], 4) for m in ("bf16", "fp8")}, flush=True)
        res["batches"].append(row)
        del ops, graphs
        torch.cuda.empty_cache()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
