"""Evaluation of a trained model on the test split, beyond the reference (its README: "we have not implemented a test
or validation yet").

`DepthMetrics` accumulates the standard depth-estimation metrics of Eigen et al. (2014) on the device:
`a3d_depth_metrics` samples each prediction at every pixel of the full-resolution ground truth and reduces the per-image
sums (include/a3d.h); `update` adds them to a float64 device vector without a host sync, `reduce` sums that vector over
the ranks (gloo), `result` turns it into the metrics.  Dataset metrics pool all valid pixels of all images (abs_rel,
sq_rel, rmse, rmse_log, log10, delta1-3); silog = sqrt(mean d^2 - (mean d)^2), d = ln p - ln g, is taken per image and
averaged over the images with a valid pixel.  The defaults suit the reference's data: its depths are min-max byte-scaled
relative depths k/255 (tools/data_tf_converter.py), so min_depth = 1e-3 excludes exactly the zeros.

    python -m ann3depth_b200.evaluate nyu --model msdn --ckptdir checkpoints --id run1 --batchsize 32 --datadir data
                                          [--scale median] [--dtype fp8] [--json metrics.json]

restores `<ckptdir>/<model>[_<id>]/model.ckpt` into the inference net and reads `<datadir>/<dataset>/test.tfrecords`
once.  MSDN reports its two outputs `fine` (the reference's prediction) and `coarse`; DCNF its `output`.  Under
`torchrun` the ranks evaluate disjoint shards of the file and the chief logs / writes the reduced result.  `--dtype fp8`
evaluates MSDN in its FP8 inference mode (E4M3 products; include/a3d.h "FP8 inference"), so the metrics show what FP8
costs on the user's own model.
"""
from __future__ import annotations

import argparse
import json
import logging
import math
import os
import sys

import torch

from . import _lib as L

logger = logging.getLogger("ann3depth.evaluate")

_NS = len(L.DM_SLOTS)
_SILOG, _SILOG_IMAGES, _IMAGES = _NS, _NS + 1, _NS + 2
METRICS = ("abs_rel", "sq_rel", "rmse", "rmse_log", "log10", "silog", "delta1", "delta2", "delta3")


class DepthMetrics:
    """Accumulator of the metrics of one prediction stream.  ctx: ops.Context (None: `add_sums` only)."""

    def __init__(self, ctx, min_depth=1e-3, max_depth=1.0, scale="none", device=None):
        if scale not in ("none", "median"):
            raise ValueError("scale must be 'none' or 'median'")
        self.ctx, self.min_depth, self.max_depth, self.median = ctx, float(min_depth), float(max_depth), scale == "median"
        if device is None:
            device = f"cuda:{ctx.device}" if ctx is not None else "cpu"
        self.acc = torch.zeros(_NS + 3, dtype=torch.float64, device=device)
        self._sums = None

    def reset(self):
        self.acc.zero_()

    def update(self, pred, gt, n_valid=None):
        """pred f32 [B,ph,pw(,1)], gt f32 [B,gh,gw(,1)] (CUDA, contiguous); only the first n_valid images count."""
        n = pred.shape[0] if n_valid is None else int(n_valid)
        if n <= 0:
            return
        if self._sums is None or self._sums.shape[0] < n:
            self._sums = torch.empty(pred.shape[0], _NS, dtype=torch.float64, device=pred.device)
        sums = self.ctx.depth_metrics(pred[:n], gt[:n], self.min_depth, self.max_depth, self.median, sums=self._sums[:n])
        self.add_sums(sums)

    def add_sums(self, sums):
        """Accumulate per-image slot sums [n, len(DM_SLOTS)] (what a3d_depth_metrics writes)."""
        npx = sums[:, 0]
        has = npx > 0
        m = sums[:, 4] / npx.clamp(min=1)
        silog = torch.sqrt(torch.clamp(sums[:, 5] / npx.clamp(min=1) - m * m, min=0.0))
        self.acc[:_NS] += sums.sum(0)
        self.acc[_SILOG] += torch.where(has, silog, torch.zeros_like(silog)).sum()
        self.acc[_SILOG_IMAGES] += has.sum()
        self.acc[_IMAGES] += sums.shape[0]

    def reduce(self, group=None):
        """Sum the accumulators of all ranks (torch.distributed all_reduce on the float64 vector; gloo: through the host).
        No-op without an initialised process group of more than one rank."""
        import torch.distributed as dist
        if not (dist.is_available() and dist.is_initialized()) or dist.get_world_size(group) == 1:
            return
        t = self.acc.cpu()
        dist.all_reduce(t, group=group)
        self.acc.copy_(t)

    def result(self):
        a = [float(x) for x in self.acc.cpu()]
        N = a[0]
        res = {"images": int(a[_IMAGES]), "pixels": int(N), "nonfinite": int(a[10])}
        if N == 0:
            res.update({k: None for k in METRICS})
            return res
        res.update(abs_rel=a[1] / N, sq_rel=a[2] / N, rmse=math.sqrt(a[3] / N), rmse_log=math.sqrt(a[5] / N),
                   log10=a[6] / N, silog=a[_SILOG] / max(a[_SILOG_IMAGES], 1.0), delta1=a[7] / N, delta2=a[8] / N,
                   delta3=a[9] / N)
        return res


def model_outputs(op):
    """{name: prediction tensor [B,h,w,1]} of an op built by models.msdn / models.dcnf."""
    net = op.net
    if hasattr(net, "fine"):
        return {"fine": op.outputs, "coarse": op.coarse}
    return {"output": op.outputs}


def evaluate_split(op, inp, meters):
    """Run `op` (train=False) over the single-pass reader `inp` once; update one DepthMetrics per output name."""
    outs = model_outputs(op)
    while True:
        n = inp.next_batch()
        if not n:
            break
        op.net.infer()
        for name, m in meters.items():
            m.update(outs[name], inp.depths, n)
    return meters


def make_meters(op, ctx, scale="none", min_depth=1e-3, max_depth=1.0):
    return {name: DepthMetrics(ctx, min_depth, max_depth, scale) for name in model_outputs(op)}


def main(argv=None):
    logging.basicConfig(level=logging.INFO, stream=sys.stdout, format="%(asctime)s %(name)s %(levelname)s %(message)s")
    args = parse_args(argv)
    from . import data, models
    from .ann3depth import restore_checkpoint
    rank, world = int(os.environ.get("RANK", 0)), int(os.environ.get("WORLD_SIZE", 1))
    torch.cuda.set_device(int(os.environ.get("LOCAL_RANK", 0)))
    path = os.path.join(args.datadir, args.dataset, "test.tfrecords")
    if not os.path.exists(path):
        raise SystemExit(f"evaluate: {path} not found (the test split is required; there is no synthetic evaluation)")
    run_id = args.model + ("" if not args.id else f"_{args.id}")
    ckptdir = os.path.join(args.ckptdir, run_id)
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("gloo")
    if args.dtype == "fp8" and args.model != "msdn":
        raise SystemExit(f"evaluate: {args.model.upper()} has no FP8 mode (--dtype fp8 runs MSDN only)")
    inp = data.inputs(args.datadir, args.dataset, args.batchsize, "test", epochs=1, shard=(rank, world))
    op = getattr(models, args.model)(inp.images, inp.depths, train=False,
                                     **({"dtype": "fp8"} if args.dtype == "fp8" else {}))
    if not restore_checkpoint(op, ckptdir):
        raise SystemExit(f"evaluate: no checkpoint in {ckptdir}")
    meters = evaluate_split(op, inp, make_meters(op, op.net.ctx, args.scale, args.min_depth, args.max_depth))
    inp.close()
    for m in meters.values():
        m.reduce()
    results = {name: m.result() for name, m in meters.items()}
    first = next(iter(results.values()))
    out = {"model": args.model, "dtype": args.dtype, "global_step": op.global_step, "scale": args.scale, "images": first["images"],
           "pixels": first["pixels"], "metrics": {name: {k: r[k] for k in ("nonfinite",) + METRICS}
                                                  for name, r in results.items()}}
    if rank == 0:
        for name, r in out["metrics"].items():
            logger.info(f"{args.model}/{name} at step {out['global_step']} on {out['images']} images: " +
                        " ".join(f"{k}={v:.4g}" if v is not None else f"{k}=n/a" for k, v in r.items()))
        if args.json:
            with open(args.json, "w") as f:
                json.dump(out, f, indent=1)
    if world > 1:
        import torch.distributed as dist
        dist.destroy_process_group()
    return out


def parse_args(argv=None):
    p = argparse.ArgumentParser(description="Depth metrics of a checkpoint on the test split.")
    p.add_argument("dataset", default="nyu", type=str, nargs="?", help="The dataset to use.")
    p.add_argument("--model", "-m", default="msdn", choices=("msdn", "dcnf"))
    p.add_argument("--ckptdir", "-p", default="checkpoints", help="Checkpoint directory (as for training).")
    p.add_argument("--id", default="", type=str, help="Checkpoint path suffix (as for training).")
    p.add_argument("--batchsize", "-b", default=32, type=int)
    p.add_argument("--datadir", "-d", default="data", type=str, help="The data directory containing the datasets.")
    p.add_argument("--scale", default="none", choices=("none", "median"), help="Median-scale each prediction first.")
    p.add_argument("--min-depth", default=1e-3, type=float, help="Valid pixels: min_depth < gt <= max_depth.")
    p.add_argument("--max-depth", default=1.0, type=float)
    p.add_argument("--dtype", default="bf16", choices=("bf16", "fp8"),
                   help="Inference precision: bf16, or fp8 (MSDN only: E4M3 products with per-channel weight and "
                        "per-image activation scales).")
    p.add_argument("--json", default="", help="Write the result to this file.")
    return p.parse_args(argv)


if __name__ == "__main__":
    main()
