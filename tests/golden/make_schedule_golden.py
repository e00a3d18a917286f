"""Regenerates tests/golden/msdn_schedule.json, the launch schedule of one eager MSDN step per configuration (needs a GPU;
run from the repo root: python tests/golden/make_schedule_golden.py [--out PATH]).

Every public `ops.Context` method that enqueues work is wrapped; only the outermost call counts as a launch.  A launch
is recorded as its method, every argument by name (defaults included), its scalars and `ConvDesc`, every tensor named symbolically (the `MSDNNet` attribute, the
arena buffer + segment + byte offset, `ws:<key>/<tag>` for a `ctx.workspace` scratch buffer, the `DataParallel`
attribute) with its shape and dtype, the workspaces it takes, and its lane: the stream, numbered by its first launch,
with its priority.  `torch.cuda.Event.record` and `torch.cuda.Stream.wait_event` are wrapped too, which gives each
launch the set of launches that happen before it (same-stream order plus event waits, transitively closed), stored as
a bit mask over the launch indices.

The recorded step is the second one (the first allocates the persistent buffers and, data parallel, leaves the rows
`publish_rows` sends at the start of the next step).  The data-parallel configurations are world 2, recorded for each
rank in this one process: the collectives are recorded but not executed (NCCL needs a GPU per rank, and no host
decision depends on what they compute).
"""
import argparse
import functools
import inspect
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
import torch  # noqa: E402

from ann3depth_b200 import _lib as L, models, ops  # noqa: E402
from ann3depth_b200.augment import Augment  # noqa: E402
from ann3depth_b200.dp import DataParallel  # noqa: E402
from ann3depth_b200.init import glorot_params  # noqa: E402

COLLECTIVES = ("comm_init", "allreduce_sum", "reduce_scatter_sum", "allgather_multi", "allgather")
NOT_LAUNCHES = ("close", "workspace", "conv_ws", "stamp")      # stamp enqueues nothing without a StepTimeline


class Recorder:
    def __init__(self):
        self.on, self.stub, self.depth, self.cur = False, False, 0, None
        self.ctx = self.net = self.comm = None

    def start(self, net):
        self.net, self.comm, self.ctx = net, net.comm, net.ctx
        self.launches, self.lanes, self.prio = [], {}, []
        self.before = {}          # stream handle -> mask of the launches ordered before its next launch
        self.events = {}          # id(event) -> (event, mask at its record)
        self.on = True

    def stop(self):
        self.on = False
        return {"lanes": self.prio, "launches": self.launches}

    # ---- symbolic tensor names
    def regions(self):
        out = []

        def add(name, v):
            if isinstance(v, torch.Tensor) and v.is_cuda and v.numel():
                out.append((v.data_ptr(), v.data_ptr() + v.numel() * v.element_size(), name, v))
            elif isinstance(v, dict):
                for k, x in v.items():
                    add(f"{name}[{k}]", x)
            elif isinstance(v, (list, tuple)):
                for i, x in enumerate(v):
                    add(f"{name}[{i}]", x)
        for k, v in vars(self.net).items():
            if k != "arena":
                add("net." + k, v)
        for k in ("w", "m", "v", "wb", "g", "gb"):
            add("arena." + k, getattr(self.net.arena, k, None))
        add("masks", self.net.arena.masks)
        for (key, tag), v in self.ctx._ws.items():
            add(f"ws:{key}/{tag}", v)
        if self.comm is not None:
            for k, v in vars(self.comm).items():
                add("comm." + k, v)
        return sorted(out, key=lambda r: r[1] - r[0])

    def name(self, t, regions):
        p = t.data_ptr()
        for lo, hi, name, base in regions:
            if lo <= p < hi:
                off = p - lo
                if name.startswith("arena."):
                    e = off // base.element_size()
                    for s_name, s in self.net.arena.specs.items():
                        if s.offset <= e < s.offset + s.size:
                            return f"{name}:{s_name}+{(e - s.offset) * base.element_size()}"
                return f"{name}+{off}" if off else name
        return "anonymous"

    def enc(self, v, regions):
        if isinstance(v, torch.Tensor):
            return {"t": self.name(v, regions), "shape": list(v.shape), "dtype": str(v.dtype)[6:]}
        if isinstance(v, L.ConvDesc):
            return {"desc": {f: getattr(v, f) for f, _ in v._fields_}}
        if isinstance(v, (tuple, list)):
            return [self.enc(x, regions) for x in v]
        if v is None or isinstance(v, (bool, int, float, str)):
            return v
        return {"obj": type(v).__name__}

    # ---- hooks
    def stream_key(self, s):
        return s.cuda_stream

    def launch(self, method, args, fn):
        s = torch.cuda.current_stream()
        h = self.stream_key(s)
        if h not in self.lanes:
            self.lanes[h] = len(self.prio)
            self.prio.append(s.priority)
        i = len(self.launches)
        rec = {"m": method, "lane": self.lanes[h], "ws": [], "hb": format(self.before.get(h, 0), "x")}
        self.launches.append(rec)
        self.cur = rec
        try:
            result = fn() if method not in COLLECTIVES else None
        finally:
            self.cur = None
        if method == "silog_loss" and args["dout_ld"] <= 0:      # include/a3d.h: dout_ld 0 means n
            args["dout_ld"] = args["out"].numel() // args["out"].shape[0]
        regions = self.regions()
        rec["args"] = {n: self.enc(x, regions) for n, x in sorted(args.items())}
        self.before[h] = self.before.get(h, 0) | (1 << i)
        return result

    def record_event(self, ev, stream):
        s = stream if stream is not None else torch.cuda.current_stream()
        self.events[id(ev)] = (ev, self.before.get(self.stream_key(s), 0))

    def wait_event(self, s, ev):
        h = self.stream_key(s)
        self.before[h] = self.before.get(h, 0) | self.events.get(id(ev), (None, 0))[1]


R = Recorder()


def wrap(name, fn):
    sig = inspect.signature(fn)

    @functools.wraps(fn)
    def recorded(self, *a, **k):
        if R.depth or not R.on:
            if name in COLLECTIVES and R.stub:
                return None
            R.depth += 1
            try:
                return fn(self, *a, **k)
            finally:
                R.depth -= 1
        R.depth += 1
        try:
            bound = sig.bind(self, *a, **k)      # positional or keyword, passed or defaulted: the same call
            bound.apply_defaults()
            args = {n: v for n, v in bound.arguments.items() if n != "self"}
            return R.launch(name, args, lambda: fn(self, *a, **k))
        finally:
            R.depth -= 1
    return recorded


def install():
    for name, fn in list(vars(ops.Context).items()):
        if callable(fn) and not name.startswith("_") and name not in NOT_LAUNCHES:
            setattr(ops.Context, name, wrap(name, fn))
    ws = ops.Context.workspace

    def workspace(self, key, nbytes):
        if R.on and R.cur is not None:
            R.cur["ws"].append([repr(key), self.ws_tag])
        return ws(self, key, nbytes)
    ops.Context.workspace = workspace
    rec = torch.cuda.Event.record

    def record(self, stream=None):
        if R.on:
            R.record_event(self, stream)
        return rec(self, stream)
    torch.cuda.Event.record = record
    wait = torch.cuda.Stream.wait_event

    def wait_event(self, event):
        if R.on:
            R.wait_event(self, event)
        return wait(self, event)
    torch.cuda.Stream.wait_event = wait_event


def msdn(B, train=True, comm=None, **kw):
    g = torch.Generator().manual_seed(B)
    images = torch.rand(B, 480, 640, 3, generator=g).cuda()
    depths = (torch.rand(B, 55, 73, 1, generator=g) + 0.05).cuda()
    op = models.msdn(images, depths, train=train, comm=comm, **kw)
    op.net.load_params(glorot_params(1))
    return op


def record_step(op, phase=1):
    """One untimed step, then the recorded one (both eager)."""
    net = op.net
    if phase == 2:
        net.global_step = 2000000 // net.B                # first step of phase 2 (msdn.phase_of)
    op.run(use_graph=False)
    torch.cuda.synchronize()
    R.start(net)
    op.run(use_graph=False)
    out = R.stop()
    torch.cuda.synchronize()
    return out


def single(B, phase=1, train=True, **kw):
    return lambda: record_step(msdn(B, train, **kw), phase)


def data_parallel(B, rank, **kw):
    def run():
        R.stub = True
        try:
            comm = DataParallel(models.get_context(0), rank, 2, b"\0" * 128)
            comm.ctx._world = 2
            return record_step(msdn(B, comm=comm, **kw))
        finally:
            R.stub = False
    return run


# name -> (kind, recorder): "overlapped" compares launch multisets and happens-before, "sequential" the launch list
CONFIGS = {
    "overlap B=32 fused": ("overlapped", single(32)),
    "overlap B=32 unfused": ("overlapped", single(32, fuse_dense_adam=False)),
    "overlap B=32 augment": ("overlapped", single(32, augment=Augment.eigen_nyu())),
    "sequential B=32 fused": ("sequential", single(32, overlap=False)),
    "sequential B=32 unfused": ("sequential", single(32, overlap=False, fuse_dense_adam=False)),
    "phase 2 B=2": ("sequential", single(2, phase=2)),
    "inference B=2": ("sequential", single(2, train=False)),
    "tf32 phase 1 B=2": ("sequential", single(2, dtype="tf32")),
}
for r in (0, 1):
    CONFIGS[f"dp2 rank {r} gather B=32"] = ("overlapped", data_parallel(32, r))
    CONFIGS[f"dp2 rank {r} sharded B=256"] = ("overlapped", data_parallel(256, r))
CONFIGS["dp2 rank 0 sequential B=32"] = ("sequential", data_parallel(32, 0, overlap=False))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(os.path.dirname(os.path.abspath(__file__)), "msdn_schedule.json"))
    args = ap.parse_args()
    install()
    out = {}
    for name, (kind, run) in CONFIGS.items():
        out[name] = dict(kind=kind, **run())
        print(f"{name}: {len(out[name]['launches'])} launches on {len(out[name]['lanes'])} streams", file=sys.stderr)
    with open(args.out, "w") as f:
        json.dump(out, f, indent=None, separators=(",", ":"), sort_keys=True)
        f.write("\n")


if __name__ == "__main__":
    main()
