#!/usr/bin/env python
"""bench.py -- MSDN train images/s (BASELINE.json metric) on N B200s of one node.

    python bench.py --gpus N --steps K --warmup W            # this repo (liba3d, sm_100a)
    python bench.py --impl reference --gpus N --steps K ...   # restated reference on the host CPU cores
    python bench.py ... --dump-outputs DIR                   # + what the last timed step computed, as DIR/*.npy
    python bench.py ... --ops-json PATH                      # + per-kernel CUDA-event table of one sequential step

A "step" is one `session.run(model_op)` of the reference loop (src/ann3depth.py:126-127) at the
default schedule position (phase 1, src/models.py:301-305): forward of the coarse and fine stacks on
a batch of 32 synthetic 640x480 RGB images (+55x73 depth targets), both scale-invariant losses,
backward through the coarse stack and the two TF-Adam groups.  For N > 1 the driver launches one
rank per GPU with torch.distributed.run; every rank holds a replica and its own batch of 32 (weak
scaling), gradients are sum-allreduced with NCCL.  Rank 0 prints ONE JSON line.
"""
import argparse
import json
import os
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

BATCH = 32
FLOP_PER_IMAGE_PHASE1 = 9.357e9          # BASELINE.md section 4 (2*MAC, unpadded dims)
H2D_BYTES = BATCH * (480 * 640 * 3 + 55 * 73) * 4
D2H_BYTES = 8


def workload_config(world):
    return {"workload": "msdn phase-1 train step (fwd coarse+fine, 2 losses, coarse bwd, 2 TF-Adam groups), batch 32/GPU, "
                        "640x480 RGB -> 55x73 depth, glorot init seed 1",
            "parallelism": f"dp{world}", "global_batch": BATCH * world,
            "l2": "working set per step (~2.6 GB: activations + 283 MB weights + Adam slots) >> 126 MB L2",
            "adam": "reference TF-Adam(beta1=0.9, beta2=1, eps=1e-8)"}


def peaks():
    try:
        return json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json"))), "measured"
    except Exception:
        return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0}, "fallback"


class ClockSampler(threading.Thread):
    """Samples SM clock and throttle reasons (NVML) during the timed region."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.samples, self.reasons, self.stop_flag, self.max_mhz = index, [], set(), False, None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nv = None

    def run(self):
        if not self.nv:
            return
        nv = self.nv
        names = {nv.nvmlClocksThrottleReasonHwSlowdown: "hw_slowdown",
                 nv.nvmlClocksThrottleReasonHwThermalSlowdown: "hw_thermal_slowdown",
                 nv.nvmlClocksThrottleReasonSwThermalSlowdown: "sw_thermal_slowdown",
                 nv.nvmlClocksThrottleReasonSwPowerCap: "sw_power_cap"}
        while not self.stop_flag:
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for bit, nm in names.items():
                    if r & bit:
                        self.reasons.add(nm)
            except Exception:
                pass
            time.sleep(0.005)

    def summary(self):
        s = sorted(self.samples)
        return {"sm_mhz": s[len(s) // 2] if s else None, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons),
                "samples": len(s)}


def bind_to_gpu_numa(index):
    """Best effort: run this rank on the CPUs next to its GPU (NVML's ideal affinity), so that the pinned input buffers
    it allocates afterwards are first-touched on the GPU's own memory node.  Returns the CPU list or None."""
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(index)
        words = (os.cpu_count() + 63) // 64
        mask = pynvml.nvmlDeviceGetCpuAffinity(h, words)
        cpus = [w * 64 + b for w, m in enumerate(mask) for b in range(64) if (m >> b) & 1]
        cpus = [c for c in cpus if c < os.cpu_count()]
        if cpus:
            os.sched_setaffinity(0, cpus)
            return cpus
    except Exception:
        pass
    return None


def synthetic_batch(rank, torch):
    g = torch.Generator().manual_seed(100 + rank)
    images = torch.rand(BATCH, 480, 640, 3, generator=g)
    depths = torch.rand(BATCH, 55, 73, 1, generator=g) * 0.95 + 0.05
    return images, depths


def dump_outputs(op, out_dir, torch):
    """Writes what the last step gave its caller, as float32 DIR/<name>.npy (~1 MB): both losses and both depth maps.
    The trainable variables are not written: the reference's Adam (beta2 = 1) has a zero step size, so they stay at their
    initial values.  Nor are the Adam slots, which are optimizer state, not results: at the initial weights the loss
    takes log(depth + 1e-8) of predictions that straddle zero, so the few nearest zero dominate the gradient, and the
    float32 atomics of the split-K reductions move them from run to run.  Two runs of one build (B200, 50 timed steps)
    agreed per slot to a cosine >= 0.9995 but differed by ~39 % RMS, while the depth maps and losses agreed to 8e-4."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    arrays = {"loss_coarse": op.losses["loss/coarse_loss"], "loss_fine": op.losses["loss/fine_loss"],
              "coarse": op.coarse, "fine": op.outputs}
    for name, t in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), t.detach().to("cpu", torch.float32).numpy())


# --------------------------------------------------------------------------------------- CPU arm
def cpu_train_step_rate(steps, warmup, budget_s=150.0):
    """Times the CPU restatement of the reference step (oracle/, float32, all host threads).
    Returns (images_per_s, cores, sample description, ms_per_step)."""
    import torch
    from oracle import msdn as OM
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    p = OM.init_params(1, torch.float32)
    images, depths = synthetic_batch(0, torch)
    mask = (torch.rand(BATCH, 4096, generator=torch.Generator().manual_seed(2)) < 0.5).float()

    # Variables + Adam slots are created ONCE (TF keeps them in place across session.run calls) and updated in place;
    # the timed region holds nothing but the step itself.  global_step is rewound so every run is a phase-1 step.
    st = OM.TrainState(p)

    def run(b):
        st.global_step = 0
        t0 = time.perf_counter()
        OM.train_step(st, images[:b], depths[:b], mask[:b], inplace=True)
        return time.perf_counter() - t0

    run(2)                                    # page-in / oneDNN primitive cache
    per_img = run(4) / 4
    b = BATCH
    while b > 4 and (steps + warmup) * b * per_img > budget_s:
        b //= 2
    for _ in range(warmup):
        run(b)
    t0 = time.perf_counter()
    for _ in range(steps):
        run(b)
    dt = time.perf_counter() - t0
    sample = (f"{steps} phase-1 train steps of {b} images each (of the 32-image batch), float32 PyTorch-CPU "
              f"restatement of src/models.py (TensorFlow 1.3 is not installable here), {cores} threads")
    return steps * b / dt, cores, sample, dt / steps * 1e3


def reference_arm(args, rank):
    if rank != 0:
        return
    v, cores, sample, ms = cpu_train_step_rate(args.steps, args.warmup)
    line = {"impl": "reference", "metric": "MSDN train images/s (bs32/GPU, phase-1 step)", "value": v,
            "unit": "images/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": workload_config(args.gpus),
            "cpu_baseline": {"value": v, "unit": "images/s", "cores": cores, "kind": "port", "sample": sample},
            "e2e": {"value": v, "unit": "images/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


# --------------------------------------------------------------------------------------- GPU arm
def per_op_profile(op, torch, reps=3):
    """Times every liba3d call of one (non-graph) step with CUDA events on the launching stream."""
    ctx = op.net.ctx
    records = []
    lib = ctx.lib
    from ann3depth_b200 import _lib as L
    wrapped = {}
    stream = torch.cuda.current_stream()
    for name in L.SIGNATURES:
        fn = getattr(lib, name)
        if name in ("a3d_last_error", "a3d_version", "a3d_launch_count", "a3d_sm_count", "a3d_conv2d_ws_bytes",
                    "a3d_pairwise_ws_bytes", "a3d_create", "a3d_destroy"):
            continue

        def make(fn, name):
            def w(*a):
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record(stream)
                rc = fn(*a)
                e1.record(stream)
                detail = ""
                if name.startswith("a3d_conv2d"):
                    d = a[1]._obj
                    detail = f"N{d.N} {d.H}x{d.W}x{d.C}->{d.P}x{d.Q}x{d.K} k{d.R}x{d.S} s{d.stride_h}"
                elif name == "a3d_adam_tf":
                    detail = f"n={int(a[6])}"
                elif name in ("a3d_dense_fwd", "a3d_dense_dgrad", "a3d_dense_wgrad", "a3d_dense_wgrad_adam"):
                    i0 = {"a3d_dense_fwd": 10, "a3d_dense_dgrad": 6, "a3d_dense_wgrad": 7, "a3d_dense_wgrad_adam": 10}[name]
                    detail = "MNK=" + "x".join(str(int(x)) for x in a[i0:i0 + 3])
                records.append((name, detail, e0, e1))
                return rc
            return w
        wrapped[name] = fn
        setattr(lib, name, make(fn, name))
    try:
        agg = {}
        for r in range(reps):
            records.clear()
            op.net.global_step = 0
            op.run(use_graph=False)
            torch.cuda.synchronize()
            for i, (name, detail, e0, e1) in enumerate(records):
                key = (i, name, detail)
                agg.setdefault(key, []).append(e0.elapsed_time(e1))
    finally:
        for name, fn in wrapped.items():
            setattr(lib, name, fn)
    rows = [{"seq": k[0], "op": k[1], "detail": k[2], "ms": min(v)} for k, v in sorted(agg.items())]
    return rows


# Layers whose stored shape is a padded re-expression of the reference layer: ALGORITHMIC FLOPs per image
# (SURVEY.md section 8a, unpadded dims) instead of the stored dims.
ALGORITHMIC_FLOPS_PER_IMAGE = {
    "57x76x64->55x74x96 k3x3 s1": 2.0 * 55 * 74 * 96 * 11 * 11 * 3,        # coarse/conv2d_0: 11x11x3 s4 (M1)
    "57x76x64->55x74x256 k3x3 s1": 2.0 * 110 * 148 * 63 * 9 * 9 * 3,       # fine/first 9x9x3 s2 -> 63 (+pool) (M12)
    "27x37x128->27x37x256 k5x5 s1": 2.0 * 27 * 37 * 256 * 5 * 5 * 96,      # coarse/conv2d_1: 96 input channels stored as 128 (M3)
}


def conv_flops(detail):
    try:
        left, right = detail.split("->")
        key = detail.split(" ", 1)[1]
        if key in ALGORITHMIC_FLOPS_PER_IMAGE:
            return ALGORITHMIC_FLOPS_PER_IMAGE[key] * int(left.split()[0][1:])
        n = int(left.split()[0][1:])
        c = int(left.split()[1].split("x")[2])
        p, q, k = (int(x) for x in right.split()[0].split("x"))
        r, s = (int(x) for x in right.split()[1][1:].split("x"))
        return 2.0 * n * p * q * k * r * s * c
    except Exception:
        return 0.0


def other_configs(torch, pk):
    """BASELINE.json configs 4 and 5 and the TF32 precision mode, as short extra measurements on rank 0 of a single-GPU
    run (the headline stays config 2: MSDN bs32 phase-1 train step).  CUDA events, inputs resident in HBM."""
    from ann3depth_b200 import models
    from ann3depth_b200.init import glorot_params
    out = {}
    dev = torch.device("cuda:0")

    def timed(fn, n):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        e0.record()
        for _ in range(n):
            fn()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / n

    # ---- TF32 precision mode: the same phase-1 step with float32 storage and tcgen05 kind::tf32
    images, depths = synthetic_batch(0, torch)
    notes = {"tf32": "float32 activations + tcgen05.mma kind::tf32, sequential schedule, CUDA graph",
             "tf32x3": "as tf32, forward contractions as 3xTF32 sums over hi/lo-split operands (worst pixel < 1e-4)"}
    for mode in ("tf32", "tf32x3"):
        op = models.msdn(images.to(dev), depths.to(dev), train=True, dtype=mode)
        op.net.load_params(glorot_params(seed=1))
        for _ in range(3):
            op.run()
        ms = timed(op.run, 20)
        out["msdn_train_bs32_" + mode] = {"ms_per_step": ms, "images_per_s": BATCH / ms * 1e3,
                                          "step_tflops_algorithmic": FLOP_PER_IMAGE_PHASE1 * BATCH / ms / 1e9,
                                          "note": notes[mode]}
        del op
        torch.cuda.empty_cache()
    # ---- config 5: inference-only depth-map throughput (forward of both stacks, dropout off), CUDA graph replay
    p = glorot_params(seed=1)
    inf = {}
    for bs in (1, 32, 512):
        g = torch.Generator().manual_seed(bs)
        im = torch.rand(bs, 480, 640, 3, generator=g).to(dev)
        opi = models.msdn(im, torch.zeros(bs, 55, 73, 1, device=dev), train=False)
        opi.net.load_params(p)
        for _ in range(3):
            opi.run()
        torch.cuda.synchronize()
        gr = torch.cuda.CUDAGraph()
        with torch.cuda.graph(gr):
            opi.net.forward()
        gr.replay()
        ms = timed(gr.replay, 20)
        tf = 4.110e9 * bs / ms / 1e9                      # BASELINE.md section 4: 4.110 GFLOP forward per image
        inf[f"bs{bs}"] = {"latency_ms": ms, "images_per_s": bs / ms * 1e3, "tflops_algorithmic": tf,
                          "frac_of_bf16_burst": tf / pk["bf16_tflops"]}
        del opi, gr, im
        torch.cuda.empty_cache()
    out["msdn_inference"] = inf
    # ---- config 4: DCNF train step, batch 16 (768 patches through the unary CNN, 16 CRF graphs, SGD)
    g = torch.Generator().manual_seed(3)
    im = torch.rand(16, 480, 640, 3, generator=g).to(dev)
    dp = (torch.rand(16, 480, 640, 1, generator=g) * 0.95 + 0.05).to(dev)
    opd = models.dcnf(im, dp, train=True)
    pp = glorot_params(5, "dcnf")
    pp["pairwise/pairwise_layers/dense/kernel"].abs_()
    opd.net.load_params(pp)
    step = lambda: opd.run(use_graph=True)               # one captured CUDA graph per step (dcnf.py train_step)
    for _ in range(2):
        step()
    ms = timed(step, 10)
    # The reference formulation (48 overlapping patches per image, BASELINE.md section 4) is 2.672 GFLOP forward per patch;
    # the fully convolutional evaluation computes every shared activation once: 46.14 GFLOP forward per IMAGE
    # (11x11x3 at 290x370, 5x5x64 at 141x181, 3x3x256 at 68x88 / 66x86 / 64x84, the dense layers per patch).
    # fwd + dgrad + wgrad ~ 3x forward.  `frac_of_bf16_burst` is on the FLOPs actually needed, not the patch-wise count.
    tf_ref = 3.0 * 2.672e9 * 768 / ms / 1e9
    tf = 3.0 * 46.14e9 * 16 / ms / 1e9
    out["dcnf_train_bs16"] = {"ms_per_step": ms, "images_per_s": 16 / ms * 1e3, "tflops_algorithmic": tf,
                              "tflops_patchwise_equivalent": tf_ref, "frac_of_bf16_burst": tf / pk["bf16_tflops"],
                              "formulation": "fully convolutional (one pass per padded image, 7x7 windows gathered)",
                              "crf_status_max": int(opd.net.status.max())}
    del opd
    torch.cuda.empty_cache()
    return out


def gpu_arm(args, rank, world, local_rank):
    import torch
    import torch.distributed as dist
    from ann3depth_b200 import models, ops
    from ann3depth_b200.dp import DataParallel
    from ann3depth_b200.init import glorot_params

    torch.cuda.set_device(local_rank)
    dev = torch.device(f"cuda:{local_rank}")
    if world > 1 and os.environ.get("A3D_NUMA_BIND", "1") != "0":
        # pinned host batches next to the GPU: e2e at N GPUs is bound by what the host can feed (tools/h2d_ceiling.py).
        # Single-GPU runs stay unbound: the same process times the CPU baseline on ALL host cores.
        bind_to_gpu_numa(local_rank)
    comm = None
    ctx = models.get_context(local_rank)
    if world > 1:
        # torch.distributed (gloo) is control-plane only: rendezvous, barriers, max-over-ranks of the timings.
        # The data path (gradient allreduce) runs on liba3d's own NCCL communicator; keeping a single NCCL
        # communicator per process avoids cross-communicator ordering deadlocks.
        dist.init_process_group("gloo")
        # NCCL prints its version banner on stdout: keep stdout clean for the single JSON line
        sys.stdout.flush()
        saved_fd = os.dup(1)
        os.dup2(2, 1)
        try:
            ids = [ops.comm_unique_id() if rank == 0 else None]
            dist.broadcast_object_list(ids, src=0)
            comm = DataParallel(ctx, rank, world, ids[0])
            warm = torch.zeros(1024, device=dev)
            ctx.allreduce_sum(warm)
            torch.cuda.synchronize()
        finally:
            sys.stdout.flush()
            os.dup2(saved_fd, 1)
            os.close(saved_fd)

    images_h, depths_h = synthetic_batch(rank, torch)
    images_h, depths_h = images_h.pin_memory(), depths_h.pin_memory()
    images, depths = images_h.to(dev), depths_h.to(dev)
    op = models.msdn(images, depths, train=True, comm=comm)
    params_cpu = glorot_params(seed=1)
    op.net.load_params(params_cpu)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    if args.ncu:
        # profiling hook (never a bench value): warm up (autotuning, graph capture), then expose exactly one
        # un-graphed sequential step and one graph replay to `ncu --profile-from-start off`
        for _ in range(3):
            op.run()
        torch.cuda.synchronize()
        torch.cuda.profiler.start()
        saved_overlap, op.net.overlap = op.net.overlap, False
        op.run(use_graph=False)
        op.net.overlap = saved_overlap
        torch.cuda.synchronize()
        op.run()
        torch.cuda.synchronize()
        torch.cuda.profiler.stop()
        print(json.dumps({"ncu": "one sequential step + one graph replay profiled"}), flush=True)
        return

    # ---- device-resident inputs: value
    op.run(use_graph=False)                 # first launch of every shape: autotuning candidates are timed here
    launches0 = ctx.launches
    op.run(use_graph=False)
    launches_per_step = ctx.launches - launches0
    for _ in range(max(args.warmup, 3)):
        op.run()
    sampler = ClockSampler(local_rank)
    barrier()
    sampler.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.steps):
        op.run()
    op.net.flush()          # DP: the last step's deferred weight-row exchange belongs to the timed region (no-op at N=1)
    e1.record()
    barrier()
    sampler.stop_flag = True
    ms_total = e0.elapsed_time(e1)
    t = torch.tensor([ms_total])
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_total = float(t)
    value = BATCH * world * args.steps / (ms_total * 1e-3)
    if args.dump_outputs and rank == 0:
        dump_outputs(op, args.dump_outputs, torch)        # before the e2e passes below step the same op further

    # ---- end to end: pinned host batch -> H2D (prefetched on a copy stream) -> step -> loss D2H
    copy_stream = torch.cuda.Stream(device=dev)

    def measure_e2e(op_, images_dev, images_host):
        stage = [(torch.empty_like(images_dev), torch.empty_like(depths)) for _ in range(2)]
        loss_h = torch.empty(2, dtype=torch.float32).pin_memory()
        ready = [torch.cuda.Event(), torch.cuda.Event()]
        freed = [torch.cuda.Event(), torch.cuda.Event()]

        def prefetch(i):
            with torch.cuda.stream(copy_stream):
                copy_stream.wait_event(freed[i % 2])
                stage[i % 2][0].copy_(images_host, non_blocking=True)
                stage[i % 2][1].copy_(depths_h, non_blocking=True)
                ready[i % 2].record(copy_stream)

        def e2e_loop(n):
            cur = torch.cuda.current_stream()
            for f in freed:
                f.record(cur)
            prefetch(0)
            for i in range(n):
                if i + 1 < n:
                    prefetch(i + 1)
                cur.wait_event(ready[i % 2])
                images_dev.copy_(stage[i % 2][0], non_blocking=True)
                depths.copy_(stage[i % 2][1], non_blocking=True)
                freed[i % 2].record(cur)
                op_.run()
                loss_h[0:1].copy_(op_.losses["loss/coarse_loss"], non_blocking=True)
                loss_h[1:2].copy_(op_.losses["loss/fine_loss"], non_blocking=True)
                cur.synchronize()                       # the driver reads the loss every step
            return float(loss_h[0])

        e2e_loop(3)
        barrier()
        t0 = time.perf_counter()
        last = e2e_loop(args.steps)
        barrier()
        tt = torch.tensor([time.perf_counter() - t0])
        if world > 1:
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        return BATCH * world * args.steps / float(tt), last

    # headline e2e: the reference's tensor contract (float32 images, src/data.py:82-86)
    e2e_value, last_loss = measure_e2e(op, images, images_h)
    # secondary: the same pixels as uint8 (0..255, read as pixel / 255 by the resize kernel) -- a quarter of the
    # PCIe bytes.  Single GPU only (a second net: its own arena, graph and inputs).
    e2e_u8 = None
    if world == 1 and os.environ.get("A3D_BENCH_U8", "1") != "0":
        images8_h = (images_h * 255.0).round().clamp_(0, 255).to(torch.uint8).pin_memory()
        images8 = images8_h.to(dev)
        op8 = models.msdn(images8, depths, train=True)
        op8.net.load_params(params_cpu)
        for _ in range(3):
            op8.run()
        torch.cuda.synchronize()
        v8, loss8 = measure_e2e(op8, images8, images8_h)
        e2e_u8 = {"value": v8, "unit": "images/s", "h2d_bytes_per_step": BATCH * (480 * 640 * 3 + 55 * 73 * 4),
                  "d2h_bytes_per_step": D2H_BYTES, "last_loss": loss8,
                  "note": "uint8 images (pixel/255 in the resize kernel); beyond the reference's float32 contract"}
        del op8

    if rank == 0:
        pk, pk_kind = peaks()
        # per-kernel timing pass runs on rank 0 alone: detach the communicator so that it contains no collective
        # ... and the single-stream schedule, so that each kernel is timed alone on the launching stream
        saved_comm, op.net.comm = op.net.comm, None
        saved_overlap, op.net.overlap = op.net.overlap, False
        rows = per_op_profile(op, torch)
        op.net.comm, op.net.overlap = saved_comm, saved_overlap
        step_ms = ms_total / args.steps
        # dominant kernel of the step, and the conv/FC tensor-pipe aggregate
        top = max(rows, key=lambda r: r["ms"])
        tensor_ops = [r for r in rows if r["op"].startswith("a3d_conv2d")]
        tflops = sum(conv_flops(r["detail"]) for r in tensor_ops)
        tms = sum(r["ms"] for r in tensor_ops)
        if top["op"].startswith("a3d_conv2d"):
            fl = conv_flops(top["detail"])
            ach = fl / (top["ms"] * 1e-3) / 1e12
            roof = {"bound": "tensor", "kernel": f'{top["op"]} {top["detail"]}', "achieved": ach,
                    "peak": pk["bf16_tflops"], "unit": "TFLOP/s", "frac": ach / pk["bf16_tflops"], "traffic": None,
                    "peak_kind": pk_kind + " burst", "share_of_step": top["ms"] / sum(r["ms"] for r in rows)}
        else:
            # algorithmic bytes of the HBM-bound kernels (DESIGN.md 4.2): TF-Adam = 30 B/param (read w,g,m,v;
            # write w,m,v + bf16 mirror); fused dense wgrad + TF-Adam = 26 B/param (no gradient in memory)
            ach = None
            if top["op"] == "a3d_adam_tf" and top["detail"].startswith("n="):
                ach = 30.0 * int(top["detail"][2:]) / (top["ms"] * 1e-3) / 1e9
            elif top["op"] == "a3d_dense_wgrad_adam" and top["detail"].startswith("MNK="):
                mm, nn, kk = (int(x) for x in top["detail"][4:].split("x"))
                ach = (26.0 * nn * kk + 2.0 * mm * (nn + kk)) / (top["ms"] * 1e-3) / 1e9
            roof = {"bound": "hbm", "kernel": f'{top["op"]} {top["detail"]}', "achieved": ach, "peak": pk["hbm_gbs"],
                    "unit": "GB/s", "frac": ach / pk["hbm_gbs"] if ach else None, "traffic": None, "peak_kind": pk_kind,
                    "share_of_step": top["ms"] / sum(r["ms"] for r in rows)}
        # DRAM traffic of the dominant kernel from the committed `ncu --set full` capture (profiles/), if listed
        try:
            traffic = json.load(open(os.path.join(ROOT, "profiles", "ncu_traffic.json")))
            roof["traffic"] = traffic.get(roof["kernel"])
        except Exception:
            pass
        if world > 1 and saved_comm is not None and getattr(saved_comm, "rows_launches", None):
            # Data parallel: the dominant kernel of the step is not the single-GPU fused update but its row-sharded
            # form on the all-gathered batch (dp.dense_gather_adam_merged -> a3d_dense_wgrad_adam_rows).  Time exactly
            # that launch (rank 0, no collective inside) with CUDA events and report ITS roofline.
            kn = "coarse/dense/dense_0/kernel"
            rows_launch, g = saved_comm.rows_launches[kn]
            for _ in range(3):
                rows_launch()
            ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
            ev[0].record()
            for _ in range(10):
                rows_launch()
            ev[1].record()
            torch.cuda.synchronize()
            ms = ev[0].elapsed_time(ev[1]) / 10
            ach = (g["bytes_per_param"] * g["rows"] * g["K"] + 2.0 * g["M"] * (g["K"] + g["lddy"])) / (ms * 1e-3) / 1e9
            roof = {"bound": "hbm", "kernel": f"{g['kernel']} M={g['M']} rows={g['rows']}/{g['rows_all']} K={g['K']}",
                    "achieved": ach, "peak": pk["hbm_gbs"], "unit": "GB/s", "frac": ach / pk["hbm_gbs"],
                    "traffic": None, "peak_kind": pk_kind, "launch_ms": ms,
                    "note": "timed alone on rank 0 (10 launches, CUDA events); this rank's row slice is %.0f B x %d params "
                            "per launch" % (g["bytes_per_param"], g["rows"] * g["K"])}
        roof["conv_tensor_tflops"] = tflops / (tms * 1e-3) / 1e12 if tms else None
        roof["conv_tensor_frac_of_burst"] = roof["conv_tensor_tflops"] / pk["bf16_tflops"] if tms else None
        # conv + FC aggregate (the dense layers at batch 32 are weight-streaming, i.e. HBM-bound, kernels)
        dense_ops = [r for r in rows if r["op"] in ("a3d_dense_fwd", "a3d_dense_dgrad", "a3d_dense_wgrad")]
        # (the fused wgrad + Adam pass runs its 32 FMAs per parameter on the CUDA cores: optimizer, not tensor, time)
        dfl = 0.0
        for r in dense_ops:
            try:
                m, n, k = (int(x) for x in r["detail"][4:].split("x"))
                dfl += 2.0 * m * n * k
            except Exception:
                pass
        dms = sum(r["ms"] for r in dense_ops)
        roof["conv_fc_tensor_tflops"] = (tflops + dfl) / ((tms + dms) * 1e-3) / 1e12 if tms + dms else None
        roof["step_tflops_algorithmic"] = FLOP_PER_IMAGE_PHASE1 * BATCH / (step_ms * 1e-3) / 1e12
        if args.ops_json:
            with open(args.ops_json, "w") as f:
                json.dump({"step_ms_graph": step_ms, "ops": rows}, f, indent=1)
        cpu = None
        if world == 1 and not args.no_cpu_baseline:
            v, cores, sample, _ = cpu_train_step_rate(2, 1, budget_s=25.0)
            cpu = {"value": v, "unit": "images/s", "cores": cores, "kind": "port", "sample": sample}
        line = {"metric": "MSDN train images/s (bs32/GPU, phase-1 step)", "value": value, "unit": "images/s",
                "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": step_ms,
                "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "bf16",
                "data": "synthetic",
                "config": workload_config(world),
                "implementation": {"cuda_graph": True,
                                   "streams": "main (high priority) + fine-forward + dense wgrad/Adam + conv-wgrad (+ NCCL comm)",
                                   "autotune": "tile width / split-K per layer chosen by timing candidates on first use",
                                   "dp": ("dense: all-gather(activations) -> row-sharded fused wgrad+Adam -> all-gather(bf16 weights); "
                                          "conv: reduce-scatter(bf16) -> sharded Adam -> all-gather(bf16 weights)") if world > 1 else None},
                "e2e": {"value": e2e_value, "unit": "images/s", "h2d_bytes_per_step": H2D_BYTES,
                        "d2h_bytes_per_step": D2H_BYTES, "last_loss": last_loss},
                "e2e_u8": e2e_u8,
                "gpu_launches": launches_per_step * args.steps,
                "clocks": sampler.summary(), "roofline": roof, "cpu_baseline": cpu}
        if world == 1 and not args.no_extra:
            try:
                line["other_configs"] = other_configs(torch, pk)
            except Exception as e:                                   # never lose the headline line to an extra
                line["other_configs"] = {"error": repr(e)}
        print(json.dumps(line), flush=True)
    if world > 1:
        # Leave without running destructors: NCCL communicator teardown at interpreter exit is collective and
        # its order across ranks is undefined (observed to hang the launcher for minutes).
        dist.barrier()
        sys.stdout.flush()
        sys.stderr.flush()
        os._exit(0)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="a3d", choices=["a3d", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extra", action="store_true", help="skip the TF32 / inference / DCNF extra measurements")
    ap.add_argument("--ncu", action="store_true", help="profiling hook: cudaProfilerStart/Stop around two steps")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the losses, depth maps and (sampled) variables of the last timed step as DIR/*.npy")
    ap.add_argument("--ops-json", metavar="PATH", help="write the per-kernel CUDA-event table of one sequential step")
    args = ap.parse_args()
    rank = int(os.environ.get("RANK", 0))
    world = int(os.environ.get("WORLD_SIZE", 1))
    local_rank = int(os.environ.get("LOCAL_RANK", 0))
    if (args.dump_outputs or args.ops_json) and (args.impl == "reference" or args.ncu):
        ap.error("--dump-outputs and --ops-json apply to the timed liba3d arm, not to --impl reference or --ncu")
    if args.impl == "reference":
        reference_arm(args, rank)
        return
    gpu_arm(args, rank, world, local_rank)


if __name__ == "__main__":
    main()
