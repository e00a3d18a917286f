"""Synchronous data parallelism for the MSDN/DCNF step: one process per GPU, full weight replica per
rank, gradient sum-allreduce (NCCL over NVLink 5 / NVSwitch) of flat arena buckets on a dedicated
communication stream, overlapped with the rest of the backward pass.

Replaces the asynchronous parameter-server replication of the reference (src/ann3depth.py:78-92,
`replica_device_setter` + gRPC variable pulls / gradient pushes every `session.run`).  Semantics
change: the reference applies stale per-worker gradients; here n ranks x batch B behave like one
rank x batch n*B (gradients averaged: sum-allreduce, 1/n folded into the optimizer's grad_scale).
"""
from __future__ import annotations

import torch

from . import ops


class DataParallel:
    def __init__(self, ctx: ops.Context, rank: int, world: int, unique_id: bytes, nccl_path: str | None = None):
        self.ctx, self.rank, self.world = ctx, rank, world
        ctx.comm_init(unique_id, rank, world, nccl_path)
        # The communication stream outranks the compute streams: its kernels are few and short (NCCL CTAs, the row-sharded
        # dense update) but sit on the step's critical chain; at normal priority the 13 / 35 us row updates of an 8-GPU
        # step waited ~170 / 200 us for a free SM slot among the backward GEMMs' CTAs (profiles/step_timeline_r02_n8*).
        self.stream = torch.cuda.Stream(device=ctx.device, priority=-3)
        self._done = []
        self.bytes_per_step = 0

    @staticmethod
    def bucket_range(net, name):
        a = net.arena
        if name in a.groups:
            return a.group_range(name)
        if name == "coarse_conv":
            return a.group_range("CoarseConv")
        if name in ("coarse_conv_main", "coarse_conv_0"):
            # conv2d_4 .. conv2d_1 (99 % of the group; exchanged under the rest of the backward pass) | conv2d_0
            # (55 k parameters: the only exchange left in the step's tail)
            lo, hi = a.group_range("CoarseConv")
            cut = a.specs["coarse/conv/conv2d_0/kernel"].offset
            return (lo, cut) if name == "coarse_conv_main" else (cut, hi)
        if name == "fine":
            lo_a, hi_a = a.group_range("FineA")
            lo_b, hi_b = a.group_range("FineB")
            return min(lo_a, lo_b), max(hi_a, hi_b)
        if name == "all":
            return 0, a.total
        # a single layer: kernel + bias segments are adjacent
        keys = [k for k in a.specs if k.startswith(name + "/") or ("/" + name + "/") in k]
        lo = min(a.specs[k].offset for k in keys)
        hi = max(a.specs[k].offset + a.specs[k].size for k in keys)
        return lo, hi

    def bucket_ready(self, net, name, then=None, after=None):
        """Called right after the wgrad kernels of a bucket were enqueued on the current stream.
        `then(lo, hi)`: optional work enqueued on the comm stream right behind the allreduce (the bucket's
        optimizer update); `after`: an extra event that work must wait for (e.g. the last reader of the
        weights the update overwrites)."""
        lo, hi = self.bucket_range(net, name)
        ready = torch.cuda.Event()
        ready.record(torch.cuda.current_stream())
        with torch.cuda.stream(self.stream):
            self.stream.wait_event(ready)
            self.ctx.stamp(f"comm: allreduce {name} begin")
            self.ctx.allreduce_sum(net.arena.g[lo:hi])
            self.ctx.stamp(f"comm: allreduce {name} end")
            if then is not None:
                if after is not None:
                    self.stream.wait_event(after)
                then(lo, hi)
            done = torch.cuda.Event()
            done.record(self.stream)
        self._done.append(done)
        self.bytes_per_step += (hi - lo) * 4

    def sharded_adam(self, net, name, group, lr, beta1, eps, after=None):
        """ZeRO-1 style exchange for one bucket, enqueued on the comm stream behind the bucket's wgrads:
             f32 grads -> bf16  |  reduce-scatter (sum)  |  TF-Adam on this rank's 1/n slice (grad_scale 1/n)
             |  all-gather of the bf16 weight mirror.
        Half the NVLink bytes of an f32 allreduce and 1/n of the optimizer's HBM traffic per rank.  The f32
        master weights and Adam slots of the other ranks' slices are not kept up to date on this rank
        (`gather_master` refreshes them, e.g. before a checkpoint)."""
        a = net.arena
        lo, hi = self.bucket_range(net, name)
        n = hi - lo
        assert n % (self.world * 8) == 0, "bucket must split into 16-byte aligned rank slices"
        chunk = n // self.world
        if a.gb is None:
            a.gb = torch.zeros(a.total, dtype=torch.bfloat16, device=a.w.device)
        ready = torch.cuda.Event()
        ready.record(torch.cuda.current_stream())
        with torch.cuda.stream(self.stream):
            self.stream.wait_event(ready)
            self.ctx.cast_f32_bf16(a.g[lo:hi], a.gb[lo:hi])
            self.ctx.stamp(f"comm: reduce-scatter {name} begin")
            ops.reduce_scatter_sum(self.ctx, a.gb[lo:hi], chunk)
            self.ctx.stamp(f"comm: reduce-scatter {name} end")
            if after is not None:
                self.stream.wait_event(after)
            s = lo + self.rank * chunk
            self.ctx.adam_tf_bf16g(a.w[s:s + chunk], a.gb[s:s + chunk], a.m[s:s + chunk], a.v[s:s + chunk],
                                   a.wb[s:s + chunk], lr, beta1, net.beta2, eps, max(net.adam_t[group], 1),
                                   1.0 / self.world, lr_t_dev=net.lr_dev[group])
            ops.allgather(self.ctx, a.wb[lo:hi], chunk)
            self._sync_sharded_biases(net, lo, hi, chunk)
            self.ctx.stamp(f"comm: sharded adam + allgather {name} end")
            done = torch.cuda.Event()
            done.record(self.stream)
        self._done.append(done)
        self.bytes_per_step += n * 2 * 2
        self._sharded = getattr(self, "_sharded", set()) | {name}

    def _sync_sharded_biases(self, net, lo, hi, chunk):
        """The kernels read biases as f32 from the MASTER buffer (msdn.MSDNNet.bias), which a sharded Adam updates only
        on the rank that owns the slice: publish the owners' values of every bias segment in [lo, hi) to all ranks.
        A few KB: each rank contributes its owned elements (zeros elsewhere) to one small f32 sum-allreduce."""
        a = net.arena
        key = ("bias_sync", lo, hi)
        plan = getattr(self, "_bias_plans", None)
        if plan is None:
            plan = self._bias_plans = {}
        if key not in plan:
            segs, pos = [], 0
            for s in a.specs.values():
                if s.kind == "bias" and lo <= s.offset and s.offset + s.numel <= hi:
                    segs.append((s.offset, s.numel, pos))
                    pos += (s.numel + 3) // 4 * 4
            own_lo, own_hi = lo + self.rank * chunk, lo + (self.rank + 1) * chunk
            mine = []
            for off, n, pos_ in segs:
                b, e = max(off, own_lo), min(off + n, own_hi)
                if b < e:
                    mine.append((b, e, pos_ + b - off))
            plan[key] = (segs, mine, torch.zeros(max(pos, 4), dtype=torch.float32, device=a.w.device))
        segs, mine, stage = plan[key]
        if not segs:
            return
        stage.zero_()
        for b, e, p0 in mine:
            stage[p0:p0 + e - b].copy_(a.w[b:e])
        self.ctx.allreduce_sum(stage)
        for off, n, p0 in segs:
            a.w[off:off + n].copy_(stage[p0:p0 + n])

    def can_gather_dense(self, net, kernel_name, batch):
        """The activation-gather update needs equal 16-row-aligned row slices and a gathered batch <= 256."""
        s = net.arena.specs[kernel_name]
        rows = s.packed_shape[0]
        return rows % (self.world * 16) == 0 and batch * self.world <= 256 and s.packed_shape[1] % 256 == 0

    def dense_gather_adam_merged(self, net, layers, group, lr, beta1, eps, ready):
        """Data-parallel step of the dense layers without a gradient all-reduce: ranks exchange activations, not gradients.
             ONE all-gather of every layer's x [B,K] and dy [B,N] (one latency-bound collective instead of one per layer)
             |  per layer: this rank updates its row slice of the kernel from the gathered batch (grad_scale 1/n) and the
                replicated bias, behind that layer's `after` event (its dgrad: the last reader of the old weights).
           NVLink traffic per rank: the bf16 weights once (no reduce-scatter of gradients).
           The all-gather of the updated bf16 rows of dense_0 is NOT enqueued here: nobody reads those weights before the
           next step's dense forward, so `publish_rows` runs at the START of the next step on the comm stream, under the next step's
           resize + convolution forward (the 134 MB weight exchange was ~330 us of serial NCCL time at the end of the
           8-GPU step; profiles/step_timeline_r02_n8_rank0.json).  `flush` publishes outside a step (checkpoint, export,
           end of a timed loop).
        layers: [(kernel_name, bias_name, x, dy, after_event)]; ready: event after which every x / dy is final."""
        a, c, n = net.arena, self.ctx, self.world
        B = layers[0][2].shape[0]
        # The slice's gradient comes from the tcgen05 wgrad GEMM (f32) followed by the streaming TF-Adam pass (34 B/param;
        # 0.77-0.91 of the HBM roofline at 8 / 4 / 2 GPUs).  An mma.sync row kernel that formed the gradient in registers
        # and applied TF-Adam in the same pass (26 B/param) reloaded x per row tile: 0.49 of the roofline at a gathered
        # batch of 64, 0.22 at 256 -- measured slower in the step at every world size (2 GPUs: 1.096 vs 1.047 ms).
        bufs = getattr(self, "_gbufs", None)
        if bufs is None:
            bufs = self._gbufs = {}
        t = max(net.adam_t[group], 1)
        self.rows_launches = getattr(self, "rows_launches", {})
        key = ("gather_plain",) + tuple(l[0] for l in layers)
        if key not in bufs:
            bufs[key] = [(torch.zeros(n * B, x.shape[1], dtype=torch.bfloat16, device=x.device),
                          torch.zeros(n * B, dy.shape[1], dtype=torch.bfloat16, device=x.device))
                         for _, _, x, dy, _ in layers]
        mats = bufs[key]
        with torch.cuda.stream(self.stream):
            self.stream.wait_event(ready)
            for (kn, bn_, x, dy, after), (xg, dyg) in zip(layers, mats):
                xg[self.rank * B:(self.rank + 1) * B].copy_(x)
                dyg[self.rank * B:(self.rank + 1) * B].copy_(dy)
            c.stamp("comm: allgather x,dy (all dense layers) begin")
            c.allgather_multi([m_.view(-1) for pair in mats for m_ in pair])
            c.stamp("comm: allgather x,dy (all dense layers) end")
            for (kn, bn_, x, dy, after), (xg, dyg) in zip(layers, mats):
                ks = a.specs[kn]
                rows, K = ks.packed_shape
                N, lddy = ks.tf_shape[1], dy.shape[1]
                r = rows // n
                lo_r = self.rank * r
                s0_ = ks.offset + lo_r * K
                if after is not None:
                    self.stream.wait_event(after)

                def rows_launch(kn=kn, xg=xg, dyg=dyg, lo_r=lo_r, r=r, K=K, s0_=s0_):
                    c.dense_wgrad(xg, dyg[:, lo_r:lo_r + r], dw=a.view(a.g, kn)[lo_r:lo_r + r], db=None, N=r)
                    sl = slice(s0_, s0_ + r * K)
                    c.adam_tf(a.w[sl], a.g[sl], a.m[sl], a.v[sl], a.wb[sl], lr, beta1, net.beta2, eps, t, 1.0 / n,
                              lr_t_dev=net.lr_dev[group])
                rows_launch()
                # bench.py times exactly this launch for the data-parallel roofline line
                self.rows_launches[kn] = (rows_launch, dict(M=n * B, rows=r, rows_all=rows, K=K, lddy=lddy,
                                                            kernel="a3d_dense_wgrad (row slice, tcgen05) + a3d_adam_tf",
                                                            bytes_per_param=34.0))
                # bias: replicated update from the gathered dy
                bs = a.specs[bn_]
                sl = slice(bs.offset, bs.offset + bs.size)
                c.bias_grad_bf16(dyg, N, a.g[bs.offset:bs.offset + N], rows=n * B, ld=lddy)
                c.adam_tf(a.w[sl], a.g[sl], a.m[sl], a.v[sl], a.wb[sl], lr, beta1, net.beta2, eps, t, 1.0 / n,
                          lr_t_dev=net.lr_dev[group])
                c.stamp(f"comm: rows update {kn.split('/')[-2]} end")
                self.bytes_per_step += rows * K * 2
                self._row_sharded = getattr(self, "_row_sharded", set()) | {kn}
                if kn.split("/")[-2] == "dense_1":
                    # a layer updated early in the backward pass is published right away: the comm stream is idle until
                    # the conv gradients exist, and the next step's start then only carries the rest
                    ops.allgather(c, a.view(a.wb, kn).view(-1), r * K)
                    c.stamp(f"comm: publish bf16 rows {kn.split('/')[-2]} (in step) end")
                else:
                    self._unpublished = getattr(self, "_unpublished", set()) | {kn}
            done = torch.cuda.Event()
            done.record(self.stream)
        self._done.append(done)
        self.bytes_per_step += sum(m_.numel() for pair in mats for m_ in pair) * 2

    def publish_rows(self, net):
        """All-gather of the bf16 rows updated by the previous step's dense_gather_adam_merged; enqueued on the comm stream
        behind whatever the current stream has done so far.  Returns the event the first reader of the dense weights has
        to wait for (None when nothing is pending)."""
        pending = sorted(getattr(self, "_unpublished", ()))
        if not pending:
            return None
        a, c = net.arena, self.ctx
        start = torch.cuda.Event()
        start.record(torch.cuda.current_stream())
        with torch.cuda.stream(self.stream):
            self.stream.wait_event(start)
            c.stamp("comm: publish bf16 rows begin")
            for kn in pending:
                rows, K = a.specs[kn].packed_shape
                ops.allgather(c, a.view(a.wb, kn).view(-1), rows // self.world * K)
            c.stamp("comm: publish bf16 rows end")
            ev = torch.cuda.Event()
            ev.record(self.stream)
        return ev

    def flush(self, net):
        """Publish pending weight rows NOW (outside a step): before anything reads the bf16 mirror of rows another rank
        owns -- checkpoints, exports, parity checks, the end of a timed loop."""
        ev = self.publish_rows(net)
        if ev is not None:
            torch.cuda.current_stream().wait_event(ev)

    def gather_master(self, net):
        """All-gather the f32 master weights and Adam slots of every sharded bucket (checkpoint / export)."""
        a = net.arena
        pending = sorted(getattr(self, "_unpublished", ()))
        for kn in pending:                                   # runs on the caller's (comm) stream, like the rest below
            rows, K = a.specs[kn].packed_shape
            ops.allgather(self.ctx, a.view(a.wb, kn).view(-1), rows // self.world * K)
        for name in sorted(getattr(self, "_sharded", ())):
            lo, hi = self.bucket_range(net, name)
            chunk = (hi - lo) // self.world
            for buf in (a.w, a.m, a.v):
                ops.allgather(self.ctx, buf[lo:hi], chunk)
        for name in sorted(getattr(self, "_row_sharded", ())):
            rows, K = a.specs[name].packed_shape
            for buf in (a.w, a.m, a.v):
                ops.allgather(self.ctx, a.view(buf, name).view(-1), rows // self.world * K)

    def wait_all(self, net):
        cur = torch.cuda.current_stream()
        for e in self._done:
            cur.wait_event(e)
        self._done = []
