"""MSDN (Eigen et al. 2014) train / inference step on liba3d -- host-side orchestration.

Mirrors `_MultiScaleDeepNetwork` of the reference (src/models.py:203-367): preprocessing resize,
coarse stack, fine stack, two scale-invariant log losses, and the three-phase schedule with four
TF-Adam instances.  Every arithmetic operation is a liba3d kernel launched on the current CUDA
stream; PyTorch only owns the buffers.  The whole step is captured in a CUDA graph per phase.
"""
from __future__ import annotations

import contextlib
import os

import torch

from . import _lib as L
from . import ops
from .params import Arena, msdn_specs, fine_first_index_maps, FINE_FIRST_EMBEDDED_SHAPE

IN_H, IN_W = 228, 304          # src/models.py:282
OUT_H, OUT_W = 55, 74          # src/models.py:283
N_PIX = OUT_H * OUT_W          # 4070 == the 74*55 of src/models.py:269
LAMBDA_OVER_N = 0.5 / (74 * 55)
# loss="ssi": the scale-and-shift-invariant objective of MiDaS (Ranftl et al. 2020), gradient-matching weight and scales
SSI_ALPHA, SSI_SCALES = 0.5, 4
LOSSES = ("silog", "ssi")

# src/models.py:318-345 -- (learning rate) per Adam instance; beta1 = 0.9 ('momentum'), eps = 1e-8
ADAM_LR = {"CoarseConv": 0.001, "CoarseDense": 0.1, "FineA": 0.001, "FineB": 0.01}
ADAM_BETA1, ADAM_EPS = 0.9, 1e-8
ADAM_BETA2_REFERENCE = 1.0     # third positional argument of AdamOptimizer, src/models.py:309


def phase_of(global_step: int, batchsize: int) -> int:
    """src/models.py:301-305,347-364 (batchsize is the per-replica batch, as in the reference)."""
    steps_coarse = 2000000 // batchsize
    steps_fine = 1500000 // batchsize
    if global_step < steps_coarse:
        return 1
    if global_step < steps_coarse + steps_fine:
        return 2
    return 3


class _Lanes:
    """Stream placement of the phase-1 training step with `MSDNNet.overlap`, written as annotations on its one launch
    sequence.  The main stream (HIGH PRIORITY: freed SM slots go to its pending CTAs first; graph capture keeps the
    priority as a kernel-node attribute) carries the critical path: resize, coarse forward and loss, the dgrad chain.
    "fine" takes the depth target, the dropout mask and the fine forward + loss, later the conv bias gradients; "wgrad"
    the dense weight gradients and updates; "cwgrad" the conv weight gradients.  Each side stream forks from the step's
    start and joins the main stream before the step counter moves, and sets its own `ctx.ws_tag`: concurrent launches
    must not share scratch.  `lane(name, *labels)` runs a block on that stream behind the events `mark(label)` recorded
    (labels never marked are skipped).  _SEQUENTIAL, with all of it a no-op, runs every launch on the current stream."""
    SIDES = ("fine", "wgrad", "cwgrad")

    def __init__(self, net=None):
        self.on, self.net, self.events = net is not None, net, {}

    def __enter__(self):
        if self.on:
            net = self.net
            if net._streams is None:
                net._streams = {"main": torch.cuda.Stream(device=net.dev, priority=-1),
                                **{k: torch.cuda.Stream(device=net.dev) for k in self.SIDES}}
            self.caller, start = torch.cuda.current_stream(), self._record()
            self._main = torch.cuda.stream(net._streams["main"])
            self._main.__enter__()
            for st in net._streams.values():
                st.wait_event(start)
        return self

    def __exit__(self, *exc):
        if self.on:
            end = self._record()
            self._main.__exit__(*exc)
            self.caller.wait_event(end)

    @contextlib.contextmanager
    def lane(self, name, *after):
        if not self.on:
            yield
            return
        ctx = self.net.ctx
        tag, ctx.ws_tag = ctx.ws_tag, "" if name == "main" else name
        try:
            with torch.cuda.stream(self.net._streams[name]):
                self.wait(*after)
                yield
        finally:
            ctx.ws_tag = tag

    @staticmethod
    def _record(stream=None):
        e = torch.cuda.Event()
        e.record(stream)
        return e

    def mark(self, label):
        if self.on:
            self.events[label] = self._record()

    def event(self, label):
        return self.events.get(label)

    def wait(self, *labels):
        for e in filter(None, map(self.events.get, labels)):
            torch.cuda.current_stream().wait_event(e)

    def join(self):
        if self.on:
            for k in self.SIDES:
                torch.cuda.current_stream().wait_event(self._record(self.net._streams[k]))


_SEQUENTIAL = _Lanes()


class MSDNNet:
    """Buffers + launch sequence for one replica with a static batch size (the reference requires a
    static batch dimension too: `int(images.shape[0])`, src/models.py:225,256,299).

    `fuse_dense_adam=True` fuses the dense weight gradients into TF-Adam where the kernel supports it: on one GPU, at a
    batch of at most `L.DENSE_WGRAD_ADAM_MAX_M`.  A larger batch, like `fuse_dense_adam=False`, runs the separate dense
    wgrad and TF-Adam kernels over the CoarseDense group.

    `loss` picks the objective of both maps: "silog" (default) is the reference's scale-invariant log loss; "ssi" is the
    scale-and-shift-invariant loss (include/a3d.h a3d_ssi_loss, alpha 0.5, 4 scales), for ground truth that is known
    only up to a scale and a shift per image, as the min-max scaled targets of the preprocessing are."""

    def __init__(self, ctx: ops.Context, batch: int, in_hw=(480, 640), depth_hw=(55, 73), train=True,
                 beta2=ADAM_BETA2_REFERENCE, impl=L.IMPL_AUTO, dropout_seed=2, comm=None, grad_dtype=torch.float32,
                 overlap=True, fuse_dense_adam=True, dtype="bf16", augment=None, augment_seed=3, loss="silog"):
        if loss not in LOSSES:
            raise ValueError(f"loss must be one of {LOSSES}, not {loss!r}")
        self.loss = loss
        self.ctx, self.B, self.train, self.beta2, self.impl = ctx, batch, train, beta2, impl
        # dtype = "fp8": inference only.  Every convolution and dense product runs on E4M3 codes (tcgen05 kind::f8f6f4)
        # with one scale per weight row and one per image (include/a3d.h "FP8 inference"); the bf16 buffers below stay as
        # the quantisers' sources, and fine/third, the maps and the losses are computed as in the bf16 mode.
        self.fp8 = dtype == "fp8"
        if self.fp8:
            if train:
                raise ValueError("dtype='fp8' is an inference mode: build the net with train=False")
            if augment is not None:
                raise ValueError("dtype='fp8' is an inference mode and takes no augment=")
            if comm is not None:
                raise ValueError("dtype='fp8' is a single-GPU inference mode (no comm)")
        if augment is not None and not train:
            raise ValueError("augment is a training option: an inference net (train=False) sees its inputs unchanged")
        # dtype = "bf16" (default): BF16 storage of activations / activation gradients / the weight mirror, tcgen05
        # kind::f16.  dtype = "tf32": everything stays float32 in memory -- the reference's own storage type
        # (src/models.py:211-251) -- and the contractions run on tcgen05 kind::tf32 (north star: 1e-4 forward agreement).
        # The TF32 mode runs the sequential schedule with separate wgrad + TF-Adam kernels (the fused / multi-stream
        # kernels are BF16-storage kernels); single GPU.
        # dtype = "tf32x3": as "tf32", with every forward contraction as a 3xTF32 sum over hi/lo-split operands
        # (a3d_conv2d_fwd_tf32x3 / a3d_dense_fwd_tf32x3): float32-grade products, which is what the 1e-4 worst-pixel
        # bound needs (plain TF32 reaches 2.6e-4, profiles/tf32_parity_r02.log).  The backward pass stays plain TF32.
        if dtype not in ("bf16", "tf32", "tf32x3", "fp8"):
            raise ValueError("dtype must be 'bf16', 'tf32', 'tf32x3' or 'fp8'")
        self.tf32 = dtype in ("tf32", "tf32x3")
        self.x3 = dtype == "tf32x3"
        if self.tf32:
            if comm is not None:
                raise ValueError("dtype='tf32' is a single-GPU precision mode")
            overlap, fuse_dense_adam = False, False
        self.overlap = overlap                # phase-1 step on four streams (see _Lanes)
        # single GPU: the dense weight gradients (32 FMAs per parameter at batch 32) are recomputed on the CUDA cores
        # inside the HBM-bound TF-Adam pass (a3d_dense_wgrad_adam), so the 67 M-element f32 gradient is never written
        # or re-read: 26 instead of 38 bytes per dense parameter and step.  Data parallel runs need the gradient in
        # memory for the reduce-scatter and keep the separate kernels (dp.py shards the optimizer instead).
        self.fuse_dense_adam = fuse_dense_adam and batch <= L.DENSE_WGRAD_ADAM_MAX_M
        self._streams = None          # the phase-1 step's streams (_Lanes), created on first use
        self._wflip = None            # flipped filters of the stride-1 dgrads (refreshed at the start of every step)
        self.dev = torch.device(f"cuda:{ctx.device}")
        self.in_hw, self.depth_hw = in_hw, depth_hw
        self.comm = comm                      # data-parallel hook (ann3depth_b200.dp.DataParallel) or None
        self.arena = Arena(msdn_specs(), self.dev)
        self.global_step = 0
        self.adam_t = {g: 0 for g in ADAM_LR}
        self.dropout_seed = dropout_seed
        B = batch
        f32 = dict(dtype=torch.float32, device=self.dev)
        bf = f32 if self.tf32 else dict(dtype=torch.bfloat16, device=self.dev)        # the activation storage type
        z = torch.zeros
        # ---- static input buffers (the "placeholders" the driver refills each step)
        self.images = z(B, in_hw[0], in_hw[1], 3, **f32)
        self.depths = z(B, depth_hw[0], depth_hw[1], 1, **f32)
        self.keep_mask = torch.ones(B, 4096, dtype=torch.uint8, device=self.dev)
        self.external_mask = False
        # training-time augmentation (augment.Augment, beyond the reference): one transform per image and step, drawn on
        # the device from (seed, step_dev, image) and applied by the resizes that open the step.  Each data-parallel
        # rank draws with its own seed (its batch differs anyway).
        self.augment = augment
        self.aug_params = self.aug_desc = None
        self.external_aug = False
        if augment is not None:
            self.aug_desc = augment.desc()
            self.augment_seed = augment_seed + (comm.rank if comm is not None else 0)
            self.aug_params = torch.zeros(B, L.AUG_PARAMS, dtype=torch.float32, device=self.dev)
        # ---- forward activations
        # resized image in space-to-depth(4) layout: 4x4 pixel blocks -> 48 channels (+16 zero) = 128-byte pixels.
        # Both first layers are 3x3 stride-1 convolutions on it (coarse 11x11 s4; fine 9x9 s2 + pool = 11x11 s4).
        self.img4 = z(B, IN_H // 4, IN_W // 4, 64, **bf)
        self.tar = z(B, OUT_H, OUT_W, 1, **f32)         # resized target
        # conv outputs that feed a max-pool stay f32 and the pool records its routing (see a3d.h).  Inference has no routing
        # to record: the conv writes bf16 and the pool runs on bf16 -- the same values (rounding is monotone, so
        # max(bf16(x)) == bf16(max(x))) at half the bytes
        pool_src = f32 if (train or self.tf32) else bf
        self.c0 = z(B, 55, 74, 96, **pool_src)
        self.p0 = z(B, 27, 37, 128, **bf)               # 96 channels + 32 zero: 128-byte pixels for conv2d_1
        self.i0 = torch.zeros(B, 27, 37, 96, dtype=torch.uint8, device=self.dev)
        self.c1 = z(B, 27, 37, 256, **pool_src)
        self.p1 = z(B, 13, 18, 256, **bf)
        self.i1 = torch.zeros(B, 13, 18, 256, dtype=torch.uint8, device=self.dev)
        self.c2 = z(B, 13, 18, 384, **bf)
        self.c3 = z(B, 13, 18, 384, **bf)
        self.c4 = z(B, 6, 8, 256, **bf)
        self.d0 = z(B, 4096, **bf)                      # relu + dropout applied
        self.coarse = z(B, N_PIX, **f32)
        self.if1 = torch.zeros(B, 55, 74, 64, dtype=torch.uint8, device=self.dev)    # pool routing of fine/first
        self.cat = z(B, 55, 74, 64, **bf)               # pool(relu(fine/first))[...,:63] ++ coarse  (src/models.py:246)
        # derived pool-embedded fine/first filter (params.fine_first_embedded) and its index maps
        self.wbig = z(*FINE_FIRST_EMBEDDED_SHAPE, **bf)
        km, bm = fine_first_index_maps(self.arena.specs["fine/first/conv2d/kernel"],
                                       self.arena.specs["fine/first/conv2d/bias"])
        self.emb_k, self.emb_b = km.to(self.dev), bm.to(self.dev)
        self.f2 = z(B, 55, 74, 64, **bf)
        self.fine = z(B, N_PIX, **f32)
        self.loss_coarse, self.loss_fine = z(1, **f32), z(1, **f32)
        self.lps_coarse, self.lps_fine = z(B, **f32), z(B, **f32)
        self.step_dev = torch.zeros(1, dtype=torch.int64, device=self.dev)
        self.lr_dev = {g: z(1, **f32) for g in ADAM_LR}
        # ---- conv descriptors (src/models.py:211-223, 241-251)
        cd = ops.conv_desc
        self.d_c0 = cd(B, IN_H // 4, IN_W // 4, 64, 96, 3, 3, 1, "valid", impl=impl)   # 11x11x3 s4 as 3x3x64 s1
        self.d_c1 = cd(B, 27, 37, 128, 256, 5, 5, 1, "same", impl=impl)
        self.d_c2 = cd(B, 13, 18, 256, 384, 3, 3, 1, "same", impl=impl)
        self.d_c3 = cd(B, 13, 18, 384, 384, 3, 3, 1, "same", impl=impl)
        self.d_c4 = cd(B, 13, 18, 384, 256, 3, 3, 2, "valid", impl=impl)
        # 9x9x3 s2 -> 63 + pool 2x2 as 3x3x64 s1 -> 4 x 64 with the pool in the GEMM epilogue (writes `cat`)
        self.d_f1 = cd(B, IN_H // 4, IN_W // 4, 64, 256, 3, 3, 1, "valid", ldy=64, impl=impl)
        self.d_f1w = cd(B, IN_H // 4, IN_W // 4, 64, 256, 3, 3, 1, "valid", impl=impl)      # its wgrad: dy [.,256]
        self.d_f2 = cd(B, 55, 74, 64, 64, 5, 5, 1, "same", impl=impl)
        self.d_f3 = cd(B, 55, 74, 64, 1, 5, 5, 1, "same", impl=impl)
        assert (self.d_c0.P, self.d_c0.Q) == (55, 74) and (self.d_f1.P, self.d_f1.Q) == (55, 74)
        assert (self.d_c4.P, self.d_c4.Q) == (6, 8)
        if train:
            self.g_coarse = z(B, 4096, **bf)             # row stride padded 4070 -> 4096 (16-byte aligned rows)
            self.g_fine = z(B, N_PIX, **bf)
            self.g_d0a, self.g_d0 = z(B, 4096, **bf), z(B, 4096, **bf)
            self.g_c4a, self.g_c4 = z(B, 6, 8, 256, **bf), z(B, 6, 8, 256, **bf)
            self.g_c3a, self.g_c3 = z(B, 13, 18, 384, **bf), z(B, 13, 18, 384, **bf)
            self.g_c2a, self.g_c2 = z(B, 13, 18, 384, **bf), z(B, 13, 18, 384, **bf)
            self.g_p1 = z(B, 13, 18, 256, **bf)
            self.g_c1 = z(B, 27, 37, 256, **bf)
            self.g_p0 = z(B, 27, 37, 128, **bf)
            self.g_c0 = z(B, 55, 74, 96, **bf)
            self.g_f2a, self.g_f2 = z(B, 55, 74, 64, **bf), z(B, 55, 74, 64, **bf)
            self.g_cat = z(B, 55, 74, 64, **bf)
            self.g_f1big = None                          # [B*4070, 256] bf16, allocated on first use (phase 2 only)
            self.g_wbig = None
        if self.fp8:
            def e4(*shape):                                   # E4M3 codes, zero-filled as bytes
                return torch.zeros(*shape, dtype=torch.uint8, device=self.dev).view(torch.float8_e4m3fn)
            self.img4q = e4(B, IN_H // 4, IN_W // 4, 64)
            self.p0q, self.p1q = e4(B, 27, 37, 128), e4(B, 13, 18, 256)
            self.c2q, self.c3q = e4(B, 13, 18, 384), e4(B, 13, 18, 384)
            self.c4q, self.d0q, self.catq = e4(B, 12288), e4(B, 4096), e4(B, 55, 74, 64)
            self.s_img = torch.full((B,), 2.0 ** -8, **f32)            # the resized image lies in [0, 1]: fixed scale
            self.s_p0, self.s_p1, self.s_c2, self.s_c3, self.s_c4, self.s_d0, self.s_cat = (z(B, **f32) for _ in range(7))
            # E4M3 weights and their row scales, rebuilt from the bf16 mirror by refresh_derived (outside the arena)
            self.wq = {}
            for name, t in self._fp8_weight_sources().items():
                self.wq[name] = (e4(*t.shape), z(t.shape[0], **f32))
            self.refresh_derived()
        self._graphs = {}
        if os.environ.get("A3D_TIMELINE") == "1" and ctx.timeline is None:
            ctx.timeline = ops.StepTimeline(self.dev)

    # ------------------------------------------------------------------ parameters
    def _real_rows(self, buf, name):
        """Arena view of a variable; dense kernels whose output rows are padded (dense_1: 4070 -> 4096) are cut to
        their real rows (a contiguous prefix), which is what the GEMM entry points take as N."""
        s = self.arena.specs[name]
        t = self.arena.view(buf, name)
        return t[:s.tf_shape[1]] if s.kind == "dense_kernel" else t

    def w(self, name):
        """The operand copy of a kernel: the bf16 mirror, or (TF32 mode) the float32 master itself."""
        return self._real_rows(self.arena.w if self.tf32 else self.arena.wb, name)

    def bias(self, name):
        return self.arena.view(self.arena.w, name + "/bias")

    def gw(self, name):
        return self._real_rows(self.arena.g, name)

    def load_params(self, tf_params):
        self.arena.load_tf(tf_params)
        self.refresh_derived()

    def refresh_derived(self):
        """Re-embed the canonical fine/first filter into the pool-fused filter the kernels read (after a load or a
        FineA optimizer step).  Entries outside the four embedded copies stay zero."""
        a = self.arena
        s = a.specs["fine/first/conv2d/kernel"]
        self.ctx.scatter_cast_bf16(a.w[s.offset:s.offset + s.numel], self.emb_k, self.wbig)
        if self.fp8:
            for name, t in self._fp8_weight_sources().items():
                self.ctx.quantize_rows_e4m3(t, *self.wq[name])

    def _fp8_weight_sources(self):
        """The bf16 operand matrices the FP8 mode quantises per output row (name -> [rows, ...] bf16)."""
        K = "/kernel"
        src = {n: self.w(n + K) for n in ["coarse/conv/conv2d_%d" % i for i in range(5)] +
               ["coarse/dense/dense_0", "coarse/dense/dense_1", "fine/second/conv2d"]}
        src["fine/first/conv2d"] = self.wbig
        return src

    def flush(self):
        """Data parallel: make the bf16 weight mirror current on this rank (rows other ranks updated in the last step are
        otherwise fetched at the start of the next one).  Collective: every rank must call it."""
        if self.comm:
            self.comm.flush(self)

    def export_params(self):
        return self.arena.export_tf()

    def export_grads(self):
        return self.arena.export_tf(self.arena.g)

    def set_dropout_mask(self, mask):
        """Parity hook: use an externally supplied keep-mask [B,4096] instead of the device RNG."""
        self.keep_mask.copy_(mask.to(torch.uint8))
        self.external_mask = True

    def set_augment_params(self, params):
        """Parity hook: use explicit augmentation parameters [B,16] (include/a3d.h A3D_AUG_*) instead of the device
        draw."""
        if self.augment is None:
            raise ValueError("set_augment_params needs a net built with augment=Augment(...)")
        self.aug_params.copy_(params.to(torch.float32))
        self.external_aug = True

    def _augment_draw(self):
        if not self.external_aug:
            self.ctx.augment_draw(self.aug_desc, self.aug_params, self.augment_seed, self.step_dev)

    def _resize_image(self):
        if self.augment is not None:
            self.ctx.resize_affine_tf1_s2d(self.images, IN_H, IN_W, 4, self.aug_params, out=self.img4)
        else:
            self.ctx.resize_bilinear_tf1_s2d(self.images, IN_H, IN_W, 4, out=self.img4)

    def _resize_target(self):
        if self.augment is not None:
            self.ctx.resize_affine_tf1(self.depths, OUT_H, OUT_W, self.aug_params, depth=True, out=self.tar)
        else:
            self.ctx.resize_bilinear_tf1(self.depths, OUT_H, OUT_W, out=self.tar)

    # ------------------------------------------------------------------ forward
    def forward(self, lanes=None):
        """src/models.py:281-290.  Reads self.images / self.depths, fills self.coarse / self.fine / losses.  `lanes`: the
        step's stream placement (_Lanes); by default every launch runs on the current stream."""
        if self.fp8:
            return self._forward_fp8()
        self.ctx.tf32x3 = self.x3
        try:
            self._forward(lanes or _SEQUENTIAL)
        finally:
            self.ctx.tf32x3 = False

    def _forward(self, s):
        c, B = self.ctx, self.B
        K = "/kernel"
        if self.augment is not None:
            self._augment_draw()                        # the transform both resizes apply
            s.mark("draw")
        self._resize_image()
        c.stamp("resize done")
        s.mark("img")
        with s.lane("fine", "draw"):
            self._resize_target()
        # coarse (src/models.py:208-236)
        n = "coarse/conv/conv2d_"
        c.conv2d_fwd(self.d_c0, self.img4, self.w(n + "0" + K), self.bias(n + "0"), relu=True, out=self.c0)
        if self.c0.dtype == torch.bfloat16:            # inference: bf16 pool, no routing record
            c.maxpool2x2_fwd(self.c0, out=self.p0, ldy=self.p0.shape[-1])
        else:
            c.maxpool2x2_fwd_f32(self.c0, out=self.p0, idx=self.i0)
        c.conv2d_fwd(self.d_c1, self.p0, self.w(n + "1" + K), self.bias(n + "1"), relu=True, out=self.c1)
        if self.c1.dtype == torch.bfloat16:
            c.maxpool2x2_fwd(self.c1, out=self.p1)
        else:
            c.maxpool2x2_fwd_f32(self.c1, out=self.p1, idx=self.i1)
        c.conv2d_fwd(self.d_c2, self.p1, self.w(n + "2" + K), self.bias(n + "2"), relu=True, out=self.c2)
        c.conv2d_fwd(self.d_c3, self.c2, self.w(n + "3" + K), self.bias(n + "3"), relu=True, out=self.c3)
        c.conv2d_fwd(self.d_c4, self.c3, self.w(n + "4" + K), self.bias(n + "4"), relu=True, out=self.c4)
        c.stamp("coarse conv fwd done")
        mask = None
        if self.train:
            with s.lane("fine"):
                if not self.external_mask:
                    c.bernoulli_mask(self.keep_mask, 0.5, self.dropout_seed, self.step_dev)
                s.mark("aux")
                if s.on:
                    # flipped filters of the stride-1 dgrads (weights are final since the previous step's Adam): three
                    # small transposes that would otherwise sit inside the dgrad chain
                    flip = (("3", self.d_c3), ("2", self.d_c2), ("1", self.d_c1))
                    if self._wflip is None:
                        self._wflip = {i: c.conv2d_dgrad_prepare(d, self.w(n + i + K)) for i, d in flip}
                    for i, d in flip:
                        c.conv2d_dgrad_prepare(d, self.w(n + i + K), out=self._wflip[i])
                    s.mark("flip")
            mask = self.keep_mask
        s.wait("aux", "published")
        n = "coarse/dense/dense_"
        c.dense_fwd(self.c4.view(B, 12288), self.w(n + "0" + K), self.bias(n + "0"), flags=L.EPI_RELU, keep_mask=mask,
                    drop_rate=0.5, out=self.d0, impl=self.impl)
        c.dense_fwd(self.d0, self.w(n + "1" + K), self.bias(n + "1"), flags=0, out=self.coarse, impl=self.impl)
        c.stamp("dense fwd done")
        s.mark("coarse")
        # fine (src/models.py:238-253): the first conv + pool needs only the image, the rest the coarse map too
        with s.lane("fine", "img"):
            c.conv2d_pool4_fwd(self.d_f1, self.img4, self.wbig, self.bias("fine/first/conv2d"), relu=True, out=self.cat,
                               idx=self.if1 if self.train else None)
            c.stamp("fine/first done")
            s.wait("coarse")
            c.scatter_channel_bf16(self.coarse, self.cat, 63)
            c.conv2d_fwd(self.d_f2, self.cat, self.w("fine/second/conv2d" + K), self.bias("fine/second/conv2d"),
                         relu=True, out=self.f2)
            c.conv2d_fwd(self.d_f3, self.f2, self.w("fine/third" + K), self.bias("fine/third"), relu=False,
                         out=self.fine.view(B, 55, 74, 1))
        # losses (src/models.py:288-290); the gradient of the active branch is produced in the same pass
        gk = "dout" if self.tf32 else "dout_bf16"          # the gradient w.r.t. the prediction, in the storage type
        self._loss(self.coarse, loss_ps=self.lps_coarse, loss=self.loss_coarse, dout_ld=4096,
                   **{gk: self.g_coarse if self.train else None})
        with s.lane("fine"):
            self._loss(self.fine, loss_ps=self.lps_fine, loss=self.loss_fine, dout_ld=N_PIX,
                       **{gk: self.g_fine if self.train else None})
            c.stamp("fine fwd + loss done")

    def _loss(self, pred, **kw):
        """The loss of one map [B, 4070] against the resized target (and its gradient where `kw` names a buffer)."""
        if self.loss == "ssi":
            self.ctx.ssi_loss(pred, self.tar, OUT_H, OUT_W, SSI_ALPHA, SSI_SCALES, want_grad=False, **kw)
        else:
            self.ctx.silog_loss(pred, self.tar, LAMBDA_OVER_N, want_grad=False, **kw)

    def _forward_fp8(self):
        """The inference forward on E4M3 operands.  Storage points (oracle/fp8.py restates them): the resized image with
        the fixed scale 2^-8; max-pool of the bf16 conv2d_0 / conv2d_1 outputs, conv2d_2..4, dense_0 and the concat
        (bf16) with one scale per image; `coarse` f32, `f2` bf16 and fine/third as in the bf16 mode."""
        c, B, wq = self.ctx, self.B, self.wq
        c.resize_bilinear_tf1_s2d_e4m3(self.images, IN_H, IN_W, out=self.img4q)
        self._resize_target()
        n = "coarse/conv/conv2d_"
        c.conv2d_fwd_fp8(self.d_c0, self.img4q, self.s_img, *wq[n + "0"], self.bias(n + "0"), relu=True, out=self.c0)
        c.maxpool2x2_quantize_e4m3(self.c0, out=self.p0q, scale=self.s_p0)
        c.conv2d_fwd_fp8(self.d_c1, self.p0q, self.s_p0, *wq[n + "1"], self.bias(n + "1"), relu=True, out=self.c1)
        c.maxpool2x2_quantize_e4m3(self.c1, out=self.p1q, scale=self.s_p1)
        c.conv2d_fwd_fp8(self.d_c2, self.p1q, self.s_p1, *wq[n + "2"], self.bias(n + "2"), relu=True, out=self.c2)
        c.quantize_e4m3(self.c2, out=self.c2q, scale=self.s_c2)
        c.conv2d_fwd_fp8(self.d_c3, self.c2q, self.s_c2, *wq[n + "3"], self.bias(n + "3"), relu=True, out=self.c3)
        c.quantize_e4m3(self.c3, out=self.c3q, scale=self.s_c3)
        c.conv2d_fwd_fp8(self.d_c4, self.c3q, self.s_c3, *wq[n + "4"], self.bias(n + "4"), relu=True, out=self.c4)
        c.quantize_e4m3(self.c4.view(B, 12288), out=self.c4q, scale=self.s_c4)
        n = "coarse/dense/dense_"
        c.dense_fwd_fp8(self.c4q, self.s_c4, *wq[n + "0"], self.bias(n + "0"), flags=L.EPI_RELU, out=self.d0)
        c.quantize_e4m3(self.d0, out=self.d0q, scale=self.s_d0)
        c.dense_fwd_fp8(self.d0q, self.s_d0, *wq[n + "1"], self.bias(n + "1"), flags=0, out=self.coarse)
        c.conv2d_pool4_fwd_fp8(self.d_f1, self.img4q, self.s_img, *wq["fine/first/conv2d"], self.bias("fine/first/conv2d"),
                               relu=True, out=self.cat)
        c.scatter_channel_bf16(self.coarse, self.cat, 63)
        c.quantize_e4m3(self.cat, out=self.catq, scale=self.s_cat)
        c.conv2d_fwd_fp8(self.d_f2, self.catq, self.s_cat, *wq["fine/second/conv2d"], self.bias("fine/second/conv2d"),
                         relu=True, out=self.f2)
        c.conv2d_fwd(self.d_f3, self.f2, self.w("fine/third/kernel"), self.bias("fine/third"), relu=False,
                     out=self.fine.view(B, 55, 74, 1))
        self._loss(self.coarse, loss_ps=self.lps_coarse, loss=self.loss_coarse)
        self._loss(self.fine, loss_ps=self.lps_fine, loss=self.loss_fine)

    # ------------------------------------------------------------------ backward
    def _dense_wgrad_adam(self, layer, x, dy):
        """Weight gradient + TF-Adam of one dense kernel in a single pass (the gradient never reaches HBM); the bias
        gradient is produced as usual and gets its own (tiny) Adam launch.  Must run AFTER the layer's dgrad, the
        last reader of the weights it overwrites."""
        c, a, g = self.ctx, self.arena, "CoarseDense"
        kn, bn_ = "coarse/dense/dense_" + layer + "/kernel", "coarse/dense/dense_" + layer + "/bias"
        rr = self._real_rows
        c.stamp(f"dense_{layer} wgrad+adam begin")
        c.dense_wgrad_adam(x, dy, self.gw(bn_), rr(a.w, kn), rr(a.m, kn), rr(a.v, kn), rr(a.wb, kn),
                           ADAM_LR[g], ADAM_BETA1, self.beta2, ADAM_EPS, max(self.adam_t[g], 1), 1.0,
                           lr_t_dev=self.lr_dev[g])
        s = a.specs[bn_]
        self.adam_range(g, s.offset, s.offset + s.size)
        c.stamp(f"dense_{layer} wgrad+adam end")

    def backward_coarse(self, fused_dense_adam=False, lanes=None):
        """d loss_coarse / d coarse variables (compute_gradients of src/models.py:319-324).  With
        `fused_dense_adam` the two dense kernels are updated on the spot (see _dense_wgrad_adam) and the caller
        applies Adam to the CoarseConv group only.  On four streams (`lanes`) every weight gradient runs as soon as its dY
        exists and each optimizer group's update right behind its last weight gradient, so the HBM-bound Adam of the
        67 M dense parameters and the small-grid wgrad kernels run under the tensor-bound dgrad chain."""
        c, B, K, comm = self.ctx, self.B, "/kernel", self.comm
        s = lanes or _SEQUENTIAL
        hook = comm.bucket_ready if comm and not s.on else (lambda *_: None)   # sequential DP: allreduce now, Adam later
        n = "coarse/dense/dense_"
        # data parallel on four streams, dense layers: exchange activations instead of gradients where the gathered batch
        # allows it (dp.dense_gather_adam_merged), else reduce-scatter -> sharded TF-Adam -> all-gather (dp.sharded_adam)
        gather = s.on and comm and all(comm.can_gather_dense(self, n + l + K, B) for l in "01")
        sharded = s.on and comm and not gather
        s.mark("loss")
        if not fused_dense_adam and not gather:
            with s.lane("wgrad", "loss"):
                c.dense_wgrad(self.d0, self.g_coarse, dw=self.gw(n + "1" + K), db=self.gw(n + "1/bias"), impl=self.impl)
            hook(self, "dense_1")
        # dropout grad (mask * 1/(1-rate)) and relu grad (d0 > 0) ride in the dgrad's finishing pass
        c.dense_dgrad_act(self.g_coarse, self.w(n + "1" + K), self.d0, self.keep_mask, 0.5, L.EPI_RELU, out=self.g_d0,
                          impl=self.impl)
        s.mark("dgrad dense_1")          # the last reader of dense_1's weights: its update may follow
        if sharded:
            with s.lane("wgrad"):
                self._sharded_adam("1", s.event("dgrad dense_1"))
        with s.lane("wgrad", "dgrad dense_1"):
            if fused_dense_adam:
                self._dense_wgrad_adam("1", self.d0, self.g_coarse)
            elif not gather:
                c.dense_wgrad(self.c4.view(B, 12288), self.g_d0, dw=self.gw(n + "0" + K), db=self.gw(n + "0/bias"),
                              impl=self.impl)
                hook(self, "dense_0")
        c.dense_dgrad_act(self.g_d0, self.w(n + "0" + K), self.c4.view(B, 12288), None, 0.0, L.EPI_RELU,
                          out=self.g_c4.view(B, 12288), impl=self.impl)
        s.mark("dgrad dense_0")
        if gather:       # one all-gather of both layers' activations; each row update waits for its layer's dgrad
            g_ = "CoarseDense"
            comm.dense_gather_adam_merged(
                self, [(n + "1" + K, n + "1/bias", self.d0, self.g_coarse, s.event("dgrad dense_1")),
                       (n + "0" + K, n + "0/bias", self.c4.view(B, 12288), self.g_d0, s.event("dgrad dense_0"))],
                g_, ADAM_LR[g_], ADAM_BETA1, ADAM_EPS, ready=s.event("dgrad dense_1"))
        elif sharded:
            with s.lane("wgrad"):
                self._sharded_adam("0", s.event("dgrad dense_0"))
        c.stamp("dense dgrad done")
        with s.lane("wgrad", "dgrad dense_0"):
            if fused_dense_adam:
                self._dense_wgrad_adam("0", self.c4.view(B, 12288), self.g_d0)
            elif s.on and not comm:      # under the conv backward, behind the last readers of the dense weights
                self.apply_adam(("CoarseDense",))
        n = "coarse/conv/conv2d_"
        # The bias gradients (latency-bound column sums of dY, 7-10 us each) run on the fine stream, whose forward work is
        # long done by then: next to the wgrad GEMMs, not before them.  (Data parallel on four streams: measured slower at
        # 2 GPUs, 1.184 vs 1.144 ms -- the comm stream's NCCL kernels already fill those gaps -- so there the conv wgrads
        # keep their bias gradients.)
        side_bias = not (s.on and comm)

        def wgrad(desc, x, dy, name, after):
            if side_bias:
                with s.lane("fine", after):
                    c.bias_grad_bf16(dy.view(-1, dy.shape[-1]), dy.shape[-1], self.gw(name + "/bias"))
            with s.lane("cwgrad", after):
                c.conv2d_wgrad(desc, x, dy, dw=self.gw(name + K), db=None if side_bias else self.gw(name + "/bias"))
        flip = self._wflip if s.on else {}
        wgrad(self.d_c4, self.c3, self.g_c4, n + "4", "dgrad dense_0")
        c.conv2d_dgrad(self.d_c4, self.g_c4, self.w(n + "4" + K), out=self.g_c3, relu_src=self.c3)
        c.stamp("dgrad conv2d_4 done")
        s.mark("g_c3")
        wgrad(self.d_c3, self.c2, self.g_c3, n + "3", "g_c3")
        s.wait("flip")
        c.conv2d_dgrad(self.d_c3, self.g_c3, self.w(n + "3" + K), out=self.g_c2, relu_src=self.c2, wflip=flip.get("3"))
        s.mark("g_c2")
        wgrad(self.d_c2, self.p1, self.g_c2, n + "2", "g_c2")
        c.conv2d_dgrad(self.d_c2, self.g_c2, self.w(n + "2" + K), out=self.g_p1, wflip=flip.get("2"))
        c.maxpool2x2_idx_bwd(self.i1, self.g_p1, (self.B, 27, 37, 256), out=self.g_c1)
        c.stamp("dgrad conv2d_3,2 + pool bwd done")
        s.mark("g_c1")
        # (DP: exchanging conv2d_4..2 here as an early bucket was measured SLOWER at 2 GPUs, 1.30 vs 1.26 ms: three more
        # NCCL launches cost more than the shorter tail saves)
        wgrad(self.d_c1, self.p0, self.g_c1, n + "1", "g_c1")
        with s.lane("cwgrad"):
            s.mark("wgrad conv2d_1")                       # gradients of conv2d_4 .. conv2d_1 are complete
        c.conv2d_dgrad(self.d_c1, self.g_c1, self.w(n + "1" + K), out=self.g_p0, wflip=flip.get("1"))
        c.maxpool2x2_idx_bwd(self.i0, self.g_p0, (self.B, 55, 74, 96), out=self.g_c0)
        c.stamp("dgrad conv2d_1 + pool bwd done")
        s.mark("g_c0")
        # On four streams the CoarseConv update is cut at conv2d_0.  Single GPU: TF-Adam of conv2d_4 .. conv2d_1 (99 % of
        # the group) runs on the idle fine stream next to conv2d_0's weight gradient; only conv2d_0's 55 k parameters are
        # updated in the step's tail.  The group is one contiguous arena range in backward order, so this is the same
        # update as one launch.
        # Data parallel, the same cut: conv2d_4 .. conv2d_1 are all-reduced in f32 and updated behind conv2d_1's weight
        # gradient, under conv2d_1's dgrad, the pool backward and conv2d_0's wgrad; the step's tail exchanges conv2d_0's
        # 55 k parameters only.  (8 GPUs, profiles/step_timeline_r02_n8_rank0.json: the single 16 MB allreduce + Adam was
        # ~150 us of exposed tail.)  f32 allreduce + replicated Adam beats cast + reduce-scatter + sharded Adam +
        # all-gather at every world size (4 GPUs: 1.160 vs 1.185 ms; 2 GPUs, with the split: 0.972 vs 1.015 ms -- the
        # collectives are latency-bound at 8-16 MB and the sharded form needs three of them); a sharded exchange of the
        # split measured 1.20 against 1.18 ms unsplit at 2 GPUs (the extra NCCL kernels take SM slots from the GEMMs
        # they overlap with).
        lo, hi = self.arena.group_range("CoarseConv")
        cut = self.arena.specs["coarse/conv/conv2d_0/kernel"].offset
        inv_world = 1.0 / comm.world if comm else 1.0

        def adam_cc(lo, hi):
            self.adam_range("CoarseConv", lo, hi, inv_world)
        if s.on and comm:
            with s.lane("cwgrad"):
                comm.bucket_ready(self, "coarse_conv_main", after=s.event("g_c0"), then=adam_cc)
        elif s.on:       # conv2d_1's dgrad was the last reader of these weights
            with s.lane("fine", "wgrad conv2d_1", "g_c0"):
                adam_cc(lo, cut)
        if side_bias:
            with s.lane("fine", "g_c0"):
                c.bias_grad_bf16(self.g_c0.view(-1, 96), 96, self.gw(n + "0/bias"))
                s.mark("bias conv2d_0")
        with s.lane("cwgrad", "g_c0"):
            c.stamp("conv2d_0 wgrad + conv exchange/adam begin")
            c.conv2d_wgrad(self.d_c0, self.img4, self.g_c0, dw=self.gw(n + "0" + K),
                           db=None if side_bias else self.gw(n + "0/bias"))
            s.wait("bias conv2d_0")
            self._mask_padding("coarse/conv/conv2d_0/kernel")
            if s.on and comm:
                comm.bucket_ready(self, "coarse_conv_0", then=adam_cc)
                comm.wait_all(self)
            elif s.on:
                adam_cc(cut, hi)
            c.stamp("conv2d_0 wgrad + conv exchange/adam end")
        hook(self, "coarse_conv")

    def _sharded_adam(self, layer, after):
        g = "CoarseDense"
        self.comm.sharded_adam(self, "dense_" + layer, g, ADAM_LR[g], ADAM_BETA1, ADAM_EPS, after)

    def backward_fine(self):
        """d loss_fine / d fine variables (src/models.py:334-338); the coarse map is a constant input."""
        c, K = self.ctx, "/kernel"
        hook = self.comm.bucket_ready if self.comm else (lambda *_: None)
        c.conv2d_wgrad(self.d_f3, self.f2, self.g_fine.view(self.B, 55, 74, 1), dw=self.gw("fine/third" + K),
                       db=self.gw("fine/third/bias"))
        c.conv2d_dgrad(self.d_f3, self.g_fine.view(self.B, 55, 74, 1), self.w("fine/third" + K), out=self.g_f2,
                       relu_src=self.f2)
        c.conv2d_wgrad(self.d_f2, self.cat, self.g_f2, dw=self.gw("fine/second/conv2d" + K),
                       db=self.gw("fine/second/conv2d/bias"))
        c.conv2d_dgrad(self.d_f2, self.g_f2, self.w("fine/second/conv2d" + K), out=self.g_cat)
        # fine/first: MaxPoolGrad + ReluGrad on the 4 x 64 GEMM columns, wgrad of the embedded filter, then fold its
        # four copies (and the four bias groups) into the canonical variable
        if self.g_f1big is None:
            self.g_f1big = torch.zeros(self.B * N_PIX, 256, dtype=self.cat.dtype, device=self.dev)
            self.g_wbig = torch.zeros(256 * 3 * 3 * 64 + 256, dtype=torch.float32, device=self.dev)
        c.pool4_bwd(self.g_cat.view(-1, 64), self.cat.view(-1, 64), self.if1, out=self.g_f1big)
        nk = 256 * 3 * 3 * 64
        c.conv2d_wgrad(self.d_f1w, self.img4, self.g_f1big.view(self.B, 55, 74, 256),
                       dw=self.g_wbig[:nk].view(256, 3, 3, 64), db=self.g_wbig[nk:])
        c.gather_sum_f32(self.g_wbig[:nk], self.emb_k, self.gw("fine/first/conv2d" + K))
        c.gather_sum_f32(self.g_wbig[nk:], self.emb_b, self.gw("fine/first/conv2d/bias"))
        hook(self, "fine")

    def _mask_padding(self, name):
        m = self.arena.masks.get(name)
        if m is not None:
            s = self.arena.specs[name]
            self.ctx.apply_mask_f32(self.arena.g[s.offset:s.offset + s.numel], m)

    # ------------------------------------------------------------------ optimizer
    def apply_adam(self, groups, grad_scale=1.0):
        """apply_gradients of the two Adam instances of the active branch (src/models.py:326-331,340-345)."""
        for g in groups:
            self.adam_range(g, *self.arena.group_range(g), grad_scale)

    def adam_range(self, group, lo, hi, grad_scale=1.0):
        a = self.arena
        self.ctx.adam_tf(a.w[lo:hi], a.g[lo:hi], a.m[lo:hi], a.v[lo:hi], a.wb[lo:hi], ADAM_LR[group], ADAM_BETA1,
                         self.beta2, ADAM_EPS, max(self.adam_t[group], 1), grad_scale, lr_t_dev=self.lr_dev[group])

    # ------------------------------------------------------------------ one session.run(model_op)
    def _enqueue_step(self, phase):
        s = _Lanes(self) if phase == 1 and self.overlap else _SEQUENTIAL
        with s:
            c = self.ctx
            if c.timeline is not None:
                c.timeline.begin()
            c.stamp("step begin")
            if self.comm and s.on:
                # the dense rows other ranks updated in the PREVIOUS step arrive now, under this step's resize and
                # convolution forward (dp.dense_gather_adam_merged / publish_rows); the dense forward waits for them
                s.events["published"] = self.comm.publish_rows(self)
            elif self.comm:
                self.comm.flush(self)                   # rows updated by a previous (overlapped) step
            self.forward(s)
            groups = ()
            if phase == 1:
                fused = self.fuse_dense_adam and not self.comm
                self.backward_coarse(fused_dense_adam=fused, lanes=s)
                if not s.on:                            # on four streams each group was updated behind its wgrads
                    groups = ("CoarseConv",) if fused else ("CoarseDense", "CoarseConv")
            elif phase == 2:
                self.backward_fine()
                groups = ("FineA", "FineB")
            if groups:
                scale = 1.0
                if self.comm:
                    self.comm.wait_all(self)
                    scale = 1.0 / self.comm.world
                self.apply_adam(groups, scale)
                if "FineA" in groups:
                    self.refresh_derived()               # fine/first moved: re-embed it into the pool-fused filter
            s.join()
            c.increment_i64(self.step_dev)              # global_step += 1 (src/models.py:329,343,356)
            c.stamp("step end")

    def _ensure_graph(self, phase):
        """Warm-up launch outside capture (sets function attributes, allocates workspaces, autotunes first-use shapes;
        its side effects on the variables are rolled back), then capture of the phase's step in a CUDA graph."""
        gr = self._graphs.get(phase)
        if gr is None:
            saved = (self.arena.w.clone(), self.arena.m.clone(), self.arena.v.clone(), self.arena.wb.clone(),
                     self.step_dev.clone())
            self._enqueue_step(phase)
            torch.cuda.synchronize()
            self.arena.w.copy_(saved[0]); self.arena.m.copy_(saved[1]); self.arena.v.copy_(saved[2])
            self.arena.wb.copy_(saved[3]); self.step_dev.copy_(saved[4])
            self.refresh_derived()
            gr = torch.cuda.CUDAGraph()
            with torch.cuda.graph(gr):
                self._enqueue_step(phase)
            self._graphs[phase] = gr        # the capture itself does not execute
        return gr

    def train_step(self, use_graph=True):
        """One `session.run(model_op)` of the reference loop (src/ann3depth.py:126-127)."""
        assert self.train
        phase = phase_of(self.global_step, self.B)
        groups = {1: ("CoarseDense", "CoarseConv"), 2: ("FineA", "FineB"), 3: ()}[phase]
        for g in groups:                                   # each Adam instance owns its beta-power state
            self.adam_t[g] += 1
            self.lr_dev[g].fill_(ops.adam_lr_t(ADAM_LR[g], ADAM_BETA1, self.beta2, self.adam_t[g]))
        # Data parallel: the warm-up launch in front of a capture executes one extra set of collectives.  EVERY rank
        # therefore captures on its first step of a phase, also a rank whose step is about to run un-graphed (the chief's
        # traced first step, summary.TraceHook): otherwise its peers' warm-up collectives would pair with its real ones
        # and every later collective would be off by one step.
        if use_graph or self.comm is not None:
            gr = self._ensure_graph(phase)
        if use_graph:
            gr.replay()
        else:
            self._enqueue_step(phase)
        self.global_step += 1
        return phase

    def infer(self):
        """Inference = coarse + fine with train=False (dropout off), src/models.py:230,278,286."""
        self.forward()
        return self.fine.view(self.B, OUT_H, OUT_W, 1)
