"""MSDN (Eigen et al. 2014) train / inference step on liba3d -- host-side orchestration.

Mirrors `_MultiScaleDeepNetwork` of the reference (src/models.py:203-367): preprocessing resize,
coarse stack, fine stack, two scale-invariant log losses, and the three-phase schedule with four
TF-Adam instances.  Every arithmetic operation is a liba3d kernel launched on the current CUDA
stream; PyTorch only owns the buffers.  The whole step is captured in a CUDA graph per phase.
"""
from __future__ import annotations

import os

import torch

from . import _lib as L
from . import ops
from .params import Arena, msdn_specs, fine_first_index_maps, FINE_FIRST_EMBEDDED_SHAPE

IN_H, IN_W = 228, 304          # src/models.py:282
OUT_H, OUT_W = 55, 74          # src/models.py:283
N_PIX = OUT_H * OUT_W          # 4070 == the 74*55 of src/models.py:269
LAMBDA_OVER_N = 0.5 / (74 * 55)

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


class MSDNNet:
    """Buffers + launch sequence for one replica with a static batch size (the reference requires a
    static batch dimension too: `int(images.shape[0])`, src/models.py:225,256,299)."""

    def __init__(self, ctx: ops.Context, batch: int, in_hw=(480, 640), depth_hw=(55, 73), train=True,
                 beta2=ADAM_BETA2_REFERENCE, impl=L.IMPL_AUTO, dropout_seed=2, comm=None, grad_dtype=torch.float32,
                 overlap=True, fuse_dense_adam=True, dtype="bf16", augment=None, augment_seed=3):
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
        self.overlap = overlap                # phase-1 step on several streams (see _enqueue_phase1_overlapped)
        # single GPU: the dense weight gradients (32 FMAs per parameter at batch 32) are recomputed on the CUDA cores
        # inside the HBM-bound TF-Adam pass (a3d_dense_wgrad_adam), so the 67 M-element f32 gradient is never written
        # or re-read: 26 instead of 38 bytes per dense parameter and step.  Data parallel runs need the gradient in
        # memory for the reduce-scatter and keep the separate kernels (dp.py shards the optimizer instead).
        self.fuse_dense_adam = fuse_dense_adam
        self._s_fine = self._s_wgrad = self._s_cwgrad = None
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
    def forward(self):
        """src/models.py:281-290.  Reads self.images / self.depths, fills self.coarse / self.fine / losses."""
        if self.fp8:
            return self._forward_fp8()
        self.ctx.tf32x3 = self.x3
        try:
            self._forward()
        finally:
            self.ctx.tf32x3 = False

    def _forward(self):
        c, B = self.ctx, self.B
        K = "/kernel"
        if self.augment is not None:
            self._augment_draw()
        self._resize_image()
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
        mask = None
        if self.train:
            if not self.external_mask:
                c.bernoulli_mask(self.keep_mask, 0.5, self.dropout_seed, self.step_dev)
            mask = self.keep_mask
        n = "coarse/dense/dense_"
        c.dense_fwd(self.c4.view(B, 12288), self.w(n + "0" + K), self.bias(n + "0"), flags=L.EPI_RELU, keep_mask=mask,
                    drop_rate=0.5, out=self.d0, impl=self.impl)
        c.dense_fwd(self.d0, self.w(n + "1" + K), self.bias(n + "1"), flags=0, out=self.coarse, impl=self.impl)
        # fine (src/models.py:238-253)
        c.conv2d_pool4_fwd(self.d_f1, self.img4, self.wbig, self.bias("fine/first/conv2d"), relu=True, out=self.cat,
                           idx=self.if1 if self.train else None)
        c.scatter_channel_bf16(self.coarse, self.cat, 63)
        c.conv2d_fwd(self.d_f2, self.cat, self.w("fine/second/conv2d" + K), self.bias("fine/second/conv2d"), relu=True,
                     out=self.f2)
        c.conv2d_fwd(self.d_f3, self.f2, self.w("fine/third" + K), self.bias("fine/third"), relu=False,
                     out=self.fine.view(B, 55, 74, 1))
        # losses (src/models.py:288-290); the gradient of the active branch is produced in the same pass
        gk = "dout" if self.tf32 else "dout_bf16"          # the gradient w.r.t. the prediction, in the storage type
        c.silog_loss(self.coarse, self.tar, LAMBDA_OVER_N, want_grad=False, loss_ps=self.lps_coarse,
                     loss=self.loss_coarse, dout_ld=4096, **{gk: self.g_coarse if self.train else None})
        c.silog_loss(self.fine, self.tar, LAMBDA_OVER_N, want_grad=False, loss_ps=self.lps_fine, loss=self.loss_fine,
                     dout_ld=N_PIX, **{gk: self.g_fine if self.train else None})

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
        c.silog_loss(self.coarse, self.tar, LAMBDA_OVER_N, want_grad=False, loss_ps=self.lps_coarse, loss=self.loss_coarse)
        c.silog_loss(self.fine, self.tar, LAMBDA_OVER_N, want_grad=False, loss_ps=self.lps_fine, loss=self.loss_fine)

    # ------------------------------------------------------------------ backward
    def _dense_wgrad_adam(self, layer, x, dy):
        """Weight gradient + TF-Adam of one dense kernel in a single pass (the gradient never reaches HBM); the bias
        gradient is produced as usual and gets its own (tiny) Adam launch.  Must run AFTER the layer's dgrad, the
        last reader of the weights it overwrites."""
        c, a, g = self.ctx, self.arena, "CoarseDense"
        kn, bn_ = "coarse/dense/dense_" + layer + "/kernel", "coarse/dense/dense_" + layer + "/bias"
        rr = self._real_rows
        c.dense_wgrad_adam(x, dy, self.gw(bn_), rr(a.w, kn), rr(a.m, kn), rr(a.v, kn), rr(a.wb, kn),
                           ADAM_LR[g], ADAM_BETA1, self.beta2, ADAM_EPS, max(self.adam_t[g], 1), 1.0,
                           lr_t_dev=self.lr_dev[g])
        s = a.specs[bn_]
        sl = slice(s.offset, s.offset + s.size)
        c.adam_tf(a.w[sl], a.g[sl], a.m[sl], a.v[sl], a.wb[sl], ADAM_LR[g], ADAM_BETA1, self.beta2, ADAM_EPS,
                  max(self.adam_t[g], 1), 1.0, lr_t_dev=self.lr_dev[g])

    def backward_coarse(self, fused_dense_adam=False):
        """d loss_coarse / d coarse variables (compute_gradients of src/models.py:319-324).  With
        `fused_dense_adam` the two dense kernels are updated on the spot (see _dense_wgrad_adam) and the caller
        applies Adam to the CoarseConv group only."""
        c, B, K = self.ctx, self.B, "/kernel"
        hook = self.comm.bucket_ready if self.comm else (lambda *_: None)
        n = "coarse/dense/dense_"
        if not fused_dense_adam:
            c.dense_wgrad(self.d0, self.g_coarse, dw=self.gw(n + "1" + K), db=self.gw(n + "1/bias"), impl=self.impl)
            hook(self, "dense_1")
        # dropout grad (mask * 1/(1-rate)) and relu grad (d0 > 0) ride in the dgrad's finishing pass
        c.dense_dgrad_act(self.g_coarse, self.w(n + "1" + K), self.d0, self.keep_mask, 0.5, L.EPI_RELU, out=self.g_d0,
                          impl=self.impl)
        if fused_dense_adam:
            self._dense_wgrad_adam("1", self.d0, self.g_coarse)
        else:
            c.dense_wgrad(self.c4.view(B, 12288), self.g_d0, dw=self.gw(n + "0" + K), db=self.gw(n + "0/bias"),
                          impl=self.impl)
            hook(self, "dense_0")
        c.dense_dgrad_act(self.g_d0, self.w(n + "0" + K), self.c4.view(B, 12288), None, 0.0, L.EPI_RELU,
                          out=self.g_c4.view(B, 12288), impl=self.impl)
        if fused_dense_adam:
            self._dense_wgrad_adam("0", self.c4.view(B, 12288), self.g_d0)
        n = "coarse/conv/conv2d_"

        def wgrad(desc, x, dy, name):
            # bias gradient (a column sum of dY, not a tensor-core op) as its own call, like the multi-stream schedule
            # does: bench.py's per-kernel table then times the wgrad GEMM alone
            c.bias_grad_bf16(dy.view(-1, dy.shape[-1]), dy.shape[-1], self.gw(name + "/bias"))
            c.conv2d_wgrad(desc, x, dy, dw=self.gw(name + K), db=None)
        wgrad(self.d_c4, self.c3, self.g_c4, n + "4")
        c.conv2d_dgrad(self.d_c4, self.g_c4, self.w(n + "4" + K), out=self.g_c3, relu_src=self.c3)
        wgrad(self.d_c3, self.c2, self.g_c3, n + "3")
        c.conv2d_dgrad(self.d_c3, self.g_c3, self.w(n + "3" + K), out=self.g_c2, relu_src=self.c2)
        wgrad(self.d_c2, self.p1, self.g_c2, n + "2")
        c.conv2d_dgrad(self.d_c2, self.g_c2, self.w(n + "2" + K), out=self.g_p1)
        c.maxpool2x2_idx_bwd(self.i1, self.g_p1, (self.B, 27, 37, 256), out=self.g_c1)
        wgrad(self.d_c1, self.p0, self.g_c1, n + "1")
        c.conv2d_dgrad(self.d_c1, self.g_c1, self.w(n + "1" + K), out=self.g_p0)
        c.maxpool2x2_idx_bwd(self.i0, self.g_p0, (self.B, 55, 74, 96), out=self.g_c0)
        wgrad(self.d_c0, self.img4, self.g_c0, n + "0")
        self._mask_padding("coarse/conv/conv2d_0/kernel")
        hook(self, "coarse_conv")

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
        a = self.arena
        for g in groups:
            lo, hi = a.group_range(g)
            self.ctx.adam_tf(a.w[lo:hi], a.g[lo:hi], a.m[lo:hi], a.v[lo:hi], a.wb[lo:hi], ADAM_LR[g], ADAM_BETA1,
                             self.beta2, ADAM_EPS, max(self.adam_t[g], 1), grad_scale, lr_t_dev=self.lr_dev[g])

    def adam_range(self, group, lo, hi, grad_scale=1.0):
        a = self.arena
        self.ctx.adam_tf(a.w[lo:hi], a.g[lo:hi], a.m[lo:hi], a.v[lo:hi], a.wb[lo:hi], ADAM_LR[group], ADAM_BETA1,
                         self.beta2, ADAM_EPS, max(self.adam_t[group], 1), grad_scale, lr_t_dev=self.lr_dev[group])

    # ------------------------------------------------------------------ phase-1 step on four streams
    def _enqueue_phase1_overlapped(self):
        """Same launches as forward() + backward_coarse() + apply_adam(), arranged by data dependence:
             main stream : resize, coarse forward, coarse loss, the dgrad chain (the critical path)
             fine stream : fine forward + fine loss (needs only the image and the coarse map)
             wgrad stream: every weight/bias gradient as soon as its dY exists, each optimizer group's
                           gradient allreduce hand-off and TF-Adam right behind its last wgrad
           so the HBM-bound Adam of the 67 M dense parameters and the small-grid wgrad kernels run under the
           tensor-bound dgrad chain instead of after it.  Joins back before global_step += 1.
        The main stream has HIGH PRIORITY: whenever an SM slot frees up, pending CTAs of the chain are placed before those
        of the fine / wgrad / optimizer streams, which fill the remaining slots.  (CUDA graph capture keeps the priority
        as a kernel-node attribute.)"""
        c, B, K = self.ctx, self.B, "/kernel"
        dev = self.dev
        if self._s_fine is None:
            self._s_main = torch.cuda.Stream(device=dev, priority=-1)
            self._s_fine, self._s_wgrad = torch.cuda.Stream(device=dev), torch.cuda.Stream(device=dev)
            self._s_cwgrad = torch.cuda.Stream(device=dev)
        cur = torch.cuda.current_stream()
        e_in = torch.cuda.Event()
        e_in.record(cur)
        # s2: dense wgrads + dense Adam (HBM-bound) ; s3: conv wgrads + conv Adam (tensor / L2-bound)
        s0, s1, s2, s3 = self._s_main, self._s_fine, self._s_wgrad, self._s_cwgrad
        with torch.cuda.stream(s0):
            s0.wait_event(e_in)
            inv_world = 1.0 / self.comm.world if self.comm else 1.0
            if c.timeline is not None:
                c.timeline.begin()
            c.stamp("step begin")
            # data parallel: the dense rows other ranks updated in the PREVIOUS step arrive now, under this step's resize and
            # convolution forward (dp.dense_gather_adam_merged / publish_rows); the dense forward waits for them
            e_pub = self.comm.publish_rows(self) if self.comm else None

            def dp_update(bucket, group, after=None):     # DP: reduce-scatter -> sharded TF-Adam -> all-gather (dp.py)
                self.comm.sharded_adam(self, bucket, group, ADAM_LR[group], ADAM_BETA1, ADAM_EPS, after)
            hook = self.comm.bucket_ready if self.comm else (lambda *_: None)

            def mark(stream):
                e = torch.cuda.Event()
                e.record(stream)
                return e

            # ---- fine stream, part 0: what the critical path needs only later (depth target, dropout mask)
            n0 = "coarse/conv/conv2d_"
            e_start = mark(s0)
            e_draw = None
            if self.augment is not None:             # the transform both resizes apply
                self._augment_draw()
                e_draw = mark(s0)
            for side in (s2, s3):                 # every side stream forks from the step's start (a stream that happens to
                side.wait_event(e_start)          # get no work in some mode must still be part of the capture to be joined)
            with torch.cuda.stream(s1):
                s1.wait_event(e_start)
                if e_draw is not None:
                    s1.wait_event(e_draw)
                self._resize_target()
                if not self.external_mask:
                    c.bernoulli_mask(self.keep_mask, 0.5, self.dropout_seed, self.step_dev)
                e_aux = mark(s1)
                # flipped filters of the stride-1 dgrads (weights are final since the previous step's Adam): three small
                # transposes that used to sit inside the dgrad chain
                if self._wflip is None:
                    self._wflip = {}
                    for i, dsc in (("3", self.d_c3), ("2", self.d_c2), ("1", self.d_c1)):
                        self._wflip[i] = c.conv2d_dgrad_prepare(dsc, self.w(n0 + i + K))
                for i, dsc in (("3", self.d_c3), ("2", self.d_c2), ("1", self.d_c1)):
                    c.conv2d_dgrad_prepare(dsc, self.w(n0 + i + K), out=self._wflip[i])
                e_flip = mark(s1)
            # ---- main: preprocessing
            self._resize_image()
            c.stamp("resize done")
            e_img = mark(s0)
            # ---- fine stream, part 1: first conv + pool need only the image
            with torch.cuda.stream(s1):
                c.ws_tag = "fine"
                s1.wait_event(e_img)
                c.conv2d_pool4_fwd(self.d_f1, self.img4, self.wbig, self.bias("fine/first/conv2d"), relu=True, out=self.cat,
                                   idx=self.if1)
                c.stamp("fine/first done")
                c.ws_tag = ""
            # ---- main: coarse forward
            n = "coarse/conv/conv2d_"
            c.conv2d_fwd(self.d_c0, self.img4, self.w(n + "0" + K), self.bias(n + "0"), relu=True, out=self.c0)
            c.maxpool2x2_fwd_f32(self.c0, out=self.p0, idx=self.i0)
            c.conv2d_fwd(self.d_c1, self.p0, self.w(n + "1" + K), self.bias(n + "1"), relu=True, out=self.c1)
            c.maxpool2x2_fwd_f32(self.c1, out=self.p1, idx=self.i1)
            c.conv2d_fwd(self.d_c2, self.p1, self.w(n + "2" + K), self.bias(n + "2"), relu=True, out=self.c2)
            c.conv2d_fwd(self.d_c3, self.c2, self.w(n + "3" + K), self.bias(n + "3"), relu=True, out=self.c3)
            c.conv2d_fwd(self.d_c4, self.c3, self.w(n + "4" + K), self.bias(n + "4"), relu=True, out=self.c4)
            c.stamp("coarse conv fwd done")
            s0.wait_event(e_aux)
            if e_pub is not None:
                s0.wait_event(e_pub)
            nd = "coarse/dense/dense_"
            c.dense_fwd(self.c4.view(B, 12288), self.w(nd + "0" + K), self.bias(nd + "0"), flags=L.EPI_RELU,
                        keep_mask=self.keep_mask, drop_rate=0.5, out=self.d0, impl=self.impl)
            c.dense_fwd(self.d0, self.w(nd + "1" + K), self.bias(nd + "1"), flags=0, out=self.coarse, impl=self.impl)
            c.stamp("dense fwd done")
            e_coarse = mark(s0)
            # ---- fine stream, part 2
            with torch.cuda.stream(s1):
                c.ws_tag = "fine"
                s1.wait_event(e_coarse)
                c.scatter_channel_bf16(self.coarse, self.cat, 63)
                c.conv2d_fwd(self.d_f2, self.cat, self.w("fine/second/conv2d" + K), self.bias("fine/second/conv2d"),
                             relu=True, out=self.f2)
                c.conv2d_fwd(self.d_f3, self.f2, self.w("fine/third" + K), self.bias("fine/third"), relu=False,
                             out=self.fine.view(B, 55, 74, 1))
                c.silog_loss(self.fine, self.tar, LAMBDA_OVER_N, want_grad=False, loss_ps=self.lps_fine, loss=self.loss_fine,
                             dout_bf16=self.g_fine)
                c.stamp("fine fwd + loss done")
                c.ws_tag = ""
                e_fine = mark(s1)
            # ---- main: coarse loss, then the dgrad chain; wgrad stream follows each dY
            c.silog_loss(self.coarse, self.tar, LAMBDA_OVER_N, want_grad=False, loss_ps=self.lps_coarse,
                         loss=self.loss_coarse, dout_bf16=self.g_coarse, dout_ld=4096)
            e_g = mark(s0)

            def on_wgrad(event, fn, stream=None, label=None):
                stream = stream or s2
                with torch.cuda.stream(stream):
                    c.ws_tag = "wgrad" if stream is s2 else "cwgrad"
                    stream.wait_event(event)
                    if label:
                        c.stamp(label + " begin")
                    fn()
                    if label:
                        c.stamp(label + " end")
                    c.ws_tag = ""

            fused = self.fuse_dense_adam and not self.comm
            a = self.arena
            # The bias gradients (latency-bound column sums of dY, 7-10 us each) leave the conv-wgrad stream
            # for the fine stream, whose forward work is long done by then: they run next to the wgrad GEMMs, not before them.
            # (Data parallel: measured slower at 2 GPUs, 1.184 vs 1.144 ms -- the comm stream's NCCL kernels already fill
            # those gaps -- so there the conv wgrads keep their bias gradients.)
            side_bias = not self.comm

            def conv_wgrad(desc, x, dy, name, event):
                if side_bias:
                    with torch.cuda.stream(s1):
                        s1.wait_event(event)
                        c.bias_grad_bf16(dy.view(-1, dy.shape[-1]), dy.shape[-1], self.gw(name + "/bias"))
                    on_wgrad(event, lambda: c.conv2d_wgrad(desc, x, dy, dw=self.gw(name + K), db=None), s3)
                else:
                    on_wgrad(event, lambda: c.conv2d_wgrad(desc, x, dy, dw=self.gw(name + K), db=self.gw(name + "/bias")), s3)

            dense_wgrad_adam = self._dense_wgrad_adam
            nd = "coarse/dense/dense_"

            e_loss = e_g
            c.dense_dgrad_act(self.g_coarse, self.w(nd + "1" + K), self.d0, self.keep_mask, 0.5, L.EPI_RELU, out=self.g_d0,
                              impl=self.impl)
            e_g = mark(s0)
            # data parallel, dense layers: exchange activations instead of gradients (dp.dense_gather_adam_merged)
            gather = bool(self.comm) and all(self.comm.can_gather_dense(self, nd + l + K, B) for l in "01")
            e_g1 = e_g
            if not fused and not gather:
                # the bucket's Adam overwrites dense_1's weights: it waits for e_g (dense_1's dgrad has read them)
                on_wgrad(e_loss, lambda: (c.dense_wgrad(self.d0, self.g_coarse, dw=self.gw(nd + "1" + K),
                                                        db=self.gw(nd + "1/bias"), impl=self.impl),
                                          self.comm and dp_update("dense_1", "CoarseDense", e_g)))
            if fused:       # updates dense_1's weights: must follow dense_1's dgrad, their last reader
                on_wgrad(e_g, lambda: dense_wgrad_adam("1", self.d0, self.g_coarse), label="dense_1 wgrad+adam")
            e_d0 = e_g
            c.dense_dgrad_act(self.g_d0, self.w(nd + "0" + K), self.c4.view(B, 12288), None, 0.0, L.EPI_RELU,
                              out=self.g_c4.view(B, 12288), impl=self.impl)
            e_g = mark(s0)
            if gather:
                # one activation all-gather for both layers as soon as g_d0 exists (e_d0); each layer's row update waits for
                # its own dgrad; the updated rows are published at the start of the next step
                g_ = "CoarseDense"
                self.comm.dense_gather_adam_merged(
                    self, [(nd + "1" + K, nd + "1/bias", self.d0, self.g_coarse, e_g1),
                           (nd + "0" + K, nd + "0/bias", self.c4.view(B, 12288), self.g_d0, e_g)],
                    g_, ADAM_LR[g_], ADAM_BETA1, ADAM_EPS, ready=e_d0)
            elif not fused:
                on_wgrad(e_d0, lambda: (c.dense_wgrad(self.c4.view(B, 12288), self.g_d0, dw=self.gw(nd + "0" + K),
                                                      db=self.gw(nd + "0/bias"), impl=self.impl),
                                        self.comm and dp_update("dense_0", "CoarseDense", e_g)))
            c.stamp("dense dgrad done")
            if fused:
                on_wgrad(e_g, lambda: dense_wgrad_adam("0", self.c4.view(B, 12288), self.g_d0), label="dense_0 wgrad+adam")
            elif not self.comm:
                # single GPU: the dense group's Adam runs under the conv backward.  It overwrites the dense weight
                # mirror, so it waits for e_g: both dense dgrads (the last readers of those weights) are done.
                on_wgrad(e_g, lambda: self.apply_adam(("CoarseDense",)))
            conv_wgrad(self.d_c4, self.c3, self.g_c4, n + "4", e_g)
            c.conv2d_dgrad(self.d_c4, self.g_c4, self.w(n + "4" + K), out=self.g_c3, relu_src=self.c3)
            c.stamp("dgrad conv2d_4 done")
            e_g = mark(s0)
            conv_wgrad(self.d_c3, self.c2, self.g_c3, n + "3", e_g)
            s0.wait_event(e_flip)
            c.conv2d_dgrad(self.d_c3, self.g_c3, self.w(n + "3" + K), out=self.g_c2, relu_src=self.c2, wflip=self._wflip["3"])
            e_g = mark(s0)
            conv_wgrad(self.d_c2, self.p1, self.g_c2, n + "2", e_g)
            c.conv2d_dgrad(self.d_c2, self.g_c2, self.w(n + "2" + K), out=self.g_p1, wflip=self._wflip["2"])
            c.maxpool2x2_idx_bwd(self.i1, self.g_p1, (B, 27, 37, 256), out=self.g_c1)
            c.stamp("dgrad conv2d_3,2 + pool bwd done")
            e_g = mark(s0)
            # (DP: exchanging conv2d_4..2 here as an early bucket was measured SLOWER at 2 GPUs, 1.30 vs 1.26 ms: three more
            # NCCL launches cost more than the shorter tail saves)
            conv_wgrad(self.d_c1, self.p0, self.g_c1, n + "1", e_g)
            e_w1 = mark(s3)                                # gradients of conv2d_4 .. conv2d_1 are complete
            c.conv2d_dgrad(self.d_c1, self.g_c1, self.w(n + "1" + K), out=self.g_p0, wflip=self._wflip["1"])
            c.maxpool2x2_idx_bwd(self.i0, self.g_p0, (B, 55, 74, 96), out=self.g_c0)
            c.stamp("dgrad conv2d_1 + pool bwd done")
            e_g = mark(s0)
            # Single GPU: TF-Adam of conv2d_4 .. conv2d_1 (99 % of the group) runs on the idle fine stream next to
            # conv2d_0's weight gradient; only conv2d_0's 55 k parameters are updated in the step's tail.  The group is
            # one contiguous arena range in backward order, so this is the same update as two launches.
            # Data parallel, the same cut: conv2d_4 .. conv2d_1 are all-reduced in f32 and updated behind conv2d_1's weight
            # gradient, under conv2d_1's dgrad, the pool backward and conv2d_0's wgrad; the step's tail exchanges conv2d_0's
            # 55 k parameters only.  (8 GPUs, profiles/step_timeline_r02_n8_rank0.json: the single 16 MB allreduce + Adam was
            # ~150 us of exposed tail.)  f32 allreduce + replicated Adam beats cast + reduce-scatter + sharded Adam +
            # all-gather at every world size (4 GPUs: 1.160 vs 1.185 ms; 2 GPUs, with the split: 0.972 vs 1.015 ms -- the
            # collectives are latency-bound at 8-16 MB and the sharded form needs three of them); a sharded exchange of the
            # split measured 1.20 against 1.18 ms unsplit at 2 GPUs (the extra NCCL kernels take SM slots from the GEMMs
            # they overlap with).
            lo_cc, hi_cc = a.group_range("CoarseConv")
            split_cc = a.specs["coarse/conv/conv2d_0/kernel"].offset
            if self.comm:
                with torch.cuda.stream(s3):
                    self.comm.bucket_ready(self, "coarse_conv_main", after=e_g,
                                           then=lambda lo, hi: self.adam_range("CoarseConv", lo, hi, inv_world))
            else:
                with torch.cuda.stream(s1):
                    s1.wait_event(e_fine)
                    s1.wait_event(e_w1)
                    s1.wait_event(e_g)                      # conv2d_1's dgrad was the last reader of these weights
                    self.adam_range("CoarseConv", lo_cc, split_cc)
                    e_fine = mark(s1)

            e_b0 = None
            if side_bias:
                with torch.cuda.stream(s1):
                    s1.wait_event(e_g)
                    c.bias_grad_bf16(self.g_c0.view(-1, 96), 96, self.gw(n + "0/bias"))
                    e_b0 = mark(s1)

            def conv0_and_adam():
                c.conv2d_wgrad(self.d_c0, self.img4, self.g_c0, dw=self.gw(n + "0" + K), db=None if side_bias else self.gw(n + "0/bias"))
                if e_b0 is not None:
                    s3.wait_event(e_b0)
                self._mask_padding("coarse/conv/conv2d_0/kernel")
                if self.comm:
                    self.comm.bucket_ready(self, "coarse_conv_0",
                                           then=lambda lo, hi: self.adam_range("CoarseConv", lo, hi, inv_world))
                    self.comm.wait_all(self)
                else:
                    self.adam_range("CoarseConv", split_cc, hi_cc)
            on_wgrad(e_g, conv0_and_adam, s3, label="conv2d_0 wgrad + conv exchange/adam")
            # ---- join
            s0.wait_event(e_fine)
            s0.wait_event(mark(s2))
            s0.wait_event(mark(s3))
            c.increment_i64(self.step_dev)
            c.stamp("step end")
            e_out = torch.cuda.Event()
            e_out.record(s0)
        cur.wait_event(e_out)

    # ------------------------------------------------------------------ one session.run(model_op)
    def _enqueue_step(self, phase):
        if phase == 1 and self.overlap and self.train:
            return self._enqueue_phase1_overlapped()
        if self.comm:
            self.comm.flush(self)                       # rows updated by a previous (overlapped) step
        self.forward()
        if phase == 1:
            fused = self.fuse_dense_adam and not self.comm
            self.backward_coarse(fused_dense_adam=fused)
            groups = ("CoarseConv",) if fused else ("CoarseDense", "CoarseConv")
        elif phase == 2:
            self.backward_fine()
            groups = ("FineA", "FineB")
        else:
            groups = ()
        if groups:
            scale = 1.0
            if self.comm:
                self.comm.wait_all(self)
                scale = 1.0 / self.comm.world
            self.apply_adam(groups, scale)
            if "FineA" in groups:
                self.refresh_derived()                   # fine/first moved: re-embed it into the pool-fused filter
        self.ctx.increment_i64(self.step_dev)            # global_step += 1 (src/models.py:329,343,356)

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
