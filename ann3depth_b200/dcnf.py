"""DCNF (Liu et al. 2015) train / inference step on liba3d -- host-side orchestration.

Mirrors `_DistributedConvolutionalNeuralFields` of the reference (src/models.py:9-200): resize to
240x320, 100x100 patches around the 6x8 grid of 40x40 tiles, unary CNN on every patch, pairwise
colour / histogram similarities through a 2->1 dense layer, CRF negative log-likelihood with
A = I + D - R, plain SGD (lr 0.1).  The hard-coded worker devices of the reference (:63-79) and its
serial `map_fn`s are gone: the unary CNN runs once per zero-padded image (fully convolutional -- its patches
are windows of that pass; `unary="patches"` keeps the literal B*48-patch batch), and every CRF graph gets
its own CTA.

As in TF 1.3, no gradient reaches `pairwise_layers` (ScatterNdUpdate is not differentiable,
src/models.py:138-141): only the unary CNN trains.
"""
from __future__ import annotations

import math

import torch

from . import _lib as L
from . import ops
from .params import DCNF_FIRST_EMBEDDED_SHAPE, Arena, dcnf_first_index_maps, dcnf_specs

H, W = 240, 320            # src/models.py:180-181
SP = 40                    # src/models.py:16
SGD_LR = 0.1               # src/models.py:198
GAMMA = 1.0                # src/models.py:17
PATCH_PAD = 30             # zero border of the SAME patch extraction (100x100 windows, stride 40; src/models.py:50-59)


def num_superpixels(h=H, w=W):
    """src/models.py:32-35."""
    return math.ceil(h / SP), math.ceil(w / SP)


def grid4_pairs(h=H, w=W):
    """Beyond the reference (SURVEY.md 8f N4): every horizontal and vertical neighbour pair of the tile grid, once each
    (82 pairs on the 6 x 8 grid: #pairs != #nodes, which the reference's R sizing, src/models.py:149, cannot express)."""
    rows, cols = num_superpixels(h, w)
    left, right = [], []
    for r in range(rows):
        for c in range(cols):
            if c + 1 < cols:
                left.append(r * cols + c); right.append(r * cols + c + 1)
            if r + 1 < rows:
                left.append(r * cols + c); right.append((r + 1) * cols + c)
    return left, right


def pair_indices(h=H, w=W):
    """src/models.py:20-30."""
    max_rows, max_cols = num_superpixels(h, w)
    left, right = [], []
    for row in range(1, max_rows - 1):
        for col in range(2 - (row & 1), max_cols - 1, 2):
            pixel = row * max_cols + col
            for addend in [-max_cols, max_cols, -1, 1]:
                left.append(pixel)
                right.append(pixel + addend)
    return left, right


class DCNFNet:
    def __init__(self, ctx: ops.Context, batch: int, in_hw=(480, 640), depth_hw=(480, 640), train=True,
                 impl=L.IMPL_AUTO, naive_loss=True, comm=None, graph="reference", r_nonneg=False, train_pairwise=False,
                 predict="unary", unary="fullconv", augment=None, augment_seed=3):
        """Beyond-reference options (SURVEY.md 8f N4; defaults reproduce the reference):
             graph="grid4"        every neighbour pair of the tile grid (82 pairs != 48 nodes) instead of the reference's
                                  checkerboard star graph (src/models.py:20-30);
             r_nonneg=True        r = max(pairwise_dense(.), 0): A = I + D - R stays SPD whatever the layer learns;
             train_pairwise=True  the CRF's gradient w.r.t. r flows into `pairwise_layers` (TF 1.3 blocks it at
                                  ScatterNdUpdate, src/models.py:138-141) and SGD updates that layer too;
             predict="map"        the output is the CRF's MAP estimate y* = A^-1 z (Liu et al. eq. 12), bilinearly upsampled,
                                  instead of the unary prediction the reference upsamples (src/models.py:187-191);
             augment=Augment(...) training-time augmentation of image and depth (augment.py), drawn on the device from
                                  (augment_seed + rank, step_dev, image) and applied by the two resizes."""
        if augment is not None and not train:
            raise ValueError("augment is a training option: an inference net (train=False) sees its inputs unchanged")
        self.ctx, self.B, self.train, self.impl, self.naive = ctx, batch, train, impl, naive_loss
        assert graph in ("reference", "grid4") and predict in ("unary", "map") and unary in ("fullconv", "patches")
        self.r_nonneg, self.train_pairwise, self.predict = r_nonneg, train_pairwise, predict
        self.dev = torch.device(f"cuda:{ctx.device}")
        self.comm = comm
        self.arena = Arena(dcnf_specs(), self.dev, with_adam=False)
        self.global_step = 0
        self._graph = None
        rows, cols = num_superpixels()
        self.n = rows * cols
        pl, pr = pair_indices() if graph == "reference" else grid4_pairs()
        if graph == "reference":
            assert len(pl) == self.n, "the reference sizes R by #pairs, valid only when #pairs == #nodes (src/models.py:149)"
        self.n_pairs = len(pl)
        self.pl = torch.tensor(pl, dtype=torch.int32, device=self.dev)
        self.pr = torch.tensor(pr, dtype=torch.int32, device=self.dev)
        B, NP = batch, batch * self.n
        self.NP = NP
        bf, f32 = dict(dtype=torch.bfloat16, device=self.dev), dict(dtype=torch.float32, device=self.dev)
        u8 = dict(dtype=torch.uint8, device=self.dev)
        z = torch.zeros
        self.images = z(B, in_hw[0], in_hw[1], 3, **f32)
        self.depths = z(B, depth_hw[0], depth_hw[1], 1, **f32)
        self.augment = augment
        self.aug_params = self.aug_desc = None
        self.external_aug = False
        if augment is not None:
            # device global step: the draw's counter, so replays of the captured step draw fresh parameters.  Only an
            # augmenting net has one; the unaugmented step stays exactly as it was.
            self.step_dev = torch.zeros(1, dtype=torch.int64, device=self.dev)
            self.aug_desc = augment.desc()
            self.augment_seed = augment_seed + (comm.rank if comm is not None else 0)
            self.aug_params = z(B, L.AUG_PARAMS, **f32)
        self.im = z(B, H, W, 3, **f32)
        self.dp = z(B, H, W, 1, **f32)
        # Unary CNN (src/models.py:61-83).  unary = "fullconv" (default): the patches are plain windows (stride 40, zero
        # border 30) and every layer is a VALID convolution or an even-aligned 2x2 pool, so each layer of patch
        # (prow, pcol) IS a window of the same layer of the zero-padded whole image -- the network runs ONCE per image
        # (N0 = B images of 150 x 190 cells, a third of the FLOPs of 48 overlapping patches, no patch tensor at all) and
        # only the 7x7x256 inputs of the first dense layer are gathered per patch (windows of stride 5,
        # a3d_window_gather / a3d_window_scatter_sum).  unary = "patches": the reference's literal formulation (N0 = B*48
        # patches of 50 x 50 cells) on the same kernels; kept as the cross-check of the fully convolutional form.
        # First layer (:64-66: 11x11x3 -> 64, ReLU, 2x2 max-pool) in both forms: ONE pool-fused convolution over
        # space-to-depth(2) cells of 16 channels, read 4 cells (128 bytes) per tap through an overlapped-pixel view
        # (params.dcnf_first_embedded; a3d_conv_desc dil_w = 4, pix_pitch = 16).
        self.unary = unary
        if unary == "fullconv":
            N0, ch, cw = B, (H + 2 * PATCH_PAD) // 2, (W + 2 * PATCH_PAD) // 2
        else:
            N0, ch, cw = NP, 50, 50
        self.N0 = N0
        s0 = (ch - 5, cw - 5)                          # pooled first layer (one output per cell)
        s1 = (s0[0] - 4, s0[1] - 4)                    # conv2d_1 5x5
        q1 = (s1[0] // 2, s1[1] // 2)
        s2 = (q1[0] - 2, q1[1] - 2)
        s3 = (s2[0] - 2, s2[1] - 2)
        s4 = (s3[0] - 2, s3[1] - 2)
        q4 = (s4[0] // 2, s4[1] // 2)
        self.s1, self.s4, self.q4 = s1, s4, q4
        assert q4 == (((rows - 1) * 5 + 7, (cols - 1) * 5 + 7) if unary == "fullconv" else (7, 7))
        ncell = N0 * ch * cw * 16
        self._cells = z(ncell + 128, **bf)             # + slack: the last positions of the last row read past the end
        self.cells = self._cells[:ncell].view(N0, ch, cw, 16)
        cd = ops.conv_desc
        d0 = cd(N0, ch, cw, 64, 256, 6, 2, 1, "valid", ldy=64, impl=impl)
        d0.P, d0.Q = s0
        d0.dil_w = 4
        d0.pix_pitch = 16
        self.d0 = d0
        self.d0w = L.ConvDesc.from_buffer_copy(d0)     # the weight gradient sees the 4 x 64 GEMM columns
        self.d0w.ldy = 256
        self.wbig0 = z(*DCNF_FIRST_EMBEDDED_SHAPE, **bf)
        km, bm = dcnf_first_index_maps(self.arena.specs["unary/unary_layers/conv2d/kernel"],
                                       self.arena.specs["unary/unary_layers/conv2d/bias"])
        self.emb_k, self.emb_b = km.to(self.dev), bm.to(self.dev)
        self.d1 = cd(N0, s0[0], s0[1], 64, 256, 5, 5, 1, "valid", impl=impl)        # :67
        self.d2 = cd(N0, q1[0], q1[1], 256, 256, 3, 3, 1, "valid", impl=impl)       # :69
        self.d3 = cd(N0, s2[0], s2[1], 256, 256, 3, 3, 1, "valid", impl=impl)       # :71
        self.d4 = cd(N0, s3[0], s3[1], 256, 256, 3, 3, 1, "valid", impl=impl)       # :72
        self.p0, self.i0 = z(N0, *s0, 64, **bf), z(N0, *s0, 64, **u8)
        # conv outputs that feed a max-pool: f32 + routing record when training; inference pools the bf16 output (the same
        # values: rounding is monotone) at half the bytes
        pool_src = f32 if train else bf
        self.c1 = z(N0, *s1, 256, **pool_src)
        self.p1, self.i1 = z(N0, *q1, 256, **bf), z(N0, *q1, 256, **u8)
        self.c2 = z(N0, *s2, 256, **bf)
        self.c3 = z(N0, *s3, 256, **bf)
        self.c4 = z(N0, *s4, 256, **pool_src)
        self.p4, self.i4 = z(N0, *q4, 256, **bf), z(N0, *q4, 256, **u8)
        # the first dense layer's input: one 7x7x256 window per patch
        self.xd = z(NP, 12544, **bf) if unary == "fullconv" else self.p4.view(NP, 12544)
        self.h0 = z(NP, 128, **bf)
        self.h1 = z(NP, 16, **bf)
        self.z = z(NP, 1, **f32)
        self.sims = z(B, self.n_pairs, 2, **f32)
        self.r = z(B, self.n_pairs, **f32)
        self.dr = z(B, self.n_pairs, **f32) if (train and train_pairwise) else None
        self.y = z(B, self.n, **f32)
        self.ystar, self.nll, self.logdet = z(B, self.n, **f32), z(B, **f32), z(B, **f32)
        self.status = torch.zeros(B, dtype=torch.int32, device=self.dev)
        self.loss = z(1, **f32)
        self.output = z(B, H, W, 1, **f32)
        if train:
            self.dz = z(B, self.n, **f32)
            self.g_z = z(NP, 1, **bf)
            self.g_h1a, self.g_h1 = z(NP, 16, **bf), z(NP, 16, **bf)
            self.g_h0a, self.g_h0 = z(NP, 128, **bf), z(NP, 128, **bf)
            self.g_p4 = z(N0, *q4, 256, **bf)
            self.g_xd = z(NP, 12544, **bf) if unary == "fullconv" else self.g_p4.view(NP, 12544)
            self.g_c4 = z(N0, *s4, 256, **bf)
            self.g_c3 = z(N0, *s3, 256, **bf)
            self.g_c2 = z(N0, *s2, 256, **bf)
            self.g_p1 = z(N0, *q1, 256, **bf)
            self.g_c1 = z(N0, *s1, 256, **bf)
            self.g_p0 = z(N0, *s0, 64, **bf)
            self.g_big0 = z(N0 * s0[0] * s0[1], 256, **bf)   # gradient on the 4 x 64 pool-window columns
            nk = 256 * 6 * 2 * 64
            self.g_wbig0 = z(nk + 256, **f32)

    # ------------------------------------------------------------------ parameters
    def w(self, name):
        return self.arena.view(self.arena.wb, name)

    def wf(self, name):
        return self.arena.view(self.arena.w, name)

    def gw(self, name):
        return self.arena.view(self.arena.g, name)

    def load_params(self, tf_params):
        self.arena.load_tf(tf_params)
        self.refresh_derived()

    def refresh_derived(self):
        """Re-embed the canonical first-layer filter into the pool-fused filter the kernels read (after a load or an SGD
        step); entries outside the four embedded copies stay zero."""
        s = self.arena.specs["unary/unary_layers/conv2d/kernel"]
        self.ctx.scatter_cast_bf16(self.arena.w[s.offset:s.offset + s.numel], self.emb_k, self.wbig0)

    def export_params(self):
        return self.arena.export_tf()

    def export_grads(self):
        return self.arena.export_tf(self.arena.g)

    def set_augment_params(self, params):
        """Parity hook: use explicit augmentation parameters [B,16] (include/a3d.h A3D_AUG_*) instead of the device
        draw."""
        if self.augment is None:
            raise ValueError("set_augment_params needs a net built with augment=Augment(...)")
        self.aug_params.copy_(params.to(torch.float32))
        self.external_aug = True

    # ------------------------------------------------------------------ forward
    def forward(self):
        c, B, NP = self.ctx, self.B, self.NP
        U, K = "unary/unary_layers/", "/kernel"
        if self.augment is not None:
            if not self.external_aug:
                c.augment_draw(self.aug_desc, self.aug_params, self.augment_seed, self.step_dev)
            c.resize_affine_tf1(self.images, H, W, self.aug_params, depth=False, out=self.im)
            c.resize_affine_tf1(self.depths, H, W, self.aug_params, depth=True, out=self.dp)
        else:
            c.resize_bilinear_tf1(self.images, H, W, out=self.im)
            c.resize_bilinear_tf1(self.depths, H, W, out=self.dp)
        # unary part (src/models.py:61-89) on all B*48 patches at once
        if self.unary == "fullconv":
            c.image_cells_s2d(self.im, PATCH_PAD, self.cells)
        else:
            c.extract_patches_s2d(self.im, self.cells)
        c.conv2d_pool4_fwd(self.d0, self.cells, self.wbig0, self.wf(U + "conv2d/bias"), relu=True, out=self.p0, idx=self.i0)
        c.conv2d_fwd(self.d1, self.p0, self.w(U + "conv2d_1" + K), self.wf(U + "conv2d_1/bias"), relu=True, out=self.c1)
        if self.train:
            c.maxpool2x2_fwd_f32(self.c1, out=self.p1, idx=self.i1)
        else:
            c.maxpool2x2_fwd(self.c1, out=self.p1)
        c.conv2d_fwd(self.d2, self.p1, self.w(U + "conv2d_2" + K), self.wf(U + "conv2d_2/bias"), relu=True, out=self.c2)
        c.conv2d_fwd(self.d3, self.c2, self.w(U + "conv2d_3" + K), self.wf(U + "conv2d_3/bias"), relu=True, out=self.c3)
        c.conv2d_fwd(self.d4, self.c3, self.w(U + "conv2d_4" + K), self.wf(U + "conv2d_4/bias"), relu=True, out=self.c4)
        if self.train:
            c.maxpool2x2_fwd_f32(self.c4, out=self.p4, idx=self.i4)
        else:
            c.maxpool2x2_fwd(self.c4, out=self.p4)
        if self.unary == "fullconv":                  # patch (prow, pcol) reads the 7x7 window at (5 prow, 5 pcol)
            rows, cols = num_superpixels()
            c.window_gather(self.p4, rows, cols, 7, 5, self.xd)
        c.dense_fwd(self.xd, self.w(U + "dense" + K), self.wf(U + "dense/bias"), flags=L.EPI_RELU,
                    out=self.h0, impl=self.impl)
        c.dense_fwd(self.h0, self.w(U + "dense_1" + K), self.wf(U + "dense_1/bias"), flags=L.EPI_SIGMOID, out=self.h1,
                    impl=L.IMPL_SIMT)
        c.dense_fwd(self.h1, self.w(U + "dense_2" + K), self.wf(U + "dense_2/bias"), flags=0, out=self.z,
                    impl=L.IMPL_SIMT)
        # pairwise part (src/models.py:108-127)
        c.pairwise_features(self.im, self.pl, self.pr, GAMMA, out=self.sims)
        P = "pairwise/pairwise_layers/dense"
        if self.r_nonneg:
            c.pairwise_dense_act(self.sims, self.wf(P + K), self.wf(P + "/bias"), flags=L.EPI_RELU, out=self.r)
        else:
            c.pairwise_dense(self.sims, self.wf(P + K), self.wf(P + "/bias"), out=self.r)
        # loss part (src/models.py:129-177)
        c.tile_means(self.dp, out=self.y)
        c.crf(self.z.view(B, self.n), self.y, self.r, self.pl, self.pr, grad_scale=1.0 / B, naive=self.naive,
              out=dict(ystar=self.ystar, nll=self.nll, logdet=self.logdet, dz=self.dz if self.train else None,
                       dr=self.dr, status=self.status))
        c.mean_f32(self.nll, self.loss)
        # output (src/models.py:187-191): the unary prediction, upsampled
        rows, cols = num_superpixels()
        src = self.ystar if self.predict == "map" else self.z
        c.resize_bilinear_tf1(src.view(B, rows, cols, 1), H, W, out=self.output)

    # ------------------------------------------------------------------ backward (unary CNN only)
    def backward(self):
        c, NP = self.ctx, self.NP
        U, K = "unary/unary_layers/", "/kernel"
        hook = self.comm.bucket_ready if self.comm else (lambda *_: None)
        if self.train_pairwise:
            P = "pairwise/pairwise_layers/dense"
            c.pairwise_dense_bwd(self.sims, self.r, self.dr, self.gw(P + K), self.gw(P + "/bias"),
                                 flags=L.EPI_RELU if self.r_nonneg else 0)
        c.scale_cast_bf16(self.dz.view(-1), self.g_z.view(-1), 1.0)
        S = L.IMPL_SIMT
        c.dense_wgrad(self.h1, self.g_z, dw=self.gw(U + "dense_2" + K), db=self.gw(U + "dense_2/bias"), N=1, impl=S)
        c.dense_dgrad(self.g_z, self.w(U + "dense_2" + K), out=self.g_h1a, impl=S)
        c.dense_epilogue_bwd(self.g_h1a, self.h1, None, 0.0, L.EPI_SIGMOID, out=self.g_h1)
        c.dense_wgrad(self.h0, self.g_h1, dw=self.gw(U + "dense_1" + K), db=self.gw(U + "dense_1/bias"), impl=S)
        c.dense_dgrad(self.g_h1, self.w(U + "dense_1" + K), out=self.g_h0a, impl=S)
        c.dense_epilogue_bwd(self.g_h0a, self.h0, None, 0.0, L.EPI_RELU, out=self.g_h0)
        c.dense_wgrad(self.xd, self.g_h0, dw=self.gw(U + "dense" + K), db=self.gw(U + "dense/bias"), impl=self.impl)
        c.dense_dgrad(self.g_h0, self.w(U + "dense" + K), out=self.g_xd, impl=self.impl)
        if self.unary == "fullconv":                  # shared activations: sum over the (up to 4) windows covering them
            rows, cols = num_superpixels()
            c.window_scatter_sum(self.g_xd, rows, cols, 7, 5, self.g_p4)
        N0 = self.N0
        c.maxpool2x2_idx_bwd(self.i4, self.g_p4, (N0, *self.s4, 256), out=self.g_c4)
        c.conv2d_wgrad(self.d4, self.c3, self.g_c4, dw=self.gw(U + "conv2d_4" + K), db=self.gw(U + "conv2d_4/bias"))
        c.conv2d_dgrad(self.d4, self.g_c4, self.w(U + "conv2d_4" + K), out=self.g_c3, relu_src=self.c3)
        c.conv2d_wgrad(self.d3, self.c2, self.g_c3, dw=self.gw(U + "conv2d_3" + K), db=self.gw(U + "conv2d_3/bias"))
        c.conv2d_dgrad(self.d3, self.g_c3, self.w(U + "conv2d_3" + K), out=self.g_c2, relu_src=self.c2)
        c.conv2d_wgrad(self.d2, self.p1, self.g_c2, dw=self.gw(U + "conv2d_2" + K), db=self.gw(U + "conv2d_2/bias"))
        c.conv2d_dgrad(self.d2, self.g_c2, self.w(U + "conv2d_2" + K), out=self.g_p1)
        c.maxpool2x2_idx_bwd(self.i1, self.g_p1, (N0, *self.s1, 256), out=self.g_c1)
        c.conv2d_wgrad(self.d1, self.p0, self.g_c1, dw=self.gw(U + "conv2d_1" + K), db=self.gw(U + "conv2d_1/bias"))
        c.conv2d_dgrad(self.d1, self.g_c1, self.w(U + "conv2d_1" + K), out=self.g_p0)
        # first layer: MaxPoolGrad + ReluGrad onto the 4 x 64 GEMM columns, weight gradient of the embedded filter, then
        # fold its four copies (and the four bias groups) into the canonical variable (padding channels receive 0)
        c.pool4_bwd(self.g_p0.view(-1, 64), self.p0.view(-1, 64), self.i0, out=self.g_big0)
        nk = 256 * 6 * 2 * 64
        c.conv2d_wgrad(self.d0w, self.cells, self.g_big0.view(N0, self.d0.P, self.d0.Q, 256), dw=self.g_wbig0[:nk].view(256, 6, 2, 64),
                       db=self.g_wbig0[nk:])
        c.gather_sum_f32(self.g_wbig0[:nk], self.emb_k, self.gw(U + "conv2d" + K))
        c.gather_sum_f32(self.g_wbig0[nk:], self.emb_b, self.gw(U + "conv2d/bias"))
        hook(self, "SGD")

    def _enqueue_step(self):
        self.forward()
        self.backward()
        scale = 1.0
        if self.comm:
            self.comm.wait_all(self)
            scale = 1.0 / self.comm.world
        lo, hi = self.arena.group_range("SGD")
        self.ctx.sgd(self.arena.w[lo:hi], self.arena.g[lo:hi], self.arena.wb[lo:hi], SGD_LR, scale)
        if self.train_pairwise:
            assert not self.comm, "train_pairwise is a single-GPU option"
            lo, hi = self.arena.group_range("Pairwise")
            self.ctx.sgd(self.arena.w[lo:hi], self.arena.g[lo:hi], self.arena.wb[lo:hi], SGD_LR, 1.0)
        self.refresh_derived()
        if self.augment is not None:
            self.ctx.increment_i64(self.step_dev)

    def train_step(self, use_graph=False):
        """One `session.run(model_op)` (src/models.py:198-200).  use_graph (single GPU): the ~45 launches of the step are
        captured once -- after an untimed eager pass that lets the GEMM tuner settle, whose effect is undone -- and
        replayed; the step reads the caller's image / depth buffers in place."""
        if use_graph and not self.comm:
            if self._graph is None:
                saved = (self.arena.w.clone(), self.arena.wb.clone())
                step0 = self.step_dev.clone() if self.augment is not None else None
                self._enqueue_step()
                torch.cuda.synchronize()
                self.arena.w.copy_(saved[0]); self.arena.wb.copy_(saved[1])
                if step0 is not None:
                    self.step_dev.copy_(step0)
                self.refresh_derived()
                gr = torch.cuda.CUDAGraph()
                with torch.cuda.graph(gr):
                    self._enqueue_step()
                self._graph = gr
            self._graph.replay()
        else:
            self._enqueue_step()
        self.global_step += 1
        return 1

    def infer(self):
        self.forward()
        return self.output


class DCNFTrainOp:
    """The object `models.dcnf(images, depths)` returns (src/models.py:198-200: minimize(loss, global_step))."""

    def __init__(self, net: DCNFNet):
        self.net = net
        self.losses = {"loss/mean_loss": net.loss}
        self.outputs = net.output

    @property
    def global_step(self):
        return self.net.global_step

    @property
    def trainable_variables(self):
        return {n: s.tf_shape for n, s in self.net.arena.specs.items()}

    def run(self, use_graph=False):
        if self.net.train:
            return self.net.train_step(use_graph=use_graph)
        return self.net.infer()

    __call__ = run
