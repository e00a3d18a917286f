"""Torch-tensor front end of the liba3d C-ABI: one thin method per entry point of include/a3d.h.

Tensors are only carriers of device memory (`data_ptr()`); all arithmetic happens in liba3d.so.
Every method launches on torch's current CUDA stream, so callers can wrap a whole step in a
`torch.cuda.graph` capture.
"""
from __future__ import annotations

import ctypes as C
import math

import torch

from . import _lib as L
from ._lib import ConvDesc


def _ptr(t):
    return None if t is None else C.c_void_p(t.data_ptr())


def _stream():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def adam_lr_t(lr, beta1, beta2, t):
    """lr_t = lr * sqrt(1 - beta2^t) / (1 - beta1^t)  (TF1 AdamOptimizer; t >= 1)."""
    return lr * math.sqrt(1.0 - beta2 ** t) / (1.0 - beta1 ** t)


def conv_desc(N, H, W, Cin, K, R, S, stride=1, padding="valid", ldy=None, impl=L.IMPL_AUTO):
    """Build an `a3d_conv_desc` with TF padding rules (src/models.py conv2d call sites)."""
    if isinstance(stride, int):
        stride = (stride, stride)
    sh, sw = stride
    if isinstance(padding, str):
        if padding.lower() == "same":
            P, Q = -(-H // sh), -(-W // sw)
            pt = max((P - 1) * sh + R - H, 0) // 2
            pl = max((Q - 1) * sw + S - W, 0) // 2
        else:
            P, Q = (H - R) // sh + 1, (W - S) // sw + 1
            pt = pl = 0
    else:
        pt, pl = padding
        P, Q = (H + 2 * pt - R) // sh + 1, (W + 2 * pl - S) // sw + 1
    d = ConvDesc()
    d.N, d.H, d.W, d.C, d.K, d.R, d.S = N, H, W, Cin, K, R, S
    d.stride_h, d.stride_w, d.pad_t, d.pad_l, d.P, d.Q = sh, sw, pt, pl, P, Q
    d.ldy = ldy if ldy is not None else K
    d.impl = impl
    return d


class Context:
    """Owns one `a3d_ctx` (one per device / rank)."""

    def __init__(self, device: int = 0):
        if not torch.cuda.is_available():
            raise L.A3DError("ann3depth_b200 needs a CUDA device (sm_100a); there is no CPU fallback")
        self.lib = L.load()
        self.device = device
        torch.cuda.set_device(device)
        h = C.c_void_p()
        L.check(self.lib.a3d_create(device, C.byref(h)), "a3d_create")
        self.h = h
        self._ws = {}
        self.ws_tag = ""          # set per stream by multi-stream callers: concurrent launches must not share scratch
        self.timeline = None      # StepTimeline when A3D_TIMELINE=1 (stamp() is a no-op otherwise)
        self.tf32x3 = False       # float32 conv2d_fwd / dense_fwd through the 3xTF32 entry points (set around a forward)

    def close(self):
        if getattr(self, "h", None):
            self.lib.a3d_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    @property
    def sm_count(self):
        return self.lib.a3d_sm_count(self.h)

    @property
    def launches(self):
        return int(self.lib.a3d_launch_count(self.h))

    def stamp(self, label):
        """In-graph timeline mark on the current stream (see StepTimeline); no-op unless a timeline is attached."""
        if self.timeline is not None:
            self.timeline.mark(self, label)

    def workspace(self, key, nbytes):
        """Persistent scratch buffers (allocated once, so steps stay CUDA-graph capturable)."""
        nbytes = max(int(nbytes), 256)
        key = (key, self.ws_tag)
        t = self._ws.get(key)
        if t is None or t.numel() < nbytes:
            t = torch.empty(nbytes, dtype=torch.uint8, device=f"cuda:{self.device}")
            self._ws[key] = t
        return t

    # ------------------------------------------------------------------ elementwise
    def resize_bilinear_tf1(self, src, OH, OW, dstC=None, dtype=torch.float32, out=None):
        B, H, W, Cc = src.shape
        if out is None:
            out = torch.empty(B, OH, OW, dstC or Cc, dtype=dtype, device=src.device)
        dstC = out.shape[-1]
        code = L.A3D_BF16 if out.dtype == torch.bfloat16 else L.A3D_F32
        L.check(self.lib.a3d_resize_bilinear_tf1(self.h, _ptr(src), B, H, W, Cc, _ptr(out), OH, OW, dstC, code,
                                                 _stream()), "resize")
        return out

    def resize_bilinear_tf1_s2d(self, src, OH, OW, s, out):
        """Resize + space-to-depth(s): out bf16 [B, OH/s, OW/s, dstC >= s*s*C]."""
        B, H, W, Cc = src.shape
        if out.dtype == torch.float32:             # TF32 mode: float32 activations
            L.check(self.lib.a3d_resize_bilinear_tf1_s2d_f32(self.h, _ptr(src), B, H, W, Cc, _ptr(out), OH, OW, s,
                                                             out.shape[-1], _stream()), "resize_s2d_f32")
            return out
        if src.dtype == torch.uint8:               # 8-bit wire format: pixel / 255 folded into the kernel
            L.check(self.lib.a3d_resize_bilinear_tf1_s2d_u8(self.h, _ptr(src), B, H, W, Cc, _ptr(out), OH, OW, s,
                                                            out.shape[-1], _stream()), "resize_s2d_u8")
            return out
        L.check(self.lib.a3d_resize_bilinear_tf1_s2d(self.h, _ptr(src), B, H, W, Cc, _ptr(out), OH, OW, s,
                                                     out.shape[-1], _stream()), "resize_s2d")
        return out

    # ------------------------------------------------------------------ augmentation (include/a3d.h a3d_augment_desc)
    def augment_draw(self, desc, params, seed, counter_dev=None):
        """params [B, 16] float32 <- one random transform per image from (seed, *counter_dev, image index)."""
        assert params.dtype == torch.float32 and params.shape[-1] == L.AUG_PARAMS and params.is_contiguous()
        L.check(self.lib.a3d_augment_draw(self.h, C.byref(desc), params.shape[0], seed & (2 ** 64 - 1),
                                          _ptr(counter_dev), _ptr(params), _stream()), "augment_draw")
        return params

    def resize_affine_tf1_s2d(self, src, OH, OW, s, params, out):
        """Augmented resize + space-to-depth(s): src f32 or uint8 [B, H, W, 3], out bf16 or f32 [B, OH/s, OW/s, dstC]."""
        B, H, W, Cc = src.shape
        sd = L.A3D_U8 if src.dtype == torch.uint8 else L.A3D_F32
        dd = L.A3D_F32 if out.dtype == torch.float32 else L.A3D_BF16
        L.check(self.lib.a3d_resize_affine_tf1_s2d(self.h, _ptr(src), sd, B, H, W, Cc, _ptr(out), dd, OH, OW, s,
                                                   out.shape[-1], _ptr(params), _stream()), "resize_affine_s2d")
        return out

    def resize_affine_tf1(self, src, OH, OW, params, depth, out=None):
        """Augmented resize, f32 NHWC; depth=True: values / s (targets), False: values * c_rgb (images)."""
        B, H, W, Cc = src.shape
        if out is None:
            out = torch.empty(B, OH, OW, Cc, dtype=torch.float32, device=src.device)
        mode = L.AUG_VALUE_DEPTH if depth else L.AUG_VALUE_COLOR
        L.check(self.lib.a3d_resize_affine_tf1(self.h, _ptr(src), B, H, W, Cc, _ptr(out), OH, OW, _ptr(params), mode,
                                               _stream()), "resize_affine")
        return out

    def conv2d_pool4_fwd(self, d, x, w, bias, relu=True, out=None, idx=None):
        """conv + bias + ReLU + 2x2 max-pool as one GEMM over the pool-embedded filter (K = 4 x 64)."""
        if out is None:
            out = torch.empty(d.N, d.P, d.Q, d.ldy, dtype=x.dtype, device=x.device)
        if x.dtype == torch.float32:
            # TF32 mode: the pool-embedded GEMM writes its 4 x 64 columns in float32, a second pass takes the group max
            rows = d.N * d.P * d.Q
            acc = self.workspace(("pool4_tf32",), rows * 256 * 4).view(torch.float32)[:rows * 256].view(rows, 256)
            e = ConvDesc.from_buffer_copy(d)
            e.ldy = 256
            self.conv2d_fwd(e, x, w, None, relu=False, out=acc.view(d.N, d.P, d.Q, 256))
            L.check(self.lib.a3d_pool4_reduce_f32(self.h, _ptr(acc), _ptr(bias), _ptr(out), out.shape[-1], _ptr(idx), rows,
                                                  L.EPI_RELU if relu else 0, _stream()), "pool4_reduce_f32")
            return out
        ws = None
        if d.impl == L.IMPL_SIMT:
            ws = self.workspace(("pool4_simt",), d.N * d.P * d.Q * 256 * 4)
        L.check(self.lib.a3d_conv2d_pool4_fwd(self.h, C.byref(d), _ptr(x), _ptr(w), _ptr(bias), _ptr(out), _ptr(idx),
                                              L.EPI_RELU if relu else 0, _ptr(ws), ws.numel() if ws is not None else 0,
                                              _stream()), "conv2d_pool4_fwd")
        return out

    def pool4_bwd(self, dy, y, idx, out=None):
        rows = idx.numel() // 64
        if out is None:
            out = torch.empty(rows, 256, dtype=dy.dtype, device=dy.device)
        if dy.dtype == torch.float32:
            L.check(self.lib.a3d_pool4_bwd_f32(self.h, _ptr(dy), dy.shape[-1], _ptr(y), y.shape[-1], _ptr(idx), _ptr(out),
                                               rows, _stream()), "pool4_bwd_f32")
            return out
        L.check(self.lib.a3d_pool4_bwd(self.h, _ptr(dy), dy.shape[-1], _ptr(y), y.shape[-1], _ptr(idx), _ptr(out), rows,
                                       _stream()), "pool4_bwd")
        return out

    def gather_sum_f32(self, src, idx, dst):
        G, n = idx.shape
        L.check(self.lib.a3d_gather_sum_f32(self.h, _ptr(src), _ptr(idx), G, n, _ptr(dst), _stream()), "gather_sum")
        return dst

    def scatter_cast_bf16(self, src, idx, dst):
        G, n = idx.shape
        if dst.dtype == torch.float32:
            L.check(self.lib.a3d_scatter_f32(self.h, _ptr(src), _ptr(idx), G, n, _ptr(dst), _stream()), "scatter_f32")
            return dst
        L.check(self.lib.a3d_scatter_cast_bf16(self.h, _ptr(src), _ptr(idx), G, n, _ptr(dst), _stream()), "scatter_cast")
        return dst

    def maxpool2x2_fwd(self, x, out=None, ldy=None):
        N, H, W, Cc = x.shape
        ldy = ldy or Cc
        if out is None:
            out = torch.empty(N, H // 2, W // 2, ldy, dtype=torch.bfloat16, device=x.device)
        L.check(self.lib.a3d_maxpool2x2_fwd(self.h, _ptr(x), N, H, W, Cc, _ptr(out), ldy, _stream()), "maxpool")
        return out

    def maxpool2x2_relu_bwd(self, x, dy, lddy=None, out=None):
        N, H, W, Cc = x.shape
        lddy = lddy or dy.shape[-1]
        if out is None:
            out = torch.empty_like(x)
        L.check(self.lib.a3d_maxpool2x2_relu_bwd(self.h, _ptr(x), _ptr(dy), lddy, N, H, W, Cc, _ptr(out), _stream()),
                "maxpool_bwd")
        return out

    def maxpool2x2_fwd_f32(self, x, out=None, ldy=None, idx=None):
        N, H, W, Cc = x.shape
        ldy = ldy or (out.shape[-1] if out is not None else Cc)
        if out is None:
            out = torch.empty(N, H // 2, W // 2, ldy, dtype=torch.bfloat16, device=x.device)
        if out.dtype == torch.float32:
            L.check(self.lib.a3d_maxpool2x2_f32(self.h, _ptr(x), N, H, W, Cc, _ptr(out), ldy, _ptr(idx), _stream()),
                    "maxpool_f32_f32")
            return out
        L.check(self.lib.a3d_maxpool2x2_fwd_f32(self.h, _ptr(x), N, H, W, Cc, _ptr(out), ldy, _ptr(idx), _stream()),
                "maxpool_f32")
        return out

    def maxpool2x2_idx_bwd(self, idx, dy, shape, lddy=None, out=None):
        N, H, W, Cc = shape
        lddy = lddy or dy.shape[-1]
        if out is None:
            out = torch.empty(N, H, W, Cc, dtype=dy.dtype, device=dy.device)
        if dy.dtype == torch.float32:
            L.check(self.lib.a3d_maxpool2x2_idx_bwd_f32(self.h, _ptr(idx), _ptr(dy), lddy, N, H, W, Cc, _ptr(out), _stream()),
                    "maxpool_idx_bwd_f32")
            return out
        L.check(self.lib.a3d_maxpool2x2_idx_bwd(self.h, _ptr(idx), _ptr(dy), lddy, N, H, W, Cc, _ptr(out), _stream()),
                "maxpool_idx_bwd")
        return out

    def relu_bwd(self, y, dy, lddy=None, out=None):
        Cc = y.shape[-1]
        rows = y.numel() // Cc
        lddy = lddy or dy.shape[-1]
        if out is None:
            out = torch.empty_like(y)
        if y.dtype == torch.float32:
            L.check(self.lib.a3d_act_bwd_f32(self.h, _ptr(dy), lddy, _ptr(y), None, 0.0, _ptr(out), rows, Cc, L.EPI_RELU,
                                             _stream()), "relu_bwd_f32")
            return out
        L.check(self.lib.a3d_relu_bwd(self.h, _ptr(y), _ptr(dy), lddy, _ptr(out), rows, Cc, _stream()), "relu_bwd")
        return out

    def dense_epilogue_bwd(self, g_post, y, keep_mask, drop_rate, flags, out=None):
        if out is None:
            out = torch.empty_like(g_post)
        if g_post.dtype == torch.float32:
            Cc = g_post.shape[-1]
            L.check(self.lib.a3d_act_bwd_f32(self.h, _ptr(g_post), Cc, _ptr(y), _ptr(keep_mask), drop_rate, _ptr(out),
                                             g_post.numel() // Cc, Cc, flags, _stream()), "act_bwd_f32")
            return out
        L.check(self.lib.a3d_dense_epilogue_bwd(self.h, _ptr(g_post), _ptr(y), _ptr(keep_mask), drop_rate, _ptr(out),
                                                g_post.numel(), flags, _stream()), "dense_epilogue_bwd")
        return out

    def silog_loss(self, out, tar, lambda_over_n=0.5 / 4070, want_grad=True, grad_bf16=False,
                   loss_ps=None, loss=None, dout=None, dout_bf16=None, dout_ld=0):
        B = out.shape[0]
        n = out.numel() // B
        dev = out.device
        loss_ps = loss_ps if loss_ps is not None else torch.empty(B, dtype=torch.float32, device=dev)
        loss = loss if loss is not None else torch.empty(1, dtype=torch.float32, device=dev)
        if want_grad and dout is None and not grad_bf16:
            dout = torch.empty(B, n, dtype=torch.float32, device=dev)
        if want_grad and grad_bf16 and dout_bf16 is None:
            dout_bf16 = torch.empty(B, n, dtype=torch.bfloat16, device=dev)
        L.check(self.lib.a3d_silog_loss(self.h, _ptr(out), _ptr(tar), B, n, lambda_over_n, _ptr(loss_ps), _ptr(loss),
                                        _ptr(dout), _ptr(dout_bf16), dout_ld, _stream()), "silog_loss")
        return loss, loss_ps, dout, dout_bf16

    def adam_tf(self, w, g, m, v, w_bf16, lr, beta1, beta2, eps, t, grad_scale=1.0, n=None, lr_t_dev=None):
        """TF1 ApplyAdam.  `lr_t_dev` (1-element f32 device tensor) overrides the host-computed lr_t."""
        lr_t = adam_lr_t(lr, beta1, beta2, t)
        n = n if n is not None else w.numel()
        L.check(self.lib.a3d_adam_tf(self.h, _ptr(w), _ptr(g), _ptr(m), _ptr(v), _ptr(w_bf16), n, lr_t, beta1, beta2,
                                     eps, grad_scale, _ptr(lr_t_dev), _stream()), "adam")

    def adam_tf_bf16g(self, w, g_bf16, m, v, w_bf16, lr, beta1, beta2, eps, t, grad_scale=1.0, lr_t_dev=None):
        L.check(self.lib.a3d_adam_tf_bf16g(self.h, _ptr(w), _ptr(g_bf16), _ptr(m), _ptr(v), _ptr(w_bf16), w.numel(),
                                           adam_lr_t(lr, beta1, beta2, t), beta1, beta2, eps, grad_scale,
                                           _ptr(lr_t_dev), _stream()), "adam_bf16g")

    def sgd(self, w, g, w_bf16, lr, grad_scale=1.0, n=None):
        n = n if n is not None else w.numel()
        L.check(self.lib.a3d_sgd(self.h, _ptr(w), _ptr(g), _ptr(w_bf16), n, lr, grad_scale, _stream()), "sgd")

    def bernoulli_mask(self, keep, keep_prob, seed, counter_dev=None):
        L.check(self.lib.a3d_bernoulli_mask(self.h, _ptr(keep), keep.numel(), keep_prob, seed, _ptr(counter_dev),
                                            _stream()), "bernoulli_mask")

    def increment_i64(self, p):
        L.check(self.lib.a3d_increment_i64(self.h, _ptr(p), _stream()), "increment")

    def cast_f32_bf16(self, src, dst=None):
        if dst is None:
            dst = torch.empty(src.shape, dtype=torch.bfloat16, device=src.device)
        L.check(self.lib.a3d_cast_f32_bf16(self.h, _ptr(src), _ptr(dst), src.numel(), _stream()), "cast")
        return dst

    def scatter_channel_bf16(self, src, dst, ch):
        ld = dst.shape[-1]
        if dst.dtype == torch.float32:
            L.check(self.lib.a3d_scatter_channel_f32(self.h, _ptr(src), _ptr(dst), src.numel(), ld, ch, _stream()),
                    "scatter_channel_f32")
            return
        L.check(self.lib.a3d_scatter_channel_bf16(self.h, _ptr(src), _ptr(dst), src.numel(), ld, ch, _stream()),
                "scatter_channel")

    def space_to_depth2(self, src, out):
        N, H, W, Cc = src.shape
        L.check(self.lib.a3d_space_to_depth2(self.h, _ptr(src), N, H, W, Cc, _ptr(out), _stream()), "space_to_depth2")
        return out

    def fill_zero(self, t):
        L.check(self.lib.a3d_fill_zero(self.h, _ptr(t), t.numel() * t.element_size(), _stream()), "fill_zero")

    def apply_mask_f32(self, g, keep, n=None):
        L.check(self.lib.a3d_apply_mask_f32(self.h, _ptr(g), _ptr(keep), n if n is not None else g.numel(), _stream()),
                "apply_mask")

    # ------------------------------------------------------------------ conv / dense
    def conv_ws(self, d, op, tf32=False):
        fn = self.lib.a3d_conv2d_ws_bytes_tf32 if tf32 else self.lib.a3d_conv2d_ws_bytes
        nbytes = fn(self.h, C.byref(d), op)
        return self.workspace(("conv_tf32" if tf32 else "conv", op), nbytes), nbytes

    def conv2d_fwd(self, d, x, w, bias, relu=False, out=None, out_dtype=torch.bfloat16):
        if out is None:
            out = torch.empty(d.N, d.P, d.Q, d.ldy, dtype=torch.float32 if x.dtype == torch.float32 else out_dtype,
                              device=x.device)
        if x.dtype == torch.float32:               # TF32 mode (tcgen05 kind::tf32); K == 1: exact float32 stencil
            if d.K == 1:
                L.check(self.lib.a3d_conv_k1_fwd_f32(self.h, C.byref(d), _ptr(x), _ptr(w), _ptr(bias), _ptr(out),
                                                     L.EPI_RELU if relu else 0, _stream()), "conv_k1_fwd_f32")
                return out
            if self.tf32x3:                        # 3xTF32: hi/lo operand split, float32-grade products
                nb = self.lib.a3d_conv2d_ws_bytes_tf32x3(self.h, C.byref(d))
                ws = self.workspace(("conv_tf32x3",), nb)
                L.check(self.lib.a3d_conv2d_fwd_tf32x3(self.h, C.byref(d), _ptr(x), _ptr(w), _ptr(bias), _ptr(out),
                                                       L.EPI_RELU if relu else 0, _ptr(ws), ws.numel(), _stream()),
                        "conv2d_fwd_tf32x3")
                return out
            ws, nb = self.conv_ws(d, L.OP_FWD, tf32=True)
            L.check(self.lib.a3d_conv2d_fwd_tf32(self.h, C.byref(d), _ptr(x), _ptr(w), _ptr(bias), _ptr(out),
                                                 L.EPI_RELU if relu else 0, _ptr(ws), ws.numel(), _stream()),
                    "conv2d_fwd_tf32")
            return out
        ws, nb = self.conv_ws(d, L.OP_FWD)
        code = L.A3D_BF16 if out.dtype == torch.bfloat16 else L.A3D_F32
        L.check(self.lib.a3d_conv2d_fwd(self.h, C.byref(d), _ptr(x), _ptr(w), _ptr(bias), _ptr(out), code,
                                        L.EPI_RELU if relu else 0, _ptr(ws), ws.numel(), _stream()), "conv2d_fwd")
        return out

    def conv2d_dgrad_prepare(self, d, w, out=None):
        """Flipped, channel-transposed filter for conv2d_dgrad(wflip=...); None when the shape's dgrad does not use one."""
        if out is None:
            out = torch.empty(d.C, d.R, d.S, d.K, dtype=torch.bfloat16, device=w.device)
        rc = self.lib.a3d_conv2d_dgrad_prepare(self.h, C.byref(d), _ptr(w), _ptr(out), _stream())
        if rc == L.A3D_ENOTSUP:
            return None
        L.check(rc, "conv2d_dgrad_prepare")
        return out

    def conv2d_dgrad(self, d, dy, w, out=None, relu_src=None, wflip=None):
        """relu_src: post-ReLU activation that was the layer's input -> fused ReluGrad of the producer.
        wflip: filter prepared by conv2d_dgrad_prepare (w is then unused)."""
        if out is None:
            out = torch.empty(d.N, d.H, d.W, d.C, dtype=dy.dtype, device=dy.device)
        if dy.dtype == torch.float32:
            if d.K == 1:
                L.check(self.lib.a3d_conv_k1_dgrad_f32(self.h, C.byref(d), _ptr(dy), _ptr(w), _ptr(out), _ptr(relu_src),
                                                       _stream()), "conv_k1_dgrad_f32")
                return out
            ws, nb = self.conv_ws(d, L.OP_DGRAD, tf32=True)
            L.check(self.lib.a3d_conv2d_dgrad_tf32(self.h, C.byref(d), _ptr(dy), _ptr(w), _ptr(out), _ptr(relu_src),
                                                   _ptr(ws), ws.numel(), _stream()), "conv2d_dgrad_tf32")
            return out
        ws, nb = self.conv_ws(d, L.OP_DGRAD)
        if wflip is not None:
            L.check(self.lib.a3d_conv2d_dgrad_prepared(self.h, C.byref(d), _ptr(dy), _ptr(wflip), _ptr(out), _ptr(relu_src),
                                                       _ptr(ws), ws.numel(), _stream()), "conv2d_dgrad_prepared")
            return out
        L.check(self.lib.a3d_conv2d_dgrad(self.h, C.byref(d), _ptr(dy), _ptr(w), _ptr(out), _ptr(relu_src), _ptr(ws),
                                          ws.numel(), _stream()), "conv2d_dgrad")
        return out

    def conv2d_wgrad(self, d, x, dy, dw=None, db=None):
        if dw is None:
            dw = torch.empty(d.K, d.R, d.S, d.C, dtype=torch.float32, device=x.device)
        if x.dtype == torch.float32:
            if d.K == 1:
                L.check(self.lib.a3d_conv_k1_wgrad_f32(self.h, C.byref(d), _ptr(x), _ptr(dy), _ptr(dw), _ptr(db), _stream()),
                        "conv_k1_wgrad_f32")
                return dw, db
            L.check(self.lib.a3d_conv2d_wgrad_tf32(self.h, C.byref(d), _ptr(x), _ptr(dy), _ptr(dw), _ptr(db), _stream()),
                    "conv2d_wgrad_tf32")
            return dw, db
        ws, nb = self.conv_ws(d, L.OP_WGRAD)
        L.check(self.lib.a3d_conv2d_wgrad(self.h, C.byref(d), _ptr(x), _ptr(dy), _ptr(dw), _ptr(db), _ptr(ws),
                                          ws.numel(), _stream()), "conv2d_wgrad")
        return dw, db

    def dense_fwd(self, x, w, bias, flags=0, keep_mask=None, drop_rate=0.0, out=None, out_dtype=torch.bfloat16,
                  impl=L.IMPL_AUTO, ldx=None):
        M = x.shape[0]
        N, K = w.shape
        ldx = ldx or x.shape[1]
        if out is None:
            out = torch.empty(M, N, dtype=torch.float32 if x.dtype == torch.float32 else out_dtype, device=x.device)
        if x.dtype == torch.float32 and self.tf32x3:
            nb = self.lib.a3d_dense_ws_bytes_tf32x3(M, N, K)
            ws = self.workspace(("dense_tf32x3",), nb)
            L.check(self.lib.a3d_dense_fwd_tf32x3(self.h, _ptr(x), ldx, _ptr(w), _ptr(bias), _ptr(keep_mask), drop_rate,
                                                  _ptr(out), _ptr(ws), ws.numel(), M, N, K, flags, _stream()),
                    "dense_fwd_tf32x3")
            return out
        acc = self.workspace(("dense_acc", M, N), M * N * 4)
        if x.dtype == torch.float32:
            L.check(self.lib.a3d_dense_fwd_tf32(self.h, _ptr(x), ldx, _ptr(w), _ptr(bias), _ptr(keep_mask), drop_rate,
                                                _ptr(out), _ptr(acc), M, N, K, flags, _stream()), "dense_fwd_tf32")
            return out
        code = L.A3D_BF16 if out.dtype == torch.bfloat16 else L.A3D_F32
        L.check(self.lib.a3d_dense_fwd(self.h, _ptr(x), ldx, _ptr(w), _ptr(bias), _ptr(keep_mask), drop_rate,
                                       _ptr(out), code, _ptr(acc), M, N, K, flags, impl, _stream()), "dense_fwd")
        return out

    def dense_dgrad(self, dy, w, out=None, impl=L.IMPL_AUTO):
        """dy may be wider than N (row stride = dy.shape[1]); only the first N columns are used."""
        M, lddy = dy.shape
        N, K = w.shape
        if out is None:
            out = torch.empty(M, K, dtype=dy.dtype, device=dy.device)
        acc = self.workspace(("dense_dacc", M, K), M * K * 4)
        if dy.dtype == torch.float32:
            L.check(self.lib.a3d_dense_dgrad_tf32(self.h, _ptr(dy), lddy, _ptr(w), _ptr(out), _ptr(acc), M, N, K, None, None,
                                                  0.0, 0, _stream()), "dense_dgrad_tf32")
            return out
        L.check(self.lib.a3d_dense_dgrad(self.h, _ptr(dy), lddy, _ptr(w), _ptr(out), _ptr(acc), M, N, K, impl,
                                         _stream()), "dense_dgrad")
        return out

    def dense_dgrad_act(self, dy, w, y_act, keep_mask=None, drop_rate=0.0, flags=L.EPI_RELU, out=None, impl=L.IMPL_AUTO):
        """dense_dgrad + DropoutGrad + ReluGrad/SigmoidGrad of the producer layer in one finishing pass."""
        M, lddy = dy.shape
        N, K = w.shape
        if out is None:
            out = torch.empty(M, K, dtype=dy.dtype, device=dy.device)
        acc = self.workspace(("dense_dacc", M, K), M * K * 4)
        if dy.dtype == torch.float32:
            L.check(self.lib.a3d_dense_dgrad_tf32(self.h, _ptr(dy), lddy, _ptr(w), _ptr(out), _ptr(acc), M, N, K,
                                                  _ptr(y_act), _ptr(keep_mask), drop_rate, flags, _stream()),
                    "dense_dgrad_tf32")
            return out
        L.check(self.lib.a3d_dense_dgrad_act(self.h, _ptr(dy), lddy, _ptr(w), _ptr(out), _ptr(acc), M, N, K, impl,
                                             _ptr(y_act), _ptr(keep_mask), drop_rate, flags, _stream()), "dense_dgrad_act")
        return out

    def dense_wgrad(self, x, dy, dw=None, db=None, impl=L.IMPL_AUTO, N=None):
        """dw[N,K] = dy[:, :N]^T x ; row strides are the tensors' own (dy may be a column slice of a wider matrix)."""
        M = dy.shape[0]
        lddy, ldx = dy.stride(0), x.stride(0)
        N = N if N is not None else (dw.shape[0] if dw is not None else dy.shape[1])
        K = x.shape[1]
        if dw is None:
            dw = torch.empty(N, K, dtype=torch.float32, device=x.device)
        if x.dtype == torch.float32:
            L.check(self.lib.a3d_dense_wgrad_tf32(self.h, _ptr(x), ldx, _ptr(dy), lddy, _ptr(dw), _ptr(db), M, N, K,
                                                  _stream()), "dense_wgrad_tf32")
            return dw, db
        L.check(self.lib.a3d_dense_wgrad(self.h, _ptr(x), ldx, _ptr(dy), lddy, _ptr(dw), _ptr(db), M, N, K, impl,
                                         _stream()), "dense_wgrad")
        return dw, db

    def dense_wgrad_adam(self, x, dy, db, w, m, v, w_bf16, lr, beta1, beta2, eps, t, grad_scale=1.0, lr_t_dev=None):
        """dense wgrad with TF-Adam fused into its epilogue (w/m/v: f32 [N,K] views of the arena)."""
        M, lddy = dy.shape
        N, K = w.shape
        L.check(self.lib.a3d_dense_wgrad_adam(self.h, _ptr(x), x.shape[1], _ptr(dy), lddy, _ptr(db), _ptr(w), _ptr(m),
                                              _ptr(v), _ptr(w_bf16), M, N, K, adam_lr_t(lr, beta1, beta2, t), beta1,
                                              beta2, eps, grad_scale, _ptr(lr_t_dev), _stream()), "dense_wgrad_adam")

    def bias_grad_bf16(self, dy, C_, db, rows=None, ld=None, group_rows=0, group_stride=0):
        if rows is None:
            rows, ld = dy.shape
        if dy.dtype == torch.float32:
            L.check(self.lib.a3d_bias_grad_f32(self.h, _ptr(dy), rows, C_, ld, _ptr(db), _stream()), "bias_grad_f32")
            return db
        L.check(self.lib.a3d_bias_grad_bf16(self.h, _ptr(dy), rows, C_, ld, _ptr(db), group_rows, group_stride,
                                            _stream()), "bias_grad")
        return db

    def debug_tc_gemm(self, A, B, M, N, K, bn, kcb=128, a_mn=False, b_mn=False, splits=1, variant=0):
        """variant (K-major operands only): 0 default, 1 deeper stage ring, 2 256-row tile, 3 both, 11 / 12 CTA pair
        (tcgen05 cta_group::2) with a short / deep ring (tc_gemm.cu)"""
        D = torch.empty(M, N, dtype=torch.float32, device=A.device)
        L.check(self.lib.a3d_debug_tc_gemm_v(self.h, _ptr(A), _ptr(B), _ptr(D), M, N, K, bn, kcb, int(a_mn), int(b_mn),
                                             splits, variant, _stream()), "debug_tc_gemm")
        return D

    def debug_tc_gemm_tf32(self, A, B, M, N, K, bn, kcb=128, a_mn=False, b_mn=False, splits=1):
        """f32 operands consumed as TF32 (tcgen05.mma kind::tf32): D[M,N] = A . B^T"""
        D = torch.empty(M, N, dtype=torch.float32, device=A.device)
        L.check(self.lib.a3d_debug_tc_gemm_tf32(self.h, _ptr(A), _ptr(B), _ptr(D), M, N, K, bn, kcb, int(a_mn), int(b_mn),
                                                splits, _stream()), "debug_tc_gemm_tf32")
        return D

    def debug_tc_gemm_fp8(self, A, B, M, N, K, bn, kcb=128, splits=1, rs=None, rs_div=1, cs=None):
        """E4M3 operands (tcgen05.mma kind::f8f6f4), A [M,K] and B [N,K] codes: D[M,N] = A . B^T (x rs[m // rs_div] x cs[n])"""
        D = torch.empty(M, N, dtype=torch.float32, device=A.device)
        L.check(self.lib.a3d_debug_tc_gemm_fp8(self.h, _ptr(A), _ptr(B), _ptr(D), M, N, K, bn, kcb, splits, _ptr(rs), rs_div,
                                               _ptr(cs), _stream()), "debug_tc_gemm_fp8")
        return D

    # ------------------------------------------------------------------ FP8 inference (include/a3d.h "FP8 inference")
    def quantize_rows_e4m3(self, x, q=None, scale=None):
        """Per-row E4M3 codes of a bf16 matrix (rows = x.shape[0], the rest flattened): (q float8_e4m3fn, scale f32 [rows])."""
        rows = x.shape[0]
        cols = x.numel() // rows
        if q is None:
            q = torch.empty(x.shape, dtype=torch.float8_e4m3fn, device=x.device)
        if scale is None:
            scale = torch.empty(rows, dtype=torch.float32, device=x.device)
        L.check(self.lib.a3d_quantize_rows_e4m3(self.h, _ptr(x), rows, cols, cols, _ptr(q), _ptr(scale), _stream()),
                "quantize_rows_e4m3")
        return q, scale

    def _quant_ws(self, B, n):
        return self.workspace(("quant_e4m3",), self.lib.a3d_quantize_ws_bytes_e4m3(B, n))

    def quantize_e4m3(self, x, out=None, scale=None):
        """Per-image E4M3 codes of a bf16 tensor [B, ...]: (out float8_e4m3fn, scale f32 [B])."""
        B = x.shape[0]
        n = x.numel() // B
        if out is None:
            out = torch.empty(x.shape, dtype=torch.float8_e4m3fn, device=x.device)
        if scale is None:
            scale = torch.empty(B, dtype=torch.float32, device=x.device)
        ws = self._quant_ws(B, n)
        L.check(self.lib.a3d_quantize_e4m3(self.h, _ptr(x), B, n, _ptr(out), _ptr(scale), _ptr(ws), ws.numel(), _stream()),
                "quantize_e4m3")
        return out, scale

    def maxpool2x2_quantize_e4m3(self, x, out=None, scale=None, ldy=None):
        """2x2/2 max-pool of bf16 [B,H,W,C] into per-image E4M3 codes [B,H/2,W/2,ldy] (channels >= C zero)."""
        B, H, W, Cc = x.shape
        ldy = ldy or (out.shape[-1] if out is not None else Cc)
        if out is None:
            out = torch.empty(B, H // 2, W // 2, ldy, dtype=torch.float8_e4m3fn, device=x.device)
        if scale is None:
            scale = torch.empty(B, dtype=torch.float32, device=x.device)
        ws = self._quant_ws(B, (H // 2) * (W // 2) * ldy)
        L.check(self.lib.a3d_maxpool2x2_quantize_e4m3(self.h, _ptr(x), B, H, W, Cc, _ptr(out), ldy, _ptr(scale), _ptr(ws),
                                                      ws.numel(), _stream()), "maxpool2x2_quantize_e4m3")
        return out, scale

    def resize_bilinear_tf1_s2d_e4m3(self, src, OH, OW, out=None):
        """Resize + space-to-depth(4) of f32 or uint8 images [B,H,W,3] into E4M3 codes of 256 * value [B,OH/4,OW/4,64]."""
        B, H, W, Cc = src.shape
        if out is None:
            out = torch.empty(B, OH // 4, OW // 4, 64, dtype=torch.float8_e4m3fn, device=src.device)
        sd = L.A3D_U8 if src.dtype == torch.uint8 else L.A3D_F32
        L.check(self.lib.a3d_resize_bilinear_tf1_s2d_e4m3(self.h, _ptr(src), sd, B, H, W, Cc, _ptr(out), OH, OW, 4,
                                                          out.shape[-1], _stream()), "resize_s2d_e4m3")
        return out

    def conv2d_fwd_fp8(self, d, x, x_scale, w, w_scale, bias, relu=False, out=None, out_dtype=torch.bfloat16):
        if out is None:
            out = torch.empty(d.N, d.P, d.Q, d.ldy, dtype=out_dtype, device=x.device)
        ws, nb = self.conv_ws(d, L.OP_FWD)
        code = L.A3D_BF16 if out.dtype == torch.bfloat16 else L.A3D_F32
        L.check(self.lib.a3d_conv2d_fwd_fp8(self.h, C.byref(d), _ptr(x), _ptr(x_scale), _ptr(w), _ptr(w_scale), _ptr(bias),
                                            _ptr(out), code, L.EPI_RELU if relu else 0, _ptr(ws), ws.numel(), _stream()),
                "conv2d_fwd_fp8")
        return out

    def conv2d_pool4_fwd_fp8(self, d, x, x_scale, w, w_scale, bias, relu=True, out=None):
        if out is None:
            out = torch.empty(d.N, d.P, d.Q, d.ldy, dtype=torch.bfloat16, device=x.device)
        L.check(self.lib.a3d_conv2d_pool4_fwd_fp8(self.h, C.byref(d), _ptr(x), _ptr(x_scale), _ptr(w), _ptr(w_scale),
                                                  _ptr(bias), _ptr(out), L.EPI_RELU if relu else 0, _stream()),
                "conv2d_pool4_fwd_fp8")
        return out

    def dense_fwd_fp8(self, x, x_scale, w, w_scale, bias, flags=0, out=None, out_dtype=torch.bfloat16):
        M, K = x.shape[0], x.shape[1]
        N = w.shape[0]
        if out is None:
            out = torch.empty(M, N, dtype=out_dtype, device=x.device)
        acc = self.workspace(("dense_acc", M, N), M * N * 4)
        code = L.A3D_BF16 if out.dtype == torch.bfloat16 else L.A3D_F32
        L.check(self.lib.a3d_dense_fwd_fp8(self.h, _ptr(x), x.stride(0), _ptr(x_scale), _ptr(w), _ptr(w_scale), _ptr(bias),
                                           _ptr(out), code, _ptr(acc), M, N, K, flags, _stream()), "dense_fwd_fp8")
        return out

    # ------------------------------------------------------------------ DCNF
    def pairwise_dense(self, sims, w2, b1, out=None):
        n = sims.numel() // 2
        if out is None:
            out = torch.empty(sims.shape[:-1], dtype=torch.float32, device=sims.device)
        L.check(self.lib.a3d_pairwise_dense(self.h, _ptr(sims), _ptr(w2), _ptr(b1), _ptr(out), n, _stream()),
                "pairwise_dense")
        return out

    def pairwise_dense_act(self, sims, w2, b1, flags=0, out=None):
        """r = act(sims . w + b); flags = EPI_RELU clamps r at 0 (beyond the reference: keeps the CRF matrix SPD)."""
        n = sims.numel() // 2
        if out is None:
            out = torch.empty(sims.shape[:-1], dtype=torch.float32, device=sims.device)
        L.check(self.lib.a3d_pairwise_dense_act(self.h, _ptr(sims), _ptr(w2), _ptr(b1), _ptr(out), n, flags, _stream()),
                "pairwise_dense_act")
        return out

    def pairwise_dense_bwd(self, sims, r, dr, dw2, db1, flags=0):
        """gradient of the 2 -> 1 pairwise layer from the CRF's dr (beyond the reference)"""
        L.check(self.lib.a3d_pairwise_dense_bwd(self.h, _ptr(sims), _ptr(r), _ptr(dr), _ptr(dw2), _ptr(db1), r.numel(), flags,
                                                _stream()), "pairwise_dense_bwd")

    def mean_f32(self, v, out):
        L.check(self.lib.a3d_mean_f32(self.h, _ptr(v), v.numel(), _ptr(out), _stream()), "mean")
        return out

    def scale_cast_bf16(self, src, dst, scale=1.0):
        L.check(self.lib.a3d_scale_cast_bf16(self.h, _ptr(src), _ptr(dst), src.numel(), scale, _stream()),
                "scale_cast")
        return dst

    def crf(self, z, y, r, pl, pr, grad_scale=1.0, want_dz=True, want_dr=False, naive=False, out=None):
        B, n = z.shape[0], z.shape[1]
        n_pairs = r.shape[1]
        dev = z.device
        f32 = dict(dtype=torch.float32, device=dev)
        if out is not None:
            ystar, nll, logdet = out["ystar"], out["nll"], out["logdet"]
            dz, dr, status = out.get("dz"), out.get("dr"), out["status"]
        else:
            ystar = torch.empty(B, n, **f32)
            nll = torch.empty(B, **f32)
            logdet = torch.empty(B, **f32)
            dz = torch.empty(B, n, **f32) if want_dz else None
            dr = torch.empty(B, n_pairs, **f32) if want_dr else None
            status = torch.empty(B, dtype=torch.int32, device=dev)
        L.check(self.lib.a3d_crf_fwd_bwd(self.h, _ptr(z), _ptr(y), _ptr(r), _ptr(pl), _ptr(pr), B, n, n_pairs,
                                         grad_scale, int(naive), _ptr(ystar), _ptr(nll), _ptr(logdet), _ptr(dz),
                                         _ptr(dr), _ptr(status), _stream()), "crf")
        return dict(ystar=ystar, nll=nll, logdet=logdet, dz=dz, dr=dr, status=status)

    def pairwise_features(self, images, pl, pr, gamma=1.0, out=None):
        B, H, W, _ = images.shape
        n_pairs = pl.numel()
        ws = self.workspace(("pairwise", B, H, W), self.lib.a3d_pairwise_ws_bytes(B, H, W))
        sims = out if out is not None else torch.empty(B, n_pairs, 2, dtype=torch.float32, device=images.device)
        L.check(self.lib.a3d_pairwise_features(self.h, _ptr(images), B, H, W, _ptr(pl), _ptr(pr), n_pairs, gamma,
                                               _ptr(ws), _ptr(sims), _stream()), "pairwise_features")
        return sims

    def tile_means(self, depth, out=None):
        B, H, W = depth.shape[:3]
        n = math.ceil(H / 40) * math.ceil(W / 40)
        y = out if out is not None else torch.empty(B, n, dtype=torch.float32, device=depth.device)
        L.check(self.lib.a3d_tile_means(self.h, _ptr(depth), B, H, W, _ptr(y), _stream()), "tile_means")
        return y

    def extract_patches(self, images, dstC=16, out=None):
        B, H, W, _ = images.shape
        n = math.ceil(H / 40) * math.ceil(W / 40)
        if out is None:
            out = torch.empty(B * n, 100, 100, dstC, dtype=torch.bfloat16, device=images.device)
        dstC = out.shape[-1]
        L.check(self.lib.a3d_extract_patches(self.h, _ptr(images), B, H, W, _ptr(out), dstC, _stream()),
                "extract_patches")
        return out

    def extract_patches_s2d(self, images, out, fold=1):
        """DCNF patches after space-to-depth(2): out bf16 [B*n, 50, 50, 16*fold] (a3d_extract_patches_s2d)."""
        B, H, W, _ = images.shape
        L.check(self.lib.a3d_extract_patches_s2d(self.h, _ptr(images), B, H, W, _ptr(out), fold, _stream()),
                "extract_patches_s2d")
        return out

    def image_cells_s2d(self, images, pad, out):
        """Zero-padded image after space-to-depth(2): out bf16 [B, (H+2pad)/2, (W+2pad)/2, 16] (a3d_image_cells_s2d)."""
        B, H, W, _ = images.shape
        L.check(self.lib.a3d_image_cells_s2d(self.h, _ptr(images), B, H, W, pad, _ptr(out), _stream()), "image_cells_s2d")
        return out

    def window_gather(self, src, rows, cols, win, stride, out):
        B, Hs, Ws, Cc = src.shape
        L.check(self.lib.a3d_window_gather(self.h, _ptr(src), B, Hs, Ws, Cc, rows, cols, win, stride, _ptr(out), _stream()),
                "window_gather")
        return out

    def window_scatter_sum(self, g_out, rows, cols, win, stride, g_src):
        B, Hs, Ws, Cc = g_src.shape
        L.check(self.lib.a3d_window_scatter_sum(self.h, _ptr(g_out), B, Hs, Ws, Cc, rows, cols, win, stride, _ptr(g_src),
                                                _stream()), "window_scatter_sum")
        return g_src

    # ------------------------------------------------------------------ evaluation
    def depth_metrics(self, pred, gt, min_depth, max_depth, median=False, sums=None, scale=None):
        """pred f32 [B,ph,pw(,1)], gt f32 [B,gh,gw(,1)] -> sums f64 [B, len(L.DM_SLOTS)] (a3d_depth_metrics);
        `scale` f32 [B] (optional) receives the median scale."""
        B, ph, pw = pred.shape[:3]
        gh, gw = gt.shape[1:3]
        if gt.shape[0] != B or pred.dim() == 4 and pred.shape[3] != 1 or gt.dim() == 4 and gt.shape[3] != 1:
            raise ValueError("depth_metrics: pred [B,ph,pw(,1)] and gt [B,gh,gw(,1)] with the same B")
        for t in (pred, gt):
            if t.dtype != torch.float32 or not t.is_cuda or not t.is_contiguous():
                raise ValueError("depth_metrics: pred and gt must be contiguous float32 CUDA tensors")
        if sums is None:
            sums = torch.empty(B, len(L.DM_SLOTS), dtype=torch.float64, device=pred.device)
        mode = L.DM_SCALE_MEDIAN if median else L.DM_SCALE_NONE
        L.check(self.lib.a3d_depth_metrics(self.h, _ptr(pred), B, ph, pw, _ptr(gt), gh, gw, min_depth, max_depth, mode,
                                           _ptr(sums), _ptr(scale), _stream()), "depth_metrics")
        return sums

    # ------------------------------------------------------------------ data parallel
    def comm_init(self, id_bytes: bytes, rank: int, nranks: int, nccl_path: str | None = None):
        buf = C.create_string_buffer(id_bytes, 128)
        L.check(self.lib.a3d_comm_init(self.h, nccl_path.encode() if nccl_path else None, buf, rank, nranks),
                "comm_init")
        self._world = nranks

    def allreduce_sum(self, t, count=None):
        code = L.A3D_BF16 if t.dtype == torch.bfloat16 else L.A3D_F32
        L.check(self.lib.a3d_allreduce_sum(self.h, _ptr(t), count if count is not None else t.numel(), code,
                                           _stream()), "allreduce")

    def reduce_scatter_sum(self, t, chunk):
        """In place on t (world*chunk elements): afterwards rank r holds the sum in t[r*chunk:(r+1)*chunk]."""
        L.check(self.lib.a3d_reduce_scatter_sum(self.h, _ptr(t), chunk, _code(t), _stream()), "reduce_scatter")

    def allgather_multi(self, tensors):
        """Grouped in-place all-gather of several equal-dtype tensors (each world * chunk elements): one NCCL launch."""
        n = len(tensors)
        ptrs = (C.c_void_p * n)(*[t.data_ptr() for t in tensors])
        chunks = (C.c_size_t * n)(*[t.numel() // self._world for t in tensors])
        L.check(self.lib.a3d_allgather_multi(self.h, ptrs, chunks, n, _code(tensors[0]), _stream()), "allgather_multi")

    def allgather(self, t, chunk):
        """In place on t (world*chunk elements): publishes every rank's slice t[r*chunk:(r+1)*chunk]."""
        L.check(self.lib.a3d_allgather(self.h, _ptr(t), chunk, _code(t), _stream()), "allgather")


class StepTimeline:
    """Per-stream time marks INSIDE a captured step (the whole step is one CUDA graph, so it cannot be timed call by
    call): `ctx.stamp(label)` enqueues a one-thread kernel that stores the GPU's global timer when its stream gets there.
    Every enqueue of the step (warm-up, capture) re-registers the same labels in the same order; a graph replay then
    refreshes the slots and `read()` returns [(label, stream id, microseconds since the first mark)]."""

    def __init__(self, device, capacity=256):
        self.slots = torch.zeros(capacity, dtype=torch.int64, device=device)
        self.labels, self.n = [], 0

    def begin(self):
        self.n = 0

    def mark(self, ctx, label):
        st = torch.cuda.current_stream()
        if self.n < len(self.labels):
            self.labels[self.n] = (label, st.cuda_stream)
        else:
            self.labels.append((label, st.cuda_stream))
        L.check(ctx.lib.a3d_stamp(ctx.h, C.c_void_p(self.slots[self.n:].data_ptr()), C.c_void_p(st.cuda_stream)), "stamp")
        self.n += 1

    def read(self):
        torch.cuda.synchronize()
        t = self.slots[:self.n].cpu().tolist()
        t0 = min(t) if t else 0
        return [(lab, st, (ti - t0) / 1e3) for (lab, st), ti in zip(self.labels[:self.n], t)]


def _code(t):
    return L.A3D_BF16 if t.dtype == torch.bfloat16 else L.A3D_F32


def reduce_scatter_sum(ctx, t, chunk):
    ctx.reduce_scatter_sum(t, chunk)


def allgather(ctx, t, chunk):
    ctx.allgather(t, chunk)


def comm_unique_id(nccl_path: str | None = None) -> bytes:
    lib = L.load()
    buf = C.create_string_buffer(128)
    L.check(lib.a3d_comm_unique_id(nccl_path.encode() if nccl_path else None, buf), "comm_unique_id")
    return buf.raw
