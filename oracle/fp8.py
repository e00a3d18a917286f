"""Oracle of the FP8 inference mode (test infrastructure only): the E4M3 quantiser and the MSDN forward at exactly the
storage points of `MSDNNet(dtype="fp8")` (include/a3d.h "FP8 inference").

Quantiser (float32, as the kernels compute it):  amax = max |x|,  s = amax / 448,  inv = 448 / amax (0 when amax == 0),
code = e4m3(x * inv) with round-to-nearest-even and saturation at +-448.  torch's float8_e4m3fn conversion rounds to
nearest even too but turns overflow into NaN, hence the clamp.  Weights take one scale per output channel (the last axis
of the TF kernel), activations one per image; between the storage points the arithmetic is float64 (oracle/tf1_ops.py).
"""
from __future__ import annotations

import torch

from . import tf1_ops as T
from .msdn import IN_H, IN_W, OUT_H, OUT_W, bf16_round, silog_loss

E4M3_MAX = 448.0
IMAGE_SCALE = 2.0 ** -8          # the resized image lies in [0, 1]: fixed scale, codes of 256 * value


def e4m3(x):
    """float32 -> E4M3 codes (torch.float8_e4m3fn), round to nearest even, saturating."""
    return torch.clamp(x.float(), -E4M3_MAX, E4M3_MAX).to(torch.float8_e4m3fn)


def quantize(x, dims):
    """Codes and float32 scales of x with one scale per index of the axes NOT in `dims` (amax over `dims`)."""
    xf = x.float()
    amax = xf.abs().amax(dim=dims, keepdim=True)
    # a full tensor, not a scalar: torch's CUDA division by a CPU scalar multiplies by its reciprocal (not IEEE division)
    c = torch.full_like(amax, E4M3_MAX)
    inv = torch.where(amax > 0, c / amax, torch.zeros_like(amax))
    scale = amax / c
    return e4m3(xf * inv), scale


def quantize_images(x):
    """Per-image quantisation of [B, ...]: (codes, scale [B])."""
    q, s = quantize(x, tuple(range(1, x.dim())))
    return q, s.reshape(-1)


def quantize_rows(x):
    """Per-row quantisation of [rows, ...] (the operand matrices the kernels read): (codes, scale [rows])."""
    return quantize_images(x)


def dequantize_images(q, s):
    return q.double() * s.double().reshape((-1,) + (1,) * (q.dim() - 1))


def weight(kernel):
    """float64 value of a TF-layout kernel (R,S,C,K) or (in,out) as the FP8 mode stores it: bf16 mirror, then one E4M3
    scale per output channel (the last axis)."""
    wb = bf16_round(kernel.float())
    q, s = quantize(wb, tuple(range(wb.dim() - 1)))
    return q.double() * s.double()


def image_codes(resized):
    """float64 value of the E4M3 image: codes of 256 * float32(resized), scale 2^-8."""
    return e4m3(resized.float() * 256.0).double() * IMAGE_SCALE


def forward(p, images, depths):
    """Inference forward of MSDN in the FP8 mode.  images [B,H,W,3] in [0,1] (float), depths [B,h,w,1].
    Returns dict(coarse [B,55,74,1], fine [B,55,74,1], loss_coarse, loss_fine, scales {storage point: [B]})."""
    def b(n):
        return p[n + "/bias"].double()

    def k(n):
        return weight(p[n + "/kernel"])
    scales = {}

    def q(name, x):
        codes, s = quantize_images(x)
        scales[name] = s
        return dequantize_images(codes, s)
    dev = images.device                 # tf1_ops.resize_bilinear_tf1 builds its index tensors on the CPU
    im = image_codes(T.resize_bilinear_tf1(images.double().cpu(), IN_H, IN_W).to(dev))
    dp = T.resize_bilinear_tf1(depths.double().cpu(), OUT_H, OUT_W).to(dev)
    n = "coarse/conv/conv2d_"
    t = bf16_round(T.conv2d(im, k(n + "0"), b(n + "0"), 4, "valid", True))
    t = q("p0", T.max_pool_2x2(t))
    t = bf16_round(T.conv2d(t, k(n + "1"), b(n + "1"), 1, "same", True))
    t = q("p1", T.max_pool_2x2(t))
    t = q("c2", bf16_round(T.conv2d(t, k(n + "2"), b(n + "2"), 1, "same", True)))
    t = q("c3", bf16_round(T.conv2d(t, k(n + "3"), b(n + "3"), 1, "same", True)))
    t = bf16_round(T.conv2d(t, k(n + "4"), b(n + "4"), 2, "valid", True))
    t = q("c4", t.reshape(t.shape[0], -1))
    t = q("d0", bf16_round(T.dense(t, k("coarse/dense/dense_0"), b("coarse/dense/dense_0"), "relu")))
    coarse = T.dense(t, k("coarse/dense/dense_1"), b("coarse/dense/dense_1"), None).float().double()
    coarse = coarse.reshape(-1, OUT_H, OUT_W, 1)
    f = bf16_round(T.conv2d(im, k("fine/first/conv2d"), b("fine/first/conv2d"), 2, "valid", True))
    f = T.max_pool_2x2(f)
    f = q("cat", torch.cat([f, bf16_round(coarse)], dim=-1))
    f = bf16_round(T.conv2d(f, k("fine/second/conv2d"), b("fine/second/conv2d"), 1, "same", True))
    fine = T.conv2d(f, bf16_round(p["fine/third/kernel"].double()), b("fine/third"), 1, "same", False)
    return dict(coarse=coarse, fine=fine, loss_coarse=silog_loss(coarse, dp), loss_fine=silog_loss(fine, dp),
                scales=scales)
