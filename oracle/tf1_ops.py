"""TensorFlow-1.3 op semantics restated on CPU tensors (oracle; test infrastructure only).

All tensors are NHWC, conv kernels HWIO, dense kernels [in, out] -- the layouts
``tf.layers`` uses in ``/root/reference/src/models.py``.  Each function names the TF op it
restates and the reference call sites that rely on it.  The TF behaviour itself is not
visible in the reference source (it is inside the tensorflow==1.3.0 wheel); where a detail
is an assumption taken from TF's documented behaviour it is flagged ``ASSUMPTION``.
"""
from __future__ import annotations

import math

import torch
import torch.nn.functional as F


# ----------------------------------------------------------------------------- resize
def resize_axis(n_in: int, n_out: int):
    """(lo, hi, lerp) of one axis of the TF1 legacy bilinear resize: source rows / columns and float32 weights.
    TF computes the scale and the source coordinate in float32 (CalculateResizeScale, `in = dst * scale`), whatever
    the image dtype: mirror that so floor()/lerp agree bit-wise."""
    scale = torch.tensor(float(n_in), dtype=torch.float32) / torch.tensor(float(n_out), dtype=torch.float32)
    src = torch.arange(n_out, dtype=torch.float32) * scale
    lo = torch.floor(src).to(torch.long)
    hi = torch.clamp(lo + 1, max=n_in - 1)
    return lo, hi, src - lo.to(torch.float32)


def resize_bilinear_tf1(x: torch.Tensor, out_h: int, out_w: int) -> torch.Tensor:
    """``tf.image.resize_images(x, [out_h, out_w])`` (BILINEAR, align_corners=False).

    Reference call sites: src/models.py:180-181,189-191 (DCNF), :282-283 (MSDN).
    ASSUMPTION (TF1 legacy kernel): ``src = dst * (in / out)`` (no half-pixel shift),
    ``lo = floor(src)``, ``hi = min(lo + 1, in - 1)``, ``lerp = src - lo``; rows are
    interpolated after columns; input returned unchanged when the size already matches.
    x: [B, H, W, C].
    """
    b, h, w, c = x.shape
    if h == out_h and w == out_w:
        return x
    dt = x.dtype
    ylo, yhi, yl = resize_axis(h, out_h)
    xlo, xhi, xl = resize_axis(w, out_w)
    yl, xl = yl.to(dt), xl.to(dt)
    top = x[:, ylo]                      # [B, out_h, W, C]
    bot = x[:, yhi]
    xl_ = xl.view(1, 1, out_w, 1)
    yl_ = yl.view(1, out_h, 1, 1)
    top_i = top[:, :, xlo] + (top[:, :, xhi] - top[:, :, xlo]) * xl_
    bot_i = bot[:, :, xlo] + (bot[:, :, xhi] - bot[:, :, xlo]) * xl_
    return top_i + (bot_i - top_i) * yl_


# ----------------------------------------------------------------------------- conv / pool / dense
def same_pad(n_in: int, k: int, s: int):
    """TF 'SAME' padding: out = ceil(in/s); total = max((out-1)*s + k - in, 0); extra goes
    to the bottom/right.  Returns (out, pad_lo, pad_hi)."""
    out = -(-n_in // s)
    total = max((out - 1) * s + k - n_in, 0)
    return out, total // 2, total - total // 2


def conv2d(x, kernel, bias=None, stride=1, padding="valid", relu=False):
    """``tf.layers.conv2d`` (Conv2D + BiasAdd [+ Relu]) on NHWC x with an HWIO kernel.

    Reference call sites: src/models.py:64-72 (DCNF unary), :211-223, :241-251 (MSDN).
    ASSUMPTION: tf.layers defaults -- stride 1, padding 'valid', use_bias=True.
    """
    kh, kw, ci, co = kernel.shape
    xn = x.permute(0, 3, 1, 2)
    if padding.lower() == "same":
        _, pt, pb = same_pad(x.shape[1], kh, stride)
        _, pl, pr = same_pad(x.shape[2], kw, stride)
        xn = F.pad(xn, (pl, pr, pt, pb))
    w = kernel.permute(3, 2, 0, 1).contiguous()
    y = F.conv2d(xn, w, bias, stride=stride)
    if relu:
        y = torch.relu(y)
    return y.permute(0, 2, 3, 1)


def max_pool_2x2(x):
    """``tf.layers.max_pooling2d(x, 2, 2)`` -- VALID (odd trailing row/column dropped).
    Reference call sites: src/models.py:65,68,73,213,216,243.  Gradient goes to the (first)
    arg-max of each window (ASSUMPTION: TF MaxPoolGrad behaviour, same as torch)."""
    return F.max_pool2d(x.permute(0, 3, 1, 2), 2, 2).permute(0, 2, 3, 1)


def dense(x, kernel, bias=None, activation=None):
    """``tf.layers.dense``: x @ kernel + bias, kernel is [in, out].
    Reference call sites: src/models.py:80-82,93,228,231."""
    y = x @ kernel
    if bias is not None:
        y = y + bias
    if activation == "relu":
        y = torch.relu(y)
    elif activation == "sigmoid":
        y = torch.sigmoid(y)
    return y


def dropout(x, mask, rate=0.5):
    """``tf.layers.dropout(x, training=True)`` with an explicit keep-mask (the reference's
    mask is unseeded, src/models.py:230, hence unpinnable): y = x * mask / (1 - rate)."""
    return x * mask.to(x.dtype) / (1.0 - rate)


def glorot_uniform_(shape, gen: torch.Generator, dtype=torch.float64):
    """tf.layers default kernel initializer (glorot_uniform): U(-l, l),
    l = sqrt(6 / (fan_in + fan_out)); for HWIO kernels fan = kh*kw*channels."""
    if len(shape) == 2:
        fan_in, fan_out = shape
    else:
        rf = 1
        for s in shape[:-2]:
            rf *= s
        fan_in, fan_out = shape[-2] * rf, shape[-1] * rf
    lim = math.sqrt(6.0 / (fan_in + fan_out))
    return ((torch.rand(shape, generator=gen, dtype=torch.float64) * 2 - 1) * lim).to(dtype)


# ----------------------------------------------------------------------------- patches / histogram
def extract_image_patches_same(x, ksize, stride):
    """``tf.extract_image_patches(x, [1,kh,kw,1], [1,sh,sw,1], [1,1,1,1], 'SAME')``.

    Reference call sites: src/models.py:40-48 (40x40 tiles), :53-59 (100x100 patches).
    ASSUMPTION: zero padding, SAME rule as for convolutions, patch depth ordered
    (row, col, channel).  Returns [B, rows, cols, kh, kw, C].
    """
    kh, kw = ksize
    sh, sw = stride
    b, h, w, c = x.shape
    oh, pt, pb = same_pad(h, kh, sh)
    ow, pl, pr = same_pad(w, kw, sw)
    xp = F.pad(x.permute(0, 3, 1, 2), (pl, pr, pt, pb))          # [B,C,H',W']
    p = xp.unfold(2, kh, sh).unfold(3, kw, sw)                   # [B,C,oh,ow,kh,kw]
    return p.permute(0, 2, 3, 4, 5, 1).contiguous()


def histogram_fixed_width(values, lo, hi, nbins):
    """``tf.histogram_fixed_width(values, (lo, hi), nbins, tf.float32)`` for a 1-D tensor.
    Reference call site: src/models.py:98-99.
    ASSUMPTION: idx = clip(floor(nbins * (v - lo) / (hi - lo)), 0, nbins - 1)."""
    scaled = (values - lo) / (hi - lo)
    idx = torch.clamp(torch.floor(scaled * nbins), 0, nbins - 1).to(torch.long)
    return torch.bincount(idx, minlength=nbins).to(values.dtype)


# ----------------------------------------------------------------------------- optimizers
def tf_adam_update(w, g, m, v, t, lr, beta1=0.9, beta2=0.999, eps=1e-8):
    """One ``tf.train.AdamOptimizer`` apply step (TF1 ApplyAdam), t = 1 for the first step.

        lr_t = lr * sqrt(1 - beta2^t) / (1 - beta1^t)
        m = beta1*m + (1-beta1)*g ; v = beta2*v + (1-beta2)*g*g
        w = w - lr_t * m / (sqrt(v) + eps)

    Reference call site: src/models.py:309 constructs AdamOptimizer(rate, momentum, 1), i.e.
    beta1 = momentum, **beta2 = 1** -> lr_t = 0 and v stays 0: weights never move.
    Returns (w, m, v) new tensors.
    """
    lr_t = lr * math.sqrt(1.0 - beta2 ** t) / (1.0 - beta1 ** t)
    m = beta1 * m + (1.0 - beta1) * g
    v = beta2 * v + (1.0 - beta2) * g * g
    w = w - lr_t * m / (torch.sqrt(v) + eps)
    return w, m, v


def tf_adam_update_(w, g, m, v, t, lr, beta1=0.9, beta2=0.999, eps=1e-8):
    """In-place form of ``tf_adam_update`` (TF updates its variables and slots in place: ApplyAdam writes
    var/m/v, no copies).  Same arithmetic, same order of operations; one temporary the size of the variable."""
    lr_t = lr * math.sqrt(1.0 - beta2 ** t) / (1.0 - beta1 ** t)
    with torch.no_grad():
        m.mul_(beta1).add_(g, alpha=1.0 - beta1)
        v.mul_(beta2).addcmul_(g, g, value=1.0 - beta2)
        w.addcdiv_(m, torch.sqrt(v).add_(eps), value=-lr_t)
    return w, m, v


def sgd_update(w, g, lr):
    """``tf.train.GradientDescentOptimizer(lr)`` apply (src/models.py:198-200)."""
    return w - lr * g
