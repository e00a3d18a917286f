"""Oracle of the scale-and-shift-invariant loss (include/a3d.h a3d_ssi_loss; MiDaS, Ranftl et al. 2020).

Per image, prediction p and target g of n = H*W values (row-major H x W):
    (s, t) = argmin sum (s*p + t - g)^2,  r = s*p + t - g
    L = sum r^2 / (2n) + alpha * sum_k (1/n_k) sum_pairs |r_a - r_b|
where scale k = 0..scales-1 keeps the pixels with y % 2^k == 0 and x % 2^k == 0 (n_k of them) and its pairs are the
horizontally or vertically adjacent points of that grid.  A constant prediction gets s = 0, t = mean g.

`ssi_loss` is the mathematics in float64 torch, differentiable with autograd.  `ssi_loss_points` is the closed form of
loss and gradient in numpy; with rounded=True it keeps the kernel's storage points (float32 s, t, r and differences,
float64 sums), which is what the CUDA kernel is compared with, sign for sign.  `msdn_forward` / `msdn_grads` are the MSDN
oracle's `forward` / `grads` (oracle/msdn.py) with this loss in place of silog, as `models.msdn(..., loss="ssi")` trains.
"""
from __future__ import annotations

from collections import OrderedDict

import numpy as np
import torch

from . import msdn as OM


def grid_sizes(H, W, scales):
    """n_k = |G_k| for k < scales."""
    return [(-(-H // 2 ** k)) * (-(-W // 2 ** k)) for k in range(scales)]


def _fit(p, g):
    """(s, t) of each row by least squares, in the arithmetic of p; s = 0 for a constant row."""
    n = p.shape[-1]
    Sp, Sg = p.sum(-1), g.sum(-1)
    D = (p * p).sum(-1) - Sp * Sp / n
    N = (p * g).sum(-1) - Sp * Sg / n
    flat = (p.amax(-1) == p.amin(-1)) | (D <= 0)
    s = torch.where(flat, torch.zeros_like(D), N / torch.where(flat, torch.ones_like(D), D))
    return s, (Sg - s * Sp) / n


def ssi_loss(p, g, H, W, alpha=0.5, scales=4):
    """Per-image loss [B] of p, g [B, H*W] (float64 recommended).  Differentiable in p (and g)."""
    B = p.shape[0]
    p, g = p.reshape(B, H * W), g.reshape(B, H * W)
    s, t = _fit(p, g)
    r = (s[:, None] * p + t[:, None] - g).reshape(B, H, W)
    L = (r * r).sum((1, 2)) / (2 * H * W)
    for k, nk in enumerate(grid_sizes(H, W, scales)):
        rk = r[:, ::2 ** k, ::2 ** k]
        L = L + alpha * ((rk[:, :, 1:] - rk[:, :, :-1]).abs().sum((1, 2)) +
                         (rk[:, 1:, :] - rk[:, :-1, :]).abs().sum((1, 2))) / nk
    return L


def ssi_loss_points(p, g, H, W, alpha=0.5, scales=4, rounded=True):
    """(loss [B], gradient [B, H*W]) of the per-image loss, both float64 numpy, by the closed form of include/a3d.h:
    dL/dp_i = s*r_i/n + alpha*(s*c_i + Q*(g_i - Sg/n - 2*sd*(p_i - Sp/n))/D).  The gradient is per image (no 1/B).
    rounded=True: s, t, r and the pair differences are float32 as in the kernel (r = (f32(s*p) + t) - g); False:
    everything float64, which equals autograd of `ssi_loss`."""
    p = np.asarray(p, dtype=np.float32 if rounded else np.float64).reshape(-1, H * W)
    g = np.asarray(g, dtype=np.float32 if rounded else np.float64).reshape(-1, H * W)
    f = np.float32 if rounded else np.float64
    B, n = p.shape
    nks = grid_sizes(H, W, scales)
    losses, grads = np.zeros(B), np.zeros((B, n))
    for b in range(B):
        pb, gb = p[b], g[b]
        pd, gd = pb.astype(np.float64), gb.astype(np.float64)
        Sp, Sg = pd.sum(), gd.sum()
        D = (pd * pd).sum() - Sp * Sp / n
        N = (pd * gd).sum() - Sp * Sg / n
        flat = not (pb.min() < pb.max()) or not (D > 0)
        sd = 0.0 if flat else N / D
        s, t = f(sd), f((Sg - sd * Sp) / n)
        r = ((f(s) * pb).astype(f) + t).astype(f) - gb         # one rounding per operation in float32
        r = r.astype(f).reshape(H, W)
        P = pd.reshape(H, W)
        c = np.zeros((H, W))
        G = Q = 0.0
        for k, nk in enumerate(nks):
            h = 2 ** k
            for dy, dx in ((0, h), (h, 0)):
                ra, rb = r[0:H - dy:h, 0:W - dx:h], r[dy::h, dx::h]
                pa, pb_ = P[0:H - dy:h, 0:W - dx:h], P[dy::h, dx::h]
                m0, m1 = min(ra.shape[0], rb.shape[0]), min(ra.shape[1], rb.shape[1])
                d = (ra[:m0, :m1] - rb[:m0, :m1]).astype(f)
                sig = np.sign(d).astype(np.float64)
                G += np.abs(d.astype(np.float64)).sum() / nk
                Q += (sig * (pa[:m0, :m1] - pb_[:m0, :m1])).sum() / nk
                ca = np.zeros((H, W))
                ca[0:H - dy:h, 0:W - dx:h][:m0, :m1] += sig
                ca[dy::h, dx::h][:m0, :m1] -= sig
                c += ca / nk
        rd = r.astype(np.float64).reshape(-1)
        losses[b] = (rd * rd).sum() / (2 * n) + alpha * G
        if not flat:
            ds = (gd - Sg / n - 2 * sd * (pd - Sp / n)) / D
            grads[b] = float(s) * rd / n + alpha * (float(s) * c.reshape(-1) + Q * ds)
    return losses, grads


def msdn_loss(outputs, targets):
    """The loss of one MSDN map [B, 55, 74, 1] against the resized target: the batch mean, as for silog."""
    B = outputs.shape[0]
    return ssi_loss(outputs.reshape(B, -1), targets.reshape(B, -1), OM.OUT_H, OM.OUT_W, 0.5, 4).mean()


def msdn_forward(p, images, depths, dropout_mask=None, train=True, q=OM._ident):
    """oracle/msdn.py `forward` with loss="ssi": dict(coarse, fine, loss_coarse, loss_fine, images, depths)."""
    im, dp = OM.preprocess(images, depths, q)
    c = OM.coarse(p, im, dropout_mask, train, q)
    f = OM.fine(p, im, c, q)
    return dict(coarse=c, fine=f, loss_coarse=msdn_loss(c, dp), loss_fine=msdn_loss(f, dp), images=im, depths=dp)


def msdn_grads(p, images, depths, dropout_mask, which="coarse", q=OM._ident):
    """oracle/msdn.py `grads` with loss="ssi": 'coarse' -> d loss_coarse / d coarse vars (phase 1), 'fine' -> d loss_fine
    / d fine vars (phase 2), 'all' -> both.  Returns (gradients, forward values)."""
    leaves = OrderedDict((n, v.detach().clone().requires_grad_(True)) for n, v in p.items())
    out = msdn_forward(leaves, images, depths, dropout_mask, True, q)
    res = OrderedDict()
    for key in ("coarse", "fine"):
        if which in (key, "all"):
            names = [n for n in leaves if n.startswith(key + "/")]
            res.update(zip(names, torch.autograd.grad(out["loss_" + key], [leaves[n] for n in names], retain_graph=True)))
    return res, {k: (v.detach() if torch.is_tensor(v) else v) for k, v in out.items()}
