"""Training-time augmentation of Eigen, Puhrsch & Fergus (NIPS 2014, section 3.3) restated on CPU (oracle; test
infrastructure only).  The contract the CUDA kernels of ``ann3depth_b200/csrc/augment.cu`` follow (``a3d_augment_desc``,
include/a3d.h):

* per image: scale s, rotation theta (degrees), crop centre c = (c_x, c_y), flip bit, colour factor c_rgb, crop fraction f;
* output pixel (oy, ox) of an OH x OW output sits at the TF1 legacy position (u, v) = (ox * W/OW, oy * H/OH), normalised to
  p = (u/W, v/H) and mapped by T(p) = c + R(theta) F (p - 1/2) f/s, R a rotation in the pixel space of a frame of
  height/width ``aspect``, F = diag(+-1, 1);
* the source is sampled at T(p) * (W, H) with TF1 bilinear, coordinates clamped to [0, W-1] x [0, H-1];
* images are multiplied by c_rgb after interpolation, depths by 1/s.

The parameter draw is a splitmix64 hash of (seed, step counter, image index) mapped to the ranges in float64, so the
sequence does not depend on the build and a resumed run continues it.
"""
from __future__ import annotations

import math

import numpy as np
import torch

# packed parameter row (A3D_AUG_* of include/a3d.h)
M00, M01, M02, M10, M11, M12 = range(6)
COLOR, INV_SCALE, SCALE, THETA, FLIP, CX, CY, CROP = 6, 9, 10, 11, 12, 13, 14, 15
NPARAMS = 16
N_DRAWS = 8           # uniforms per image: scale, theta, c_x, c_y, flip, c_r, c_g, c_b
_M64 = (1 << 64) - 1


def mix64(x: int) -> int:
    """splitmix64 finaliser (bernoulli_mask_kernel / augment_draw_kernel)."""
    x = (x + 0x9E3779B97F4A7C15) & _M64
    x = ((x ^ (x >> 30)) * 0xBF58476D1CE4E5B9) & _M64
    x = ((x ^ (x >> 27)) * 0x94D049BB133111EB) & _M64
    return x ^ (x >> 31)


def uniforms(seed: int, counter: int, index: int) -> list[float]:
    """The N_DRAWS uniforms in [0, 1) of image `index` at step `counter` (53-bit mantissas)."""
    base = mix64((seed & _M64) ^ mix64(counter & _M64))
    return [(mix64((base + index * N_DRAWS + j) & _M64) >> 11) * 2.0 ** -53 for j in range(N_DRAWS)]


def params_from(s, theta_deg, cx, cy, flip, color, crop, aspect=0.75):
    """Packed float64 row of explicit parameters."""
    k = crop / s
    fl = -1.0 if flip else 1.0
    rad = theta_deg * (math.pi / 180.0)
    cs, sn = math.cos(rad), math.sin(rad)
    m00, m01 = cs * fl * k, -sn * aspect * k
    m10, m11 = sn / aspect * fl * k, cs * k
    row = np.zeros(NPARAMS, dtype=np.float64)
    row[M00:M12 + 1] = (m00, m01, cx - 0.5 * (m00 + m01), m10, m11, cy - 0.5 * (m10 + m11))
    row[COLOR:COLOR + 3] = color
    row[INV_SCALE], row[SCALE], row[THETA], row[FLIP], row[CX], row[CY], row[CROP] = (
        1.0 / s, s, theta_deg, 1.0 if flip else 0.0, cx, cy, crop)
    return row


def identity_params(batch: int) -> torch.Tensor:
    return torch.tensor(np.stack([params_from(1.0, 0.0, 0.5, 0.5, False, (1.0, 1.0, 1.0), 1.0)] * batch),
                        dtype=torch.float32)


def draw(ranges: dict, batch: int, seed: int, counter: int) -> torch.Tensor:
    """[batch, 16] float64 parameters.  ranges: scale_lo, scale_hi, max_rotation_deg, crop_fraction, flip_prob, color_lo,
    color_hi, aspect (the a3d_augment_desc fields; the kernel reads them as float32, so pass float32-representable
    values or round them first)."""
    r = {k: float(np.float32(v)) for k, v in ranges.items()}
    rows = []
    for b in range(batch):
        u = uniforms(seed, counter, b)
        s = r["scale_lo"] + (r["scale_hi"] - r["scale_lo"]) * u[0]
        theta = r["max_rotation_deg"] * (2.0 * u[1] - 1.0)
        half = 0.5 * (1.0 - r["crop_fraction"] / s)
        cx, cy = 0.5 + half * (2.0 * u[2] - 1.0), 0.5 + half * (2.0 * u[3] - 1.0)
        flip = u[4] < r["flip_prob"]
        color = [r["color_lo"] + (r["color_hi"] - r["color_lo"]) * u[5 + c] for c in range(3)]
        rows.append(params_from(s, theta, cx, cy, flip, color, r["crop_fraction"], r["aspect"]))
    return torch.tensor(np.stack(rows), dtype=torch.float64)


def _tf1_positions(n_in: int, n_out: int) -> torch.Tensor:
    """TF1 legacy source positions dst * (in/out), scale and product in float32 (tf1_ops.resize_bilinear_tf1)."""
    scale = torch.tensor(float(n_in), dtype=torch.float32) / torch.tensor(float(n_out), dtype=torch.float32)
    return (torch.arange(n_out, dtype=torch.float32) * scale).to(torch.float64)


def source_coords(params: torch.Tensor, H: int, W: int, OH: int, OW: int):
    """Unclamped source pixel coordinates (x, y) [B, OH, OW] float64 of every output pixel under each image's map."""
    p = params.to(torch.float64)
    u = _tf1_positions(W, OW).view(1, 1, OW)
    v = _tf1_positions(H, OH).view(1, OH, 1)
    col = lambda i: p[:, i].view(-1, 1, 1)
    x = col(M00) * u + col(M01) * (W / H) * v + col(M02) * W
    y = col(M10) * (H / W) * u + col(M11) * v + col(M12) * H
    return x, y


def resize_affine_tf1(x: torch.Tensor, out_h: int, out_w: int, params: torch.Tensor, mode: str = "color"):
    """x [B, H, W, C] -> [B, out_h, out_w, C] in x's dtype: the transformed TF1 bilinear resize.  mode "color": times
    c_rgb per channel, "depth": times 1/s.  Coordinates are float64; the interpolation runs in x's dtype with the
    operation order of tf1_ops.resize_bilinear_tf1, so identity parameters reproduce that function exactly."""
    b, h, w, c = x.shape
    dt = x.dtype
    xs, ys = source_coords(params, h, w, out_h, out_w)
    xs = xs.clamp(0, w - 1)
    ys = ys.clamp(0, h - 1)
    x0, y0 = torch.floor(xs).long(), torch.floor(ys).long()
    x1, y1 = (x0 + 1).clamp(max=w - 1), (y0 + 1).clamp(max=h - 1)
    lx, ly = (xs - x0).to(dt).unsqueeze(-1), (ys - y0).to(dt).unsqueeze(-1)
    bi = torch.arange(b).view(b, 1, 1)
    tl, tr = x[bi, y0, x0], x[bi, y0, x1]
    bl, br = x[bi, y1, x0], x[bi, y1, x1]
    top = tl + (tr - tl) * lx
    bot = bl + (br - bl) * lx
    out = top + (bot - top) * ly
    p = params.to(dt)
    if mode == "color":
        assert c <= 3
        return out * p[:, COLOR:COLOR + c].view(b, 1, 1, c)
    if mode == "depth":
        return out * p[:, INV_SCALE].view(b, 1, 1, 1)
    raise ValueError(mode)


def space_to_depth(x: torch.Tensor, s: int, dst_c: int) -> torch.Tensor:
    """[B, OH, OW, C] -> [B, OH/s, OW/s, dst_c]: channel (dy*s + dx)*C + c, zero beyond s*s*C."""
    b, oh, ow, c = x.shape
    y = x.view(b, oh // s, s, ow // s, s, c).permute(0, 1, 3, 2, 4, 5).reshape(b, oh // s, ow // s, s * s * c)
    return torch.nn.functional.pad(y, (0, dst_c - s * s * c))
