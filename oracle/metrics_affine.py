"""Float64 restatement of the affine (least-squares scale-and-shift) mode of `a3d_depth_metrics`, A3D_DM_SCALE_AFFINE
(test infrastructure only; the product never imports it).  Everything but the alignment is oracle/metrics.py.

Per image, over the valid pixels min_depth < g <= max_depth, with p~ the clamped prediction of oracle/metrics.py:
  n, mp = sum p~ / n, mg = sum g / n, Sxx = sum p~^2 - sum p~ * mp, Sxy = sum p~ g - sum p~ * mg   (float64)
  sd = Sxy / Sxx (may be negative), or sd = 1 when min p~ = max p~ or Sxx <= 0 (a constant prediction)
  s = float32(sd), t = float32(mg - sd * mp);  s = 1, t = 0 when n = 0
  p = fmin(fmax(float32(float32(s * p~) + t), min_depth), max_depth)   (two float32 roundings, no fused multiply-add;
      a NaN maps to min_depth)
then the slots of oracle/metrics.py on p; the non-finite count is that of the sampled prediction, as in the other modes.
"""
import numpy as np

from . import metrics as M


def affine_fit(pt, g):
    """Clamped predictions p~ and ground truth g of the valid pixels (float32) -> float32 (s, t)."""
    pt = np.asarray(pt, dtype=np.float32).reshape(-1)
    g = np.asarray(g, dtype=np.float32).reshape(-1)
    n = g.size
    if n == 0:
        return np.float32(1.0), np.float32(0.0)
    p64, g64 = pt.astype(np.float64), g.astype(np.float64)
    sp, sg = p64.sum(), g64.sum()
    mp, mg = sp / n, sg / n
    sxx, sxy = (p64 * p64).sum() - sp * mp, (p64 * g64).sum() - sp * mg
    sd = sxy / sxx if pt.min() < pt.max() and sxx > 0 else 1.0
    return np.float32(sd), np.float32(mg - sd * mp)


def image_sums(pred_up, gt, min_depth=1e-3, max_depth=1.0, fit=None):
    """pred_up, gt: float32 arrays of one image on the ground-truth grid -> (slot sums float64 [11], (s, t) float32).
    fit: an (s, t) to apply instead of the least-squares one (to check a kernel's slot sums at its own alignment)."""
    v = np.asarray(pred_up, dtype=np.float32).reshape(-1)
    g = np.asarray(gt, dtype=np.float32).reshape(-1)
    lo, hi = np.float32(min_depth), np.float32(max_depth)
    with np.errstate(invalid="ignore"):
        valid = (g > lo) & (g <= hi)
    pt = np.where(np.isnan(v), lo, np.clip(v, lo, hi)).astype(np.float32)
    s, t = (np.float32(x) for x in (fit if fit is not None else affine_fit(pt[valid], g[valid])))
    with np.errstate(over="ignore", invalid="ignore"):
        p = np.fmin(np.fmax((s * pt).astype(np.float32) + t, lo), hi).astype(np.float32)
    sums, _ = M.image_sums(p, g, min_depth, max_depth)
    sums[M.SLOTS.index("nonfinite")] = int((~np.isfinite(v[valid])).sum())
    return sums, (s, t)
