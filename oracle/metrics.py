"""Float64 restatement of the depth-estimation metrics (Eigen et al. 2014) of `a3d_depth_metrics` / `evaluate.DepthMetrics`
(test infrastructure only; the product never imports it).

Per image, over the valid pixels min_depth < g <= max_depth (g and the thresholds in float32):
  p~ = the prediction upsampled to the ground-truth grid (TF1 legacy bilinear, a3d_resize_bilinear_tf1), clamped to
       [min_depth, max_depth]; NaN -> min_depth (and counted as non-finite, like +-inf);
  median scaling: s = float32(median(g) / median(p~)), lower medians (rank floor((n-1)/2)), s = 1 when n = 0;
       p = clamp(s * p~) in float32;  otherwise p = p~;
  d = ln p - ln g.
Slots (ann3depth_b200._lib.DM_SLOTS): n, sum |p-g|/g, sum (p-g)^2/g, sum (p-g)^2, sum d, sum d^2, sum |d|/ln 10, the
counts of max(p/g, g/p) < 1.25, 1.25^2, 1.25^3 (ratios and comparisons in float32), and the non-finite count.
Dataset metrics pool the pixels of all images; silog = sqrt(sum d^2/n - (sum d/n)^2) per image, averaged over the images
with n > 0.
"""
import numpy as np

SLOTS = ("n", "abs_rel", "sq_rel", "sq", "log", "log_sq", "log10", "delta1", "delta2", "delta3", "nonfinite")
METRICS = ("abs_rel", "sq_rel", "rmse", "rmse_log", "log10", "silog", "delta1", "delta2", "delta3")


def image_sums(pred_up, gt, min_depth=1e-3, max_depth=1.0, median=False):
    """pred_up, gt: float32 arrays of one image on the ground-truth grid -> (slot sums float64 [11], scale float32)."""
    v = np.asarray(pred_up, dtype=np.float32).reshape(-1)
    g = np.asarray(gt, dtype=np.float32).reshape(-1)
    lo, hi = np.float32(min_depth), np.float32(max_depth)
    with np.errstate(invalid="ignore"):
        valid = (g > lo) & (g <= hi)
    v, g = v[valid], g[valid]
    nonfinite = int((~np.isfinite(v)).sum())
    pt = np.where(np.isnan(v), lo, np.clip(v, lo, hi)).astype(np.float32)
    n = g.size
    s = np.float32(1.0)
    if median and n:
        k = (n - 1) // 2
        s = np.float32(np.partition(g, k)[k]) / np.float32(np.partition(pt, k)[k])
        p = np.clip(np.float32(s) * pt, lo, hi).astype(np.float32)
    else:
        p = pt
    out = np.zeros(len(SLOTS))
    if n == 0:
        return out, np.float32(s)
    p64, g64 = p.astype(np.float64), g.astype(np.float64)
    d = np.log(p64) - np.log(g64)
    m = np.maximum(p / g, g / p)                         # float32
    out[:] = (n, (np.abs(p64 - g64) / g64).sum(), ((p64 - g64) ** 2 / g64).sum(), ((p64 - g64) ** 2).sum(), d.sum(),
              (d * d).sum(), np.abs(d).sum() / np.log(10.0), (m < np.float32(1.25)).sum(),
              (m < np.float32(1.25) ** 2).sum(), (m < np.float32(1.25) ** 3).sum(), nonfinite)
    return out, np.float32(s)


def dataset_metrics(per_image):
    """per-image slot sums [images, 11] -> {metric: value, images, pixels, nonfinite} (None when no pixel is valid)."""
    per_image = np.asarray(per_image, dtype=np.float64).reshape(-1, len(SLOTS))
    t = per_image.sum(0)
    N = t[0]
    res = {"images": int(per_image.shape[0]), "pixels": int(N), "nonfinite": int(t[10])}
    n = per_image[:, 0]
    has = n > 0
    si = np.sqrt(np.maximum(per_image[has, 5] / n[has] - (per_image[has, 4] / n[has]) ** 2, 0.0))
    if N == 0:
        res.update({k: None for k in METRICS})
        return res
    res.update(abs_rel=t[1] / N, sq_rel=t[2] / N, rmse=np.sqrt(t[3] / N), rmse_log=np.sqrt(t[5] / N), log10=t[6] / N,
               silog=float(si.mean()), delta1=t[7] / N, delta2=t[8] / N, delta3=t[9] / N)
    return {k: (float(v) if isinstance(v, np.floating) else v) for k, v in res.items()}

