"""CPU tests of the affine (least-squares scale-and-shift) evaluation mode: the float64 oracle
(oracle/metrics_affine.py) on known answers, its invariance to an affine map of the prediction, the fallbacks,
`DepthMetrics("affine")` and the `--scale affine` / `--evalscale` flags."""
import numpy as np
import pytest
import torch

from ann3depth_b200.evaluate import DepthMetrics
from oracle import metrics as OM
from oracle import metrics_affine as OA

N, ABS_REL, LOG, LOG10, D1, NONFINITE = (OM.SLOTS.index(k) for k in ("n", "abs_rel", "log", "log10", "delta1",
                                                                         "nonfinite"))


def _p(seed=0, shape=(30, 40), lo=0.2, hi=0.6):
    rng = np.random.default_rng(seed)
    return (rng.uniform(lo, hi, size=shape)).astype(np.float32)


def _assert_same_sums(a, b):
    log_scale = max(b[LOG10] * np.log(10.0), 1e-30)              # the signed sum d can cancel
    for k in range(len(OM.SLOTS)):
        np.testing.assert_allclose(a[k], b[k], rtol=1e-6, atol=1e-6 * log_scale if k == LOG else 0, err_msg=OM.SLOTS[k])


@pytest.mark.parametrize("a,b", [(0.5, 0.125), (1.25, -0.2), (0.8, 0.15), (-0.6, 0.9)])
def test_oracle_exact_affine_ground_truth(a, b):
    p = _p(1)
    g = (p.astype(np.float64) * a + b).astype(np.float32)           # inside (1e-3, 1]: every pixel valid
    assert g.min() > 1e-3 and g.max() <= 1.0
    sums, (s, t) = OA.image_sums(p, g)
    assert s == pytest.approx(a, rel=1e-6) and t == pytest.approx(b, abs=1e-6)
    assert sums[N] == p.size and sums[D1] == p.size
    assert sums[ABS_REL] / sums[N] == pytest.approx(0.0, abs=1e-6)
    r = OM.dataset_metrics(sums[None])
    for k in ("abs_rel", "sq_rel", "rmse", "rmse_log", "log10", "silog"):
        assert r[k] == pytest.approx(0.0, abs=1e-6), k


def test_oracle_fit_is_the_least_squares_solution():
    rng = np.random.default_rng(2)
    p = _p(2, lo=0.1, hi=0.9)
    g = np.clip(0.3 + 0.5 * p + rng.normal(0, 0.05, p.shape), 0.01, 1.0).astype(np.float32)
    _, (s, t) = OA.image_sums(p, g)
    A = np.stack([p.ravel().astype(np.float64), np.ones(p.size)], 1)
    ref, *_ = np.linalg.lstsq(A, g.ravel().astype(np.float64), rcond=None)
    assert s == np.float32(ref[0]) or s == pytest.approx(ref[0], rel=1e-6)
    assert t == pytest.approx(ref[1], rel=1e-6)


@pytest.mark.parametrize("alpha,beta", [(1.6, 0.0), (0.5, 0.3), (-0.5, 0.9), (1.5, 0.05), (-1.0, 1.0)])
def test_oracle_invariant_to_an_affine_map_of_the_prediction(alpha, beta):
    rng = np.random.default_rng(3)
    p = _p(3, lo=0.2, hi=0.6)
    g = np.clip(0.1 + 0.7 * p + rng.normal(0, 0.08, p.shape), 0.0, 1.0).astype(np.float32)
    g[0, :4] = 0.0                                                  # invalid pixels
    q = (p.astype(np.float64) * alpha + beta).astype(np.float32)
    assert q.min() > 1e-3 and q.max() <= 1.0                        # no clamping
    ref, _ = OA.image_sums(p, g)
    got, (s, _) = OA.image_sums(q, g)
    assert np.sign(s) == np.sign(alpha)
    _assert_same_sums(got, ref)


def test_oracle_negative_slope():
    p = _p(4, lo=0.1, hi=0.9)
    g = (0.95 - 0.8 * p.astype(np.float64)).astype(np.float32)
    sums, (s, t) = OA.image_sums(p, g)
    assert s == pytest.approx(-0.8, rel=1e-6) and t == pytest.approx(0.95, rel=1e-6)
    assert sums[D1] == sums[N] == p.size
    plain, _ = OM.image_sums(p, g)                                  # without alignment the same prediction scores badly
    assert plain[D1] < 0.6 * p.size


def test_oracle_no_valid_pixel():
    p = _p(5)
    sums, (s, t) = OA.image_sums(p, np.zeros_like(p))
    assert not sums.any() and s == 1.0 and t == 0.0
    sums, (s, t) = OA.image_sums(np.full_like(p, np.nan), np.full_like(p, 2.0))    # every gt above max_depth
    assert not sums.any() and (s, t) == (1.0, 0.0)


@pytest.mark.parametrize("value", [0.3, 5.0, -1.0], ids=["constant", "clamped-high", "clamped-low"])
def test_oracle_constant_prediction_shifts_only(value):
    g = _p(6, lo=0.05, hi=0.95)
    p = np.full_like(g, value)
    pt = np.float32(np.clip(value, 1e-3, 1.0))
    sums, (s, t) = OA.image_sums(p, g)
    assert s == 1.0 and t == np.float32(g.astype(np.float64).mean() - np.float64(pt))
    ref, _ = OM.image_sums(np.clip(np.full_like(g, pt) + t, 1e-3, 1.0).astype(np.float32), g)
    assert np.array_equal(sums, ref)


def test_oracle_nonfinite_predictions_are_counted_and_clamped():
    g = _p(7, lo=0.05, hi=0.95)
    p = _p(8, lo=0.1, hi=0.9)
    p[0, :5] = np.nan
    p[1, :2] = np.inf
    p[2, :3] = -np.inf
    g[3, :] = 0.0                                                   # invalid row: its NaN does not count
    p[3, :4] = np.nan
    sums, (s, t) = OA.image_sums(p, g)
    assert sums[NONFINITE] == 10 and sums[N] == g.size - g.shape[1]
    pt = np.where(np.isnan(p), np.float32(1e-3), np.clip(p, 1e-3, 1.0)).astype(np.float32)
    assert (s, t) == OA.affine_fit(pt[g > 1e-3], g[g > 1e-3])
    # applying the fit by hand (two float32 roundings) gives the same slots
    ref, _ = OM.image_sums(np.clip((s * pt).astype(np.float32) + t, 1e-3, 1.0).astype(np.float32), g)
    assert np.array_equal(sums[:NONFINITE], ref[:NONFINITE])


def test_oracle_fit_override_applies_the_given_pair():
    g = _p(9, lo=0.05, hi=0.95)
    p = _p(10)
    sums, st = OA.image_sums(p, g, fit=(np.float32(1.0), np.float32(0.0)))
    assert st == (1.0, 0.0)
    assert np.array_equal(sums, OM.image_sums(p, g)[0])


def test_depth_metrics_affine_accumulates_sums():
    rng = np.random.default_rng(11)
    per = []
    for i in range(4):
        p = _p(20 + i, lo=0.1, hi=0.9)
        g = np.clip(0.2 + rng.uniform(-1, 1) * 0.4 * p + rng.normal(0, 0.05, p.shape), 0, 1).astype(np.float32)
        per.append(OA.image_sums(p, g)[0])
    per.append(OA.image_sums(_p(30), np.zeros((30, 40), np.float32))[0])  # no valid pixel
    sums = np.stack(per)
    m = DepthMetrics(None, scale="affine")
    assert m.scale == "affine"
    m.add_sums(torch.from_numpy(sums))
    got, ref = m.result(), OM.dataset_metrics(sums)
    assert got["images"] == 5 and got["pixels"] == ref["pixels"]
    for k in OM.METRICS:
        assert got[k] == pytest.approx(ref[k], rel=1e-12), k
    with pytest.raises(ValueError):
        DepthMetrics(None, scale="shift")


def test_scale_flags():
    from ann3depth_b200 import ann3depth, evaluate
    assert evaluate.parse_args([]).scale == "none"
    assert evaluate.parse_args(["--scale", "affine"]).scale == "affine"
    assert evaluate.parse_args(["--scale", "median"]).scale == "median"
    assert ann3depth.parse_args(["nyu"]).evalscale == "none"
    assert ann3depth.parse_args(["nyu", "--evalfreq", "5", "--evalscale", "affine"]).evalscale == "affine"
    assert ann3depth.parse_args(["nyu", "--evalscale", "median"]).evalscale == "median"
    for parse, flag in ((evaluate.parse_args, "--scale"), (ann3depth.parse_args, "--evalscale")):
        with pytest.raises(SystemExit):
            parse([flag, "shift"])
