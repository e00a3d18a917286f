"""The scale-and-shift-invariant loss on the CPU: the closed-form gradient of include/a3d.h against autograd, the
invariances that make it the right objective for targets known up to a scale and a shift, the storage-point oracle the
CUDA kernel is compared with, and the `--loss` flag of the train driver."""
import numpy as np
import pytest
import torch

from oracle import ssi_loss as S

H, W = 55, 74


def images(B=2, seed=0):
    g = torch.Generator().manual_seed(seed)
    p = torch.randn(B, H * W, generator=g, dtype=torch.float64)
    t = torch.round(torch.rand(B, H * W, generator=g, dtype=torch.float64) * 255) / 255      # k/255, zeros included
    return p, t


def autograd(p, t, alpha=0.5, scales=4):
    p = p.clone().requires_grad_(True)
    L = S.ssi_loss(p, t, H, W, alpha, scales)
    (g,) = torch.autograd.grad(L.sum(), p)
    return L.detach(), g


def rel(a, b):
    a, b = np.asarray(a, dtype=np.float64), np.asarray(b, dtype=np.float64)
    return float(np.abs(a - b).max() / np.abs(b).max())


def test_grid_sizes():
    assert S.grid_sizes(H, W, 4) == [4070, 1036, 266, 70]


@pytest.mark.parametrize("alpha,scales", [(0.5, 4), (0.5, 1), (2.0, 3)])
def test_closed_form_gradient_equals_autograd(alpha, scales):
    p, t = images()
    L, g = autograd(p, t, alpha, scales)
    L2, g2 = S.ssi_loss_points(p.numpy(), t.numpy(), H, W, alpha, scales, rounded=False)
    assert rel(L2, L.numpy()) < 1e-12
    assert rel(g2, g.numpy()) < 1e-12


@pytest.mark.parametrize("a", [3.0, -0.5])
def test_invariant_to_scale_and_shift(a):
    p, t = images()
    L, g = autograd(p, t)
    La, ga = autograd(a * p + 0.7, t)
    assert rel(La.numpy(), L.numpy()) < 1e-12
    assert rel((ga * a).numpy(), g.numpy()) < 1e-10          # the gradient scales as 1/a


def test_exact_fit_has_zero_loss():
    _, t = images()
    L, _ = autograd(-2.5 * t + 4.0, t)
    assert float(L.abs().max()) < 1e-12


def test_alpha_zero_is_the_aligned_mse_gradient():
    p, t = images()
    _, g = autograd(p, t, alpha=0.0)
    s, sh = S._fit(p, t)
    r = s[:, None] * p + sh[:, None] - t
    assert rel(g.numpy(), (s[:, None] * r / (H * W)).numpy()) < 1e-12
    _, g2 = S.ssi_loss_points(p.numpy(), t.numpy(), H, W, 0.0, 4, rounded=False)
    assert rel(g2, g.numpy()) < 1e-12


def test_constant_prediction_gives_zero_scale_and_gradient():
    _, t = images()
    p = torch.full_like(t, 0.3)
    s, sh = S._fit(p, t)
    assert float(s.abs().max()) == 0.0 and torch.allclose(sh, t.mean(1))
    for rounded in (False, True):
        L, g = S.ssi_loss_points(p.numpy(), t.numpy(), H, W, 0.5, 4, rounded=rounded)
        assert np.all(g == 0.0) and np.all(L > 0)


@pytest.mark.parametrize("seed", [0, 1, 2])
def test_storage_points_agree_with_float64(seed):
    p, t = images(3, seed)
    p[1] = -0.3 * t[1] + 0.05 * p[1]                         # negative slope
    for alpha, scales in ((0.5, 4), (0.0, 1)):
        L, g = S.ssi_loss_points(p.numpy(), t.numpy(), H, W, alpha, scales, rounded=False)
        Lr, gr = S.ssi_loss_points(p.float().numpy(), t.float().numpy(), H, W, alpha, scales, rounded=True)
        assert rel(Lr, L) < 1e-5
        for b in range(3):
            assert rel(gr[b], g[b]) < 1e-5


def test_msdn_oracle_with_ssi_loss():
    """msdn_forward / msdn_grads are the MSDN oracle's forward / grads with the ssi loss in place of silog."""
    from oracle import msdn as OM
    g = torch.Generator().manual_seed(0)
    images, depths = torch.rand(1, 48, 64, 3, generator=g, dtype=torch.float64), torch.rand(1, 55, 73, 1, generator=g,
                                                                                           dtype=torch.float64) + 0.05
    prm = OM.init_params(1, torch.float64, bias_range=0.05)
    ref = OM.forward(prm, images, depths, train=False)
    got = S.msdn_forward(prm, images, depths, train=False)
    assert torch.equal(got["coarse"], ref["coarse"]) and torch.equal(got["fine"], ref["fine"])
    B = 1
    for key in ("coarse", "fine"):
        want = S.ssi_loss(ref[key].reshape(B, -1), ref["depths"].reshape(B, -1), H, W).mean()
        assert float(got["loss_" + key]) == float(want)
    mask = torch.ones(1, 4096, dtype=torch.float64)
    gr, fwd = S.msdn_grads(prm, images, depths, mask, "all")
    assert sorted(gr) == sorted(OM.param_names())
    leaf = prm["fine/third/kernel"].clone().requires_grad_(True)
    out = S.msdn_forward(dict(prm, **{"fine/third/kernel": leaf}), images, depths, mask)
    (want,) = torch.autograd.grad(out["loss_fine"], leaf)
    assert torch.allclose(gr["fine/third/kernel"], want, rtol=1e-12, atol=0)


def test_driver_loss_flag():
    from ann3depth_b200 import ann3depth
    assert ann3depth.parse_args([]).loss == "silog"
    assert ann3depth.parse_args(["nyu", "--loss", "ssi"]).loss == "ssi"
    with pytest.raises(SystemExit):
        ann3depth.parse_args(["--loss", "bogus"])
    with pytest.raises(SystemExit):
        ann3depth.parse_args(["--model", "dcnf", "--loss", "ssi"])
    assert ann3depth.parse_args(["--model", "dcnf"]).loss == "silog"


def test_msdn_rejects_unknown_loss():
    from ann3depth_b200.msdn import MSDNNet
    with pytest.raises(ValueError, match="loss"):
        MSDNNet(None, 2, loss="l1")
