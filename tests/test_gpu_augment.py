"""Training-time augmentation on the GPU: the kernels against the plain TF1 resizes (bit for bit at identity) and against
oracle/augment.py (random parameters, the draw), and the augmented MSDN / DCNF steps and driver."""
import os
import re
import subprocess
import sys

import pytest
import torch

from ann3depth_b200 import models
from ann3depth_b200.augment import Augment
from oracle import augment as OA

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
EIGEN = Augment.eigen_nyu()
# The kernels form source coordinates in float32 (two fmaf over coefficients rounded to float32); the oracle evaluates
# the same float32 parameters in float64.  At |x| <= 640 each of the ~4 roundings is <= 640 * 2^-24 = 3.8e-5 px, so the
# positions agree to ~1.5e-4 px; U[0,1) pixels change by at most 1 per pixel and the colour factor is <= 1.2, so the
# values agree to ~2e-4.  A bf16 output adds half a bf16 unit (2^-9 relative) on either side.
TOL_F32 = 3e-4


@pytest.fixture(scope="module")
def ctx():
    return models.get_context(0)


def _images(B, H=480, W=640, seed=0, u8=False):
    g = torch.Generator().manual_seed(seed)
    if u8:
        return torch.randint(0, 256, (B, H, W, 3), generator=g, dtype=torch.uint8)
    return torch.rand(B, H, W, 3, generator=g)


def _extreme_params():
    """Max scale / both rotation limits / flipped / corner crops / extreme colours, as float32 rows."""
    rows = []
    f = 0.95
    for s, th, corner, flip, col in ((1.5, 5.0, (-1, -1), True, (0.8, 1.2, 0.8)),
                                     (1.5, -5.0, (1, 1), False, (1.2, 0.8, 1.2)),
                                     (1.0, 5.0, (1, -1), True, (1.2, 1.2, 1.2)),
                                     (1.25, -5.0, (-1, 1), True, (0.8, 0.8, 0.8))):
        half = 0.5 * (1 - f / s)
        rows.append(OA.params_from(s, th, 0.5 + corner[0] * half, 0.5 + corner[1] * half, flip, col, f))
    return torch.tensor(rows, dtype=torch.float32)


def _ref_s2d(x64, params, dst_c=64):
    return OA.space_to_depth(OA.resize_affine_tf1(x64, 228, 304, params.double(), "color"), 4, dst_c)


# ----------------------------------------------------------------------------- identity: bit for bit
@pytest.mark.parametrize("kind", ["f32_bf16", "u8_bf16", "f32_f32"])
def test_s2d_identity_is_bit_identical(ctx, kind):
    B = 3
    x = _images(B, u8=kind.startswith("u8")).cuda()
    dt = torch.float32 if kind.endswith("f32") else torch.bfloat16
    ref = torch.zeros(B, 57, 76, 64, dtype=dt, device="cuda")
    got = torch.full_like(ref, 7.0)
    ctx.resize_bilinear_tf1_s2d(x, 228, 304, 4, out=ref)
    ctx.resize_affine_tf1_s2d(x, 228, 304, 4, OA.identity_params(B).cuda(), out=got)
    torch.cuda.synchronize()
    assert torch.equal(got, ref)


@pytest.mark.parametrize("src,dst", [((480, 640, 3), (228, 304)), ((480, 640, 1), (55, 74)), ((55, 73, 1), (55, 74)),
                                     ((480, 640, 3), (240, 320))])
def test_generic_identity_is_bit_identical(ctx, src, dst):
    B = 3
    g = torch.Generator().manual_seed(1)
    x = (torch.rand(B, *src, generator=g) * 5 + 0.1).cuda()
    ref = ctx.resize_bilinear_tf1(x, *dst)
    got = ctx.resize_affine_tf1(x, *dst, OA.identity_params(B).cuda(), depth=src[-1] == 1)
    torch.cuda.synchronize()
    assert torch.equal(got, ref)


# ----------------------------------------------------------------------------- random parameters vs the oracle
def _drawn(ctx, B, seed=11, counter=5):
    p = torch.zeros(B, 16, device="cuda")
    ctx.augment_draw(EIGEN.desc(), p, seed, torch.tensor([counter], dtype=torch.int64, device="cuda"))
    return p.cpu()


@pytest.mark.parametrize("kind", ["f32_bf16", "u8_bf16", "f32_f32"])
def test_s2d_random_params_match_oracle(ctx, kind):
    params = torch.cat([_extreme_params(), _drawn(ctx, 4)])
    B = params.shape[0]
    u8 = kind.startswith("u8")
    x = _images(B, seed=2, u8=u8)
    dt = torch.float32 if kind.endswith("f32") else torch.bfloat16
    out = torch.full((B, 57, 76, 64), 7.0, dtype=dt, device="cuda")
    ctx.resize_affine_tf1_s2d(x.cuda(), 228, 304, 4, params.cuda(), out=out)
    x64 = x.double() / 255.0 if u8 else x.double()
    ref = _ref_s2d(x64, params)
    got = out.cpu().double()
    err = (got - ref).abs()
    tol = TOL_F32 + (2.0 ** -8 * ref.abs() if dt == torch.bfloat16 else 0.0)
    print(f"{kind}: worst |err| {float(err.max()):.3e}, worst err/tol {float((err / tol).max()):.3f}")
    assert bool((err <= tol).all())
    assert bool((got[..., 48:] == 0).all())


@pytest.mark.parametrize("src,dst", [((480, 640, 3), (228, 304)), ((480, 640, 1), (55, 74)), ((55, 73, 1), (55, 74)),
                                     ((480, 640, 3), (240, 320))])
def test_generic_random_params_match_oracle(ctx, src, dst):
    params = torch.cat([_extreme_params(), _drawn(ctx, 4, seed=12)])
    B = params.shape[0]
    g = torch.Generator().manual_seed(3)
    x = torch.rand(B, *src, generator=g)
    depth = src[-1] == 1
    got = ctx.resize_affine_tf1(x.cuda(), *dst, params.cuda(), depth=depth).cpu().double()
    ref = OA.resize_affine_tf1(x.double(), *dst, params.double(), "depth" if depth else "color")
    err =float((got - ref).abs().max())
    print(f"{src}->{dst}: worst |err| {err:.3e}")
    assert err <= TOL_F32


def test_draw_matches_oracle(ctx):
    B = 64
    for seed, counter in ((0, 0), (2, 1), (12345, 987654321)):
        got = _drawn(ctx, B, seed=seed, counter=counter).double()
        ref = OA.draw(EIGEN.ranges(), B, seed, counter)
        assert torch.equal(got[:, OA.FLIP], ref[:, OA.FLIP].float().double())
        ref32 = ref.float().double()
        assert torch.allclose(got, ref32, rtol=1e-6, atol=1e-7), float((got - ref32).abs().max())
    a, b = _drawn(ctx, B, 0, 3), _drawn(ctx, B, 0, 4)
    assert not torch.equal(a, b)


def test_image_and_target_share_the_transform(ctx):
    """Ramps on the 480x640 image grid and the 55x73 depth grid come out as the ramp at T(p) on their own grids."""
    params = torch.cat([_extreme_params(), _drawn(ctx, 4, seed=13)])
    B = params.shape[0]

    def ramp(h, w, ch):
        yy, xx = torch.meshgrid(torch.arange(h, dtype=torch.float64), torch.arange(w, dtype=torch.float64), indexing="ij")
        r = 0.3 + 0.5 * xx / w + 0.2 * yy / h
        return r.view(1, h, w, 1).expand(B, h, w, ch).contiguous()

    def expect(h, w, oh, ow):
        xs, ys = OA.source_coords(params.double(), h, w, oh, ow)
        xs, ys = xs.clamp(0, w - 1), ys.clamp(0, h - 1)
        return 0.3 + 0.5 * xs / w + 0.2 * ys / h

    img = ramp(480, 640, 3)
    out = torch.zeros(B, 57, 76, 64, dtype=torch.float32, device="cuda")
    ctx.resize_affine_tf1_s2d(img.float().cuda(), 228, 304, 4, params.cuda(), out=out)
    want_img = OA.space_to_depth(expect(480, 640, 228, 304).unsqueeze(-1) * params[:, 6:9].double().view(B, 1, 1, 3), 4, 64)
    e1 = float((out.cpu().double() - want_img).abs().max())
    dep = ramp(55, 73, 1)
    tar = ctx.resize_affine_tf1(dep.float().cuda(), 55, 74, params.cuda(), depth=True).cpu().double()
    want_dep = (expect(55, 73, 55, 74) * params[:, 9].double().view(B, 1, 1)).unsqueeze(-1)
    e2 = float((tar - want_dep).abs().max())
    print(f"ramp image err {e1:.2e}, ramp depth err {e2:.2e}")
    assert e1 < 2e-6 and e2 < 2e-6


# ----------------------------------------------------------------------------- models
def _msdn_params():
    from oracle import msdn as OM
    p = OM.init_params(1, torch.float32, bias_range=0.05)
    p["coarse/dense/dense_1/bias"] += 1.0
    p["fine/third/bias"] += 1.0
    return p


def _msdn_inputs(B, u8=False, seed=0):
    g = torch.Generator().manual_seed(seed)
    images = _images(B, seed=seed, u8=u8).cuda()
    depths = (torch.rand(B, 55, 73, 1, generator=g) * 0.95 + 0.05).cuda()
    return images, depths


@pytest.mark.parametrize("u8,overlap", [(False, True), (True, False)])
def test_msdn_augmented_graph_draws_fresh_params(ctx, u8, overlap):
    B = 2
    images, depths = _msdn_inputs(B, u8)
    op = models.msdn(images, depths, train=True, augment=EIGEN, overlap=overlap)
    op.net.load_params(_msdn_params())
    seen = []
    for _ in range(2):
        op.run(use_graph=True)
        torch.cuda.synchronize()
        seen.append(op.net.aug_params.clone())
        net = op.net
        img4 = torch.empty_like(net.img4)
        ctx.resize_affine_tf1_s2d(images, 228, 304, 4, net.aug_params, out=img4)
        tar = ctx.resize_affine_tf1(depths, 55, 74, net.aug_params, depth=True)
        torch.cuda.synchronize()
        assert torch.equal(img4, net.img4) and torch.equal(tar, net.tar)
        for v in op.losses.values():
            assert torch.isfinite(v).all()
    assert not torch.equal(seen[0], seen[1])
    assert int(op.net.step_dev) == 2
    # the graph drew what the oracle draws at steps 0 and 1
    for step, p in enumerate(seen):
        ref = OA.draw(EIGEN.ranges(), B, op.net.augment_seed, step).float()
        assert torch.allclose(p.cpu(), ref, rtol=1e-6, atol=1e-7)


@pytest.mark.parametrize("u8", [False, True])
def test_msdn_identity_params_match_unaugmented_net(ctx, u8):
    B = 2
    images, depths = _msdn_inputs(B, u8, seed=4)
    aug = models.msdn(images, depths, train=True, augment=EIGEN)
    plain = models.msdn(images, depths, train=True)
    for op in (aug, plain):
        op.net.load_params(_msdn_params())
    aug.net.set_augment_params(OA.identity_params(B).cuda())
    aug.run(use_graph=False)
    plain.run(use_graph=False)
    torch.cuda.synchronize()
    assert torch.equal(aug.net.img4, plain.net.img4) and torch.equal(aug.net.tar, plain.net.tar)
    assert torch.equal(aug.net.aug_params.cpu(), OA.identity_params(B))


def test_msdn_resume_continues_the_draw_sequence(ctx, tmp_path):
    from ann3depth_b200.ann3depth import restore_checkpoint, save_checkpoint
    B = 2
    images, depths = _msdn_inputs(B)
    a = models.msdn(images, depths, train=True, augment=EIGEN)
    a.net.load_params(_msdn_params())
    drawn = []
    for step in range(5):
        a.run(use_graph=True)
        torch.cuda.synchronize()
        drawn.append(a.net.aug_params.clone())
        if step == 2:
            save_checkpoint(a, str(tmp_path))
    b = models.msdn(images, depths, train=True, augment=EIGEN)
    assert restore_checkpoint(b, str(tmp_path)) and b.global_step == 3
    for step in (3, 4):
        b.run(use_graph=True)
        torch.cuda.synchronize()
        assert torch.equal(b.net.aug_params, drawn[step]), step


def test_dcnf_augmented_graph(ctx):
    from ann3depth_b200.init import glorot_params
    B = 2
    g = torch.Generator().manual_seed(5)
    images = torch.rand(B, 480, 640, 3, generator=g).cuda()
    depths = (torch.rand(B, 480, 640, 1, generator=g) * 9 + 0.5).cuda()
    op = models.dcnf(images, depths, train=True, augment=EIGEN)
    op.net.load_params(glorot_params(seed=1, model="dcnf"))
    seen = []
    for _ in range(2):
        op.run(use_graph=True)
        torch.cuda.synchronize()
        net = op.net
        seen.append(net.aug_params.clone())
        im = ctx.resize_affine_tf1(images, 240, 320, net.aug_params, depth=False)
        dp = ctx.resize_affine_tf1(depths, 240, 320, net.aug_params, depth=True)
        torch.cuda.synchronize()
        assert torch.equal(im, net.im) and torch.equal(dp, net.dp)
        assert torch.isfinite(net.loss).all()
    assert not torch.equal(seen[0], seen[1]) and int(op.net.step_dev) == 2
    # injected identity parameters: the unaugmented resizes
    plain = models.dcnf(images, depths, train=True)
    plain.net.load_params(glorot_params(seed=1, model="dcnf"))
    op.net.set_augment_params(OA.identity_params(B).cuda())
    op.run(use_graph=False)
    plain.run(use_graph=False)
    torch.cuda.synchronize()
    assert torch.equal(op.net.im, plain.net.im) and torch.equal(op.net.dp, plain.net.dp)


def test_inference_with_augment_raises():
    images, depths = _msdn_inputs(1)
    with pytest.raises(ValueError):
        models.msdn(images, depths, train=False, augment=EIGEN)
    im = torch.rand(1, 480, 640, 3).cuda()
    dp = torch.rand(1, 480, 640, 1).cuda()
    with pytest.raises(ValueError):
        models.dcnf(im, dp, train=False, augment=EIGEN)


# ----------------------------------------------------------------------------- driver
def _drive(tmp_path, run_id, *extra):
    cmd = [sys.executable, "-u", "-m", "ann3depth_b200.ann3depth", "nyu", "--batchsize", "2", "--ckptdir", str(tmp_path),
           "--datadir", str(tmp_path / "no_data"), "--sumfreq", "1", "--steps", "3", "--id", run_id, *extra]
    r = subprocess.run(cmd, cwd=ROOT, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
    losses = re.findall(r"step (\d+) losses (\{[^}]*\})", r.stdout)
    assert [int(s) for s, _ in losses] == [1, 2, 3]
    return [eval(d) for _, d in losses]


def test_driver_augment_eigen(tmp_path):
    aug = _drive(tmp_path, "aug", "--augment", "eigen")
    plain = _drive(tmp_path, "plain")
    for la, lp in zip(aug, plain):
        assert all(v == v for v in la.values())                 # finite, not NaN
        assert la != lp
