"""GPU parity tests of the individual liba3d kernels (called through the C-ABI via ctypes).

Dense contractions are checked against an fp32 evaluation of the same bf16 operands (tolerance
2e-3 relative to the output scale: fp32 accumulation-order differences only); elementwise / loss /
optimizer / CRF kernels are checked against the CPU oracle (`oracle/`).
"""
import math

import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu

if torch.cuda.is_available():
    from ann3depth_b200 import _lib as L
    from ann3depth_b200 import ops

from oracle import dcnf as OD
from oracle import msdn as OM
from oracle import tf1_ops as T

import test_gpu_model_launches as ML

DEV = "cuda:0"


@pytest.fixture(scope="module")
def ctx():
    c = ops.Context(0)
    yield c
    torch.cuda.synchronize()
    c.close()


def rel_err(a, b):
    a, b = a.float(), b.float()
    return float((a - b).abs().max() / (b.abs().max() + 1e-20))


def bf16_rand(*shape, seed=0, scale=1.0, shift=0.0):
    g = torch.Generator().manual_seed(seed)
    return ((torch.rand(*shape, generator=g) * 2 - 1) * scale + shift).to(torch.bfloat16).to(DEV)


# ----------------------------------------------------------------------------- tcgen05 engine
@pytest.mark.parametrize("bn,kcb", [(32, 128), (64, 128), (96, 128), (128, 128), (192, 128), (256, 128),
                                    (64, 64), (128, 64), (256, 64), (32, 32), (128, 32)])
def test_tc_gemm_kmajor(ctx, bn, kcb):
    M, N, K = 300, bn + (16 if bn < 256 else 0) - 8, 512
    A = bf16_rand(M, K, seed=1)
    B = bf16_rand(N, K, seed=2)
    D = ctx.debug_tc_gemm(A, B, M, N, K, bn, kcb)
    ref = A.float() @ B.float().t()
    assert rel_err(D, ref) < 2e-3


def test_tc_gemm_kmajor_splitk_long(ctx):
    M, N, K = 260, 128, 64 * 50          # 50 k-blocks > ring depth: exercises phase wrap-around
    A = bf16_rand(M, K, seed=3)
    B = bf16_rand(N, K, seed=4)
    ref = A.float() @ B.float().t()
    assert rel_err(ctx.debug_tc_gemm(A, B, M, N, K, 128, 128, splits=1), ref) < 2e-3
    assert rel_err(ctx.debug_tc_gemm(A, B, M, N, K, 128, 128, splits=5), ref) < 2e-3


@pytest.mark.parametrize("variant", [1, 2, 3])
@pytest.mark.parametrize("bn", [64, 96, 128, 256])
@pytest.mark.parametrize("M", [300, 512, 129, 1000])
def test_tc_gemm_tile_variants(ctx, variant, bn, M):
    """deeper stage rings and 256-row (two-accumulator) tiles; M values leave the second sub-tile empty (129 -> one
    row), partial (300) or absent for the last CTA (1000 = 3 x 256 + 232)"""
    N, K = bn - 8, 64 * 7
    A = bf16_rand(M, K, seed=7)
    B = bf16_rand(N, K, seed=8)
    D = ctx.debug_tc_gemm(A, B, M, N, K, bn, 128, variant=variant)
    assert rel_err(D, A.float() @ B.float().t()) < 2e-3
    if variant >= 2:
        D = ctx.debug_tc_gemm(A, B, M, N, K, bn, 128, splits=3, variant=variant)
        assert rel_err(D, A.float() @ B.float().t()) < 2e-3


@pytest.mark.parametrize("a_mn,b_mn,bn", [(True, True, 128), (True, True, 64), (True, True, 256),
                                          (True, False, 32), (True, False, 128), (False, True, 128)])
def test_tc_gemm_mn_major(ctx, a_mn, b_mn, bn):
    M, N, K = 256, bn, 192
    A = bf16_rand(M, K, seed=5)
    B = bf16_rand(N, K, seed=6)
    ref = A.float() @ B.float().t()
    Ain = A.t().contiguous() if a_mn else A          # MN-major operand is stored [K][rows]
    Bin = B.t().contiguous() if b_mn else B
    D = ctx.debug_tc_gemm(Ain, Bin, M, N, K, bn, 128, a_mn=a_mn, b_mn=b_mn)
    assert rel_err(D, ref) < 2e-3


# ----------------------------------------------------------------------------- convolution
def torch_conv_ref(x_nhwc, w_ohwi, bias, stride, pad_t, pad_l, P, Q, relu):
    """fp32 evaluation of the same bf16 operands on the GPU."""
    x = x_nhwc.float().permute(0, 3, 1, 2)
    w = w_ohwi.float().permute(0, 3, 1, 2)
    R, S = w.shape[2], w.shape[3]
    H, W = x.shape[2], x.shape[3]
    pb = max((P - 1) * stride + R - H - pad_t, 0)
    pr = max((Q - 1) * stride + S - W - pad_l, 0)
    y = F.conv2d(F.pad(x, (pad_l, pr, pad_t, pb)), w, bias, stride=stride)[:, :, :P, :Q]
    if relu:
        y = torch.relu(y)
    return y.permute(0, 2, 3, 1).contiguous()


# (name, H, W, C, K, R, S, stride, padding) -- the MSDN layers (src/models.py:211-251), channel
# counts as stored by the B200 path, plus DCNF-style VALID layers (src/models.py:64-72)
def tf32_round(t):
    """round-to-nearest-even to 10 explicit mantissa bits (what a TFLOAT32 tensor map delivers to shared memory)"""
    i = t.contiguous().view(torch.int32)
    r = (i + 0x0FFF + ((i >> 13) & 1)) & ~0x1FFF
    return r.view(torch.float32)


@pytest.mark.parametrize("a_mn,b_mn,bn,kcb", [(False, False, 128, 128), (False, False, 64, 64), (False, False, 64, 32),
                                               (False, False, 256, 128), (False, False, 16, 128),
                                               (True, True, 128, 128), (True, True, 64, 128), (True, False, 32, 128),
                                               (True, False, 128, 128), (False, True, 128, 128), (False, True, 256, 128)])
@pytest.mark.parametrize("splits", [1, 3])
def test_tc_gemm_tf32(ctx, a_mn, b_mn, bn, kcb, splits):
    """tcgen05.mma kind::tf32 with f32 operands in shared memory, K-major and MN-major, against an f64 product of the
    TF32-rounded operands (exact up to f32 accumulation order) and within 1e-3 of the unrounded f32 product."""
    M, N, K = 128 * 3 + 40, 2 * bn - 8, 32 * 9
    g = torch.Generator().manual_seed(5)
    A = torch.randn(M, K, generator=g).to(DEV)
    B = torch.randn(N, K, generator=g).to(DEV)
    Ad = A.t().contiguous() if a_mn else A
    Bd = B.t().contiguous() if b_mn else B
    if a_mn and M % 4:                                   # MN-major row pitch must be 16-byte aligned
        pytest.skip("unaligned")
    D = ctx.debug_tc_gemm_tf32(Ad, Bd, M, N, K, bn, kcb, a_mn=a_mn, b_mn=b_mn, splits=splits)
    ref_r = (tf32_round(A).double() @ tf32_round(B).double().t())
    ref = A.double() @ B.double().t()
    err_r = float((D.double() - ref_r).abs().max() / ref_r.abs().max())
    err = float((D.double() - ref).abs().max() / ref.abs().max())
    print("tf32 gemm: vs rounded operands", err_r, "vs exact", err)
    assert err_r < 2e-6 and err < 2e-3


LAYERS = [
    ("conv2d_1", 27, 37, 96, 256, 5, 5, 1, "same"),
    ("conv2d_2", 13, 18, 256, 384, 3, 3, 1, "same"),
    ("conv2d_3", 13, 18, 384, 384, 3, 3, 1, "same"),
    ("conv2d_4", 13, 18, 384, 256, 3, 3, 2, "valid"),
    ("fine_second", 55, 74, 64, 64, 5, 5, 1, "same"),
    ("dcnf_conv2d_1", 45, 45, 64, 256, 5, 5, 1, "valid"),
    ("dcnf_conv2d_2", 20, 20, 256, 256, 3, 3, 1, "valid"),
    ("c16_k32", 17, 19, 16, 32, 3, 3, 1, "same"),
    # the two first layers on the space-to-depth(4) image (params.py: conv_kernel_s2d4 / fine_first_embedded)
    ("conv2d_0_s2d4", 57, 76, 64, 96, 3, 3, 1, "valid"),
    ("fine_first_pool_gemm", 57, 76, 64, 256, 3, 3, 1, "valid"),
]
# 3-channel first layers as the B200 path stores them: 4-channel pixels, filter width padded so that
# groups of 16/C pixels can be read as one 16-channel pixel (conv.cu `virtualize`)
PACKED_LAYERS = [
    ("conv2d_0_packed", 228, 304, 4, 96, 11, 12, 4, "valid"),
    ("fine_first_packed", 228, 304, 4, 64, 9, 10, 2, "valid"),
]
SMALL_C_LAYERS = [
    ("conv2d_0", 228, 304, 3, 96, 11, 11, 4, "valid"),
    ("fine_first", 228, 304, 3, 63, 9, 9, 2, "valid"),
    ("fine_third", 55, 74, 64, 1, 5, 5, 1, "same"),
]


@pytest.mark.parametrize("impl", ["simt", "tc"])
@pytest.mark.parametrize("layer", LAYERS, ids=[l[0] for l in LAYERS])
def test_conv_fwd(ctx, layer, impl):
    name, H, W, Cc, K, R, S, stride, padding = layer
    N = 3
    d = ops.conv_desc(N, H, W, Cc, K, R, S, stride, padding, impl=L.IMPL_SIMT if impl == "simt" else L.IMPL_TC)
    x = bf16_rand(N, H, W, Cc, seed=10)
    w = bf16_rand(K, R, S, Cc, seed=11, scale=1.0 / math.sqrt(R * S * Cc))
    bias = (torch.rand(K, generator=torch.Generator().manual_seed(12)) - 0.5).to(DEV)
    y = ctx.conv2d_fwd(d, x, w, bias, relu=True)
    ref = torch_conv_ref(x, w, bias, stride, d.pad_t, d.pad_l, d.P, d.Q, True)
    assert y.shape == ref.shape
    assert rel_err(y, ref) < 1e-2          # output is rounded to bf16 (2^-8 relative)
    yf = ctx.conv2d_fwd(d, x, w, bias, relu=False, out_dtype=torch.float32)
    ref = torch_conv_ref(x, w, bias, stride, d.pad_t, d.pad_l, d.P, d.Q, False)
    assert rel_err(yf, ref) < 2e-3


LAYERS_BY_NAME = {l[0]: l for l in LAYERS}


@pytest.mark.parametrize("variant", [11, 12])
@pytest.mark.parametrize("bn", [64, 96, 128, 192, 256])
@pytest.mark.parametrize("M", [100, 128 * 5 + 7, 128 * 300 + 1])
def test_tc_gemm_cta_pair(ctx, variant, bn, M):
    """tcgen05.mma.cta_group::2 (tc_pair.cuh): 256 x BN tile per CTA pair, each CTA holds half of the B tile.  Fewer rows
    than one CTA (the peer of the only pair is all padding), an odd tile count (ragged last pair), many pairs; two N
    tiles with a clipped last one; K = 9 k-blocks > the short ring's depth."""
    N, K = 2 * bn - 8, 64 * 9
    A = bf16_rand(M, K, seed=7)
    B = bf16_rand(N, K, seed=8)
    D = ctx.debug_tc_gemm(A, B, M, N, K, bn, 128, variant=variant)
    assert rel_err(D, A.float() @ B.float().t()) < 2e-3


@pytest.mark.parametrize("force", ["128,1,1", "128,1,2", "256,1,2", "256,1,3", "64,1,2", "96,1,3", "256,1,11", "128,1,12",
                                   "64,1,11", "192,1,12"])
@pytest.mark.parametrize("layer", [LAYERS_BY_NAME[n] for n in ("conv2d_1", "fine_second", "conv2d_0_s2d4", "dcnf_conv2d_1")],
                         ids=["conv2d_1", "fine_second", "conv2d_0_s2d4", "dcnf_conv2d_1"])
def test_conv_fwd_tile_variants(ctx, monkeypatch, layer, force):
    """im2col-mode A operand with 256-row tiles: the second sub-tile has its own (image, row, column) origin"""
    name, H, W, Cc, K, R, S, stride, padding = layer
    if int(force.split(",")[0]) > K + K // 3 + 15 and K > 64:
        pytest.skip("tile wider than the layer")
    Cc = (Cc + 63) // 64 * 64              # the tile variants exist for 128-byte channel blocks (conv2d_1 is stored with 128)
    N = 3
    d = ops.conv_desc(N, H, W, Cc, K, R, S, stride, padding, impl=L.IMPL_TC)
    x = bf16_rand(N, H, W, Cc, seed=10)
    w = bf16_rand(K, R, S, Cc, seed=11, scale=1.0 / math.sqrt(R * S * Cc))
    bias = (torch.rand(K, generator=torch.Generator().manual_seed(12)) - 0.5).to(DEV)
    monkeypatch.setenv("A3D_CONV_FORCE", force)
    yf = ctx.conv2d_fwd(d, x, w, bias, relu=False, out_dtype=torch.float32)
    yb = ctx.conv2d_fwd(d, x, w, bias, relu=True)
    monkeypatch.delenv("A3D_CONV_FORCE")
    ref = torch_conv_ref(x, w, bias, stride, d.pad_t, d.pad_l, d.P, d.Q, False)
    assert rel_err(yf, ref) < 2e-3
    assert rel_err(yb, torch.relu(ref)) < 1e-2


@pytest.mark.parametrize("layer", SMALL_C_LAYERS, ids=[l[0] for l in SMALL_C_LAYERS])
def test_conv_fwd_small_channels(ctx, layer):
    name, H, W, Cc, K, R, S, stride, padding = layer
    N = 2
    d = ops.conv_desc(N, H, W, Cc, K, R, S, stride, padding, impl=L.IMPL_AUTO)
    x = bf16_rand(N, H, W, Cc, seed=13)
    w = bf16_rand(K, R, S, Cc, seed=14, scale=1.0 / math.sqrt(R * S * Cc))
    yf = ctx.conv2d_fwd(d, x, w, None, relu=False, out_dtype=torch.float32)
    ref = torch_conv_ref(x, w, None, stride, d.pad_t, d.pad_l, d.P, d.Q, False)
    assert rel_err(yf, ref) < 2e-3


@pytest.mark.parametrize("layer", PACKED_LAYERS, ids=[l[0] for l in PACKED_LAYERS])
def test_conv_packed_first_layers(ctx, layer):
    name, H, W, Cc, K, R, S, stride, padding = layer
    N = 2
    d = ops.conv_desc(N, H, W, Cc, K, R, S, stride, padding, impl=L.IMPL_AUTO)
    x = bf16_rand(N, H, W, Cc, seed=17)
    w = bf16_rand(K, R, S, Cc, seed=18, scale=1.0 / math.sqrt(R * S * Cc))
    yf = ctx.conv2d_fwd(d, x, w, None, relu=False, out_dtype=torch.float32)
    ref = torch_conv_ref(x, w, None, stride, d.pad_t, d.pad_l, d.P, d.Q, False)
    assert rel_err(yf, ref) < 2e-3
    dy = bf16_rand(N, d.P, d.Q, K, seed=19)
    wr = w.float().requires_grad_(True)
    yr = F.conv2d(x.float().permute(0, 3, 1, 2), wr.permute(0, 3, 1, 2), None, stride=stride)
    (gw,) = torch.autograd.grad(yr, wr, dy.float().permute(0, 3, 1, 2))
    dw, _ = ctx.conv2d_wgrad(d, x, dy)
    assert rel_err(dw, gw) < 2e-3


def test_conv_fwd_concat_stride(ctx):
    """Output written into a wider NHWC buffer (ldy > K): the concat of src/models.py:246."""
    N, H, W, Cc, K = 2, 20, 24, 32, 48
    d = ops.conv_desc(N, H, W, Cc, K, 3, 3, 1, "same", ldy=64, impl=L.IMPL_TC)
    x = bf16_rand(N, H, W, Cc, seed=15)
    w = bf16_rand(K, 3, 3, Cc, seed=16, scale=0.1)
    out = torch.full((N, H, W, 64), 7.0, dtype=torch.bfloat16, device=DEV)
    ctx.conv2d_fwd(d, x, w, None, relu=False, out=out)
    ref = torch_conv_ref(x, w, None, 1, d.pad_t, d.pad_l, d.P, d.Q, False)
    assert rel_err(out[..., :K], ref) < 1e-2
    assert float((out[..., K:] - 7.0).abs().max()) == 0.0


@pytest.mark.parametrize("impl", ["simt", "auto"])
@pytest.mark.parametrize("layer", LAYERS, ids=[l[0] for l in LAYERS])
def test_conv_dgrad_wgrad(ctx, layer, impl):
    name, H, W, Cc, K, R, S, stride, padding = layer
    N = 2
    d = ops.conv_desc(N, H, W, Cc, K, R, S, stride, padding, impl=L.IMPL_SIMT if impl == "simt" else L.IMPL_AUTO)
    x = bf16_rand(N, H, W, Cc, seed=20)
    w = bf16_rand(K, R, S, Cc, seed=21, scale=1.0 / math.sqrt(R * S * Cc))
    dy = bf16_rand(N, d.P, d.Q, K, seed=22)
    xr = x.float().requires_grad_(True)
    wr = w.float().requires_grad_(True)
    pb = max((d.P - 1) * stride + R - H - d.pad_t, 0)
    pr = max((d.Q - 1) * stride + S - W - d.pad_l, 0)
    yr = F.conv2d(F.pad(xr.permute(0, 3, 1, 2), (d.pad_l, pr, d.pad_t, pb)), wr.permute(0, 3, 1, 2), None,
                  stride=stride)[:, :, :d.P, :d.Q]
    gx, gw = torch.autograd.grad(yr, (xr, wr), dy.float().permute(0, 3, 1, 2))
    dx = ctx.conv2d_dgrad(d, dy, w)
    assert rel_err(dx, gx) < 1e-2
    xpos = torch.relu(x)                                     # fused ReluGrad of the producing layer
    dxr = ctx.conv2d_dgrad(d, dy, w, relu_src=xpos)
    assert rel_err(dxr, gx * (xpos.float().permute(0, 3, 1, 2).permute(0, 2, 3, 1) > 0)) < 1e-2
    db = torch.empty(K, dtype=torch.float32, device=DEV)
    dw, _ = ctx.conv2d_wgrad(d, x, dy, db=db)
    assert rel_err(dw, gw) < 2e-3
    assert rel_err(db, dy.float().sum((0, 1, 2))) < 2e-3


def test_conv_dgrad_prepared_filter(ctx):
    """a3d_conv2d_dgrad_prepare + a3d_conv2d_dgrad_prepared == a3d_conv2d_dgrad """
    for name in ("conv2d_1", "conv2d_2", "conv2d_3"):
        _, H, W, Cc, K, R, S, stride, padding = LAYERS_BY_NAME[name]
        Cc = (Cc + 63) // 64 * 64
        d = ops.conv_desc(2, H, W, Cc, K, R, S, stride, padding, impl=L.IMPL_AUTO)
        w = bf16_rand(K, R, S, Cc, seed=21, scale=1.0 / math.sqrt(R * S * Cc))
        dy = bf16_rand(2, d.P, d.Q, K, seed=22)
        src = torch.relu(bf16_rand(2, H, W, Cc, seed=23))
        wf = ctx.conv2d_dgrad_prepare(d, w)
        assert wf is not None
        a = ctx.conv2d_dgrad(d, dy, w, relu_src=src)
        b = ctx.conv2d_dgrad(d, dy, None, relu_src=src, wflip=wf)
        assert torch.equal(wf, w.permute(3, 1, 2, 0).flip(1, 2).contiguous())
        assert rel_err(a, b) < 1e-2        # two tunings / split-K orders: at most one bf16 ulp (2^-7 relative) apart
    _, H, W, Cc, K, R, S, stride, padding = LAYERS_BY_NAME["conv2d_4"]      # strided: no flipped filter
    d = ops.conv_desc(2, H, W, Cc, K, R, S, stride, padding, impl=L.IMPL_AUTO)
    assert ctx.conv2d_dgrad_prepare(d, bf16_rand(K, R, S, Cc, seed=21)) is None


@pytest.mark.parametrize("force", ["4,1,256", "2,5,256", "3,2,256", "1,3,256"])
@pytest.mark.parametrize("layer", [("k256", 27, 37, 128, 256, 5, 5, 1, "same"), ("k384", 13, 18, 256, 384, 3, 3, 1, "same"),
                                   ("k256_s2", 13, 18, 384, 256, 3, 3, 2, "valid")], ids=["k256", "k384", "k256_s2"])
def test_conv_wgrad_256_filter_tiles(ctx, monkeypatch, layer, force):
    """weight gradient with two 128-filter accumulators per CTA sharing the im2col stages of X (MN-major A, BM = 256);
    384 filters = one full and one half tile"""
    name, H, W, Cc, K, R, S, stride, padding = layer
    N = 3
    d = ops.conv_desc(N, H, W, Cc, K, R, S, stride, padding, impl=L.IMPL_TC)
    x = bf16_rand(N, H, W, Cc, seed=20)
    dy = bf16_rand(N, d.P, d.Q, K, seed=21)
    monkeypatch.setenv("A3D_WGRAD_FORCE", force)
    dw, _ = ctx.conv2d_wgrad(d, x, dy)
    monkeypatch.setenv("A3D_WGRAD_FORCE", force.replace(",256", ",128"))
    dw_ref, _ = ctx.conv2d_wgrad(d, x, dy)
    monkeypatch.delenv("A3D_WGRAD_FORCE")
    wr = torch.zeros(K, R, S, Cc, device=DEV).requires_grad_(True)
    pb = max((d.P - 1) * stride + R - H - d.pad_t, 0)
    pr = max((d.Q - 1) * stride + S - W - d.pad_l, 0)
    yr = F.conv2d(F.pad(x.float().permute(0, 3, 1, 2), (d.pad_l, pr, d.pad_t, pb)), wr.permute(0, 3, 1, 2), None,
                  stride=stride)[:, :, :d.P, :d.Q]
    (gw,) = torch.autograd.grad(yr, (wr,), dy.float().permute(0, 3, 1, 2))
    assert rel_err(dw, gw) < 2e-3
    assert rel_err(dw, dw_ref) < 1e-3


# ----------------------------------------------------------------------------- dense
@pytest.mark.parametrize("impl", ["simt", "tc"])
@pytest.mark.parametrize("M,N,K", [(32, 4096, 12288), (32, 4070, 4096), (8, 128, 12544), (5, 200, 256), (300, 136, 256),
                                   (512, 264, 128)])
def test_dense_fwd(ctx, impl, M, N, K):
    x = bf16_rand(M, K, seed=30)
    w = bf16_rand(N, K, seed=31, scale=1.0 / math.sqrt(K))
    bias = (torch.rand(N, generator=torch.Generator().manual_seed(32)) - 0.5).to(DEV)
    mask = (torch.rand(M, N, generator=torch.Generator().manual_seed(33)) < 0.5).to(torch.uint8).to(DEV)
    code = L.IMPL_SIMT if impl == "simt" else L.IMPL_TC
    y = ctx.dense_fwd(x, w, bias, flags=L.EPI_RELU, keep_mask=mask, drop_rate=0.5, out_dtype=torch.float32, impl=code)
    ref = torch.relu(x.float() @ w.float().t() + bias) * mask.float() * 2.0
    assert rel_err(y, ref) < 2e-3
    y2 = ctx.dense_fwd(x, w, bias, flags=0, out_dtype=torch.float32, impl=code)
    assert rel_err(y2, x.float() @ w.float().t() + bias) < 2e-3


@pytest.mark.parametrize("impl", ["simt", "tc"])
@pytest.mark.parametrize("M,N,K,ld", [(32, 4070, 4096, 4096), (32, 4096, 12288, 4096), (6, 136, 256, 136)])
def test_dense_bwd(ctx, M, N, K, ld, impl):
    code = L.IMPL_SIMT if impl == "simt" else L.IMPL_TC
    x = bf16_rand(M, K, seed=34)
    w = bf16_rand(N, K, seed=35, scale=1.0 / math.sqrt(K))
    dyp = torch.zeros(M, ld, dtype=torch.bfloat16, device=DEV)     # padded row stride
    dyp[:, :N] = bf16_rand(M, N, seed=36)
    dy = dyp[:, :N]
    dx = ctx.dense_dgrad(dyp, w, impl=code)
    assert rel_err(dx, dy.float() @ w.float()) < 1e-2
    db = torch.empty(N, dtype=torch.float32, device=DEV)
    dw, _ = ctx.dense_wgrad(x, dyp, db=db, N=N, impl=code)
    assert rel_err(dw, dy.float().t() @ x.float()) < 2e-3
    assert rel_err(db, dy.float().sum(0)) < 2e-3


@pytest.mark.parametrize("M,N,K", [(32, 4096, 12288), (32, 4070, 4096), (7, 300, 192), (32, 256, 64), (1, 4070, 4096)])
def test_dense_stream_kernels(ctx, monkeypatch, M, N, K):
    """csrc/dense_stream.cu (weight-streaming mma.sync path for batch <= 32), forced with A3D_DENSE_FORCE=101,
    against fp32 evaluation of the same bf16 operands and against an unsplit tcgen05 tile (A3D_DENSE_FORCE=1)."""
    x = bf16_rand(M, K, seed=40)
    w = bf16_rand(N, K, seed=41, scale=1.0 / math.sqrt(K))
    bias = (torch.rand(N, generator=torch.Generator().manual_seed(42)) - 0.5).to(DEV)
    mask = (torch.rand(M, N, generator=torch.Generator().manual_seed(43)) < 0.5).to(torch.uint8).to(DEV)
    ld = (N + 7) // 8 * 8 + 8
    dyp = torch.full((M, ld), float("nan"), dtype=torch.bfloat16, device=DEV)     # padding must never be read as data
    dyp[:, :N] = bf16_rand(M, N, seed=44)
    dy = dyp[:, :N]
    out = {}
    for mode in ("101", "1"):
        monkeypatch.setenv("A3D_DENSE_FORCE", mode)
        n0 = ctx.launches
        y = ctx.dense_fwd(x, w, bias, flags=L.EPI_RELU, keep_mask=mask, drop_rate=0.5, out_dtype=torch.float32, impl=L.IMPL_TC)
        dx = ctx.dense_dgrad(dyp, w, impl=L.IMPL_TC)
        torch.cuda.synchronize()
        assert ctx.launches > n0
        out[mode] = (y, dx)
    ref_y = torch.relu(x.float() @ w.float().t() + bias) * mask.float() * 2.0
    ref_dx = dy.float() @ w.float()
    for mode in ("101", "1"):
        assert rel_err(out[mode][0], ref_y) < 2e-3, mode
        assert rel_err(out[mode][1], ref_dx) < 1e-2, mode
    assert rel_err(out["101"][0], out["1"][0]) < 1e-3


@pytest.mark.parametrize("H,W,R,pad", [(55, 74, 5, "same"), (9, 13, 3, "same"), (12, 20, 5, "valid"), (3, 150, 5, "same")])
def test_conv_k1_tiled(ctx, monkeypatch, H, W, R, pad):
    """single-filter 64-channel convolution (MSDN fine/third): tiled mma.sync kernel vs torch and vs the GEMM path"""
    N, Cc = 3, 64
    d = ops.conv_desc(N, H, W, Cc, 1, R, R, 1, pad)
    x = bf16_rand(N, H, W, Cc, seed=50)
    w = bf16_rand(1, R, R, Cc, seed=51, scale=1.0 / math.sqrt(R * R * Cc))
    bias = torch.tensor([0.37], device=DEV)
    ref = torch_conv_ref(x, w, bias, 1, d.pad_t, d.pad_l, d.P, d.Q, False)
    y = ctx.conv2d_fwd(d, x, w, bias, relu=False, out_dtype=torch.float32)
    assert y.shape == ref.shape
    assert rel_err(y, ref) < 2e-3
    yr = ctx.conv2d_fwd(d, x, w, bias, relu=True)
    assert rel_err(yr, torch.relu(ref)) < 1e-2


@pytest.mark.parametrize("force", ["6", "1006", "1011", "1001"])
def test_dense_interleaved_splits(ctx, monkeypatch, force):
    """split-K with interleaved k-blocks (Params::kb_interleave) against contiguous ranges and fp32"""
    M, N, K = 32, 4070, 4096
    x = bf16_rand(M, K, seed=45)
    w = bf16_rand(N, K, seed=46, scale=1.0 / math.sqrt(K))
    dyp = torch.zeros(M, 4096, dtype=torch.bfloat16, device=DEV)
    dyp[:, :N] = bf16_rand(M, N, seed=47)
    monkeypatch.setenv("A3D_DENSE_FORCE", force)
    y = ctx.dense_fwd(x, w, None, flags=0, out_dtype=torch.float32, impl=L.IMPL_TC)
    dx = ctx.dense_dgrad(dyp, w, impl=L.IMPL_TC)
    monkeypatch.delenv("A3D_DENSE_FORCE")
    assert rel_err(y, x.float() @ w.float().t()) < 2e-3
    assert rel_err(dx, dyp[:, :N].float() @ w.float()) < 1e-2


def test_dense_bwd_unaligned_falls_back(ctx):
    M, N, K = 6, 130, 200
    x, w, dy = bf16_rand(M, K, seed=34), bf16_rand(N, K, seed=35, scale=0.1), bf16_rand(M, N, seed=36)
    assert rel_err(ctx.dense_dgrad(dy, w), dy.float() @ w.float()) < 1e-2
    dw, _ = ctx.dense_wgrad(x, dy)
    assert rel_err(dw, dy.float().t() @ x.float()) < 2e-3


# ----------------------------------------------------------------------------- elementwise
@pytest.mark.parametrize("shape,out", [((2, 480, 640, 3), (228, 304)), ((2, 55, 73, 1), (55, 74)),
                                       ((1, 6, 8, 1), (240, 320)), ((1, 48, 64, 3), (48, 64))])
def test_resize_vs_oracle(ctx, shape, out):
    g = torch.Generator().manual_seed(40)
    x = torch.rand(*shape, generator=g)
    ref, mag = ML.resize_ref(x.double().to(DEV), *out)
    assert torch.equal(ref.cpu(), T.resize_bilinear_tf1(x.double(), *out))
    bound = ML.LERP_U * ML.U * mag                               # the float32 lerp (test_gpu_model_launches)
    y = ctx.resize_bilinear_tf1(x.to(DEV), out[0], out[1])
    assert ML.within(y, ref, bound, "float32")[0] is None
    yb = ctx.resize_bilinear_tf1(x.to(DEV), out[0], out[1], dstC=shape[3] + 1, dtype=torch.bfloat16)
    assert ML.rounded(yb[..., :shape[3]], ref, bound, "bf16")[0] is None            # round to nearest even
    assert float(yb[..., shape[3]:].abs().max()) == 0.0


@pytest.mark.parametrize("N,H,W,C", [(2, 55, 74, 96), (2, 27, 37, 256), (1, 110, 148, 64), (1, 4, 4, 8)])
def test_maxpool_fwd_bwd(ctx, N, H, W, C):
    x = torch.relu(bf16_rand(N, H, W, C, seed=41))
    y = ctx.maxpool2x2_fwd(x)
    xr = x.float().permute(0, 3, 1, 2).requires_grad_(True)
    yr = F.max_pool2d(xr, 2, 2)
    assert torch.equal(y.float(), yr.permute(0, 2, 3, 1))
    dy = bf16_rand(N, H // 2, W // 2, C, seed=42)
    # reference: MaxPoolGrad to the first arg-max, then ReluGrad (x > 0). Ties only occur at x == 0.
    (gx,) = torch.autograd.grad(yr, xr, dy.float().permute(0, 3, 1, 2))
    gx = gx.permute(0, 2, 3, 1) * (x.float() > 0)
    dx = ctx.maxpool2x2_relu_bwd(x, dy)
    assert torch.equal(dx.float(), gx)
    # concat-buffer stride
    yw = torch.zeros(N, H // 2, W // 2, C + 8, dtype=torch.bfloat16, device=DEV)
    ctx.maxpool2x2_fwd(x, out=yw, ldy=C + 8)
    assert torch.equal(yw[..., :C], y) and float(yw[..., C:].abs().max()) == 0.0


def test_relu_bwd_and_dense_epilogue_bwd(ctx):
    y = torch.relu(bf16_rand(70, 64, seed=43))
    dy = bf16_rand(70, 64, seed=44)
    assert torch.equal(ctx.relu_bwd(y, dy).float(), dy.float() * (y.float() > 0))
    mask = (torch.rand(70, 64) < 0.5).to(torch.uint8).to(DEV)
    g = ctx.dense_epilogue_bwd(dy, y, mask, 0.5, L.EPI_RELU)
    ref = (dy.float() * 2.0 * mask.float() * (y.float() > 0)).to(torch.bfloat16)
    assert torch.equal(g, ref)


@pytest.mark.parametrize("M,N,K,drop", [(32, 4070, 4096, True), (32, 4096, 12288, False), (7, 128, 512, True)])
def test_dense_dgrad_act_equals_two_passes(ctx, M, N, K, drop):
    """a3d_dense_dgrad_act (dgrad + DropoutGrad + ReluGrad in the finishing pass) == a3d_dense_dgrad followed by
    a3d_dense_epilogue_bwd, bit for bit (src/models.py:228-232 backwards)."""
    ld = (N + 7) // 8 * 8
    dy = bf16_rand(M, ld, seed=60)
    w = bf16_rand(N, K, seed=61, scale=0.05)
    y = torch.relu(bf16_rand(M, K, seed=62).float()).to(torch.bfloat16)
    mask = (torch.rand(M, K, generator=torch.Generator().manual_seed(63)) < 0.5).to(torch.uint8).to(DEV) if drop else None
    rate = 0.5 if drop else 0.0
    a = ctx.dense_dgrad(dy, w)
    a = ctx.dense_epilogue_bwd(a, y, mask, rate, L.EPI_RELU)
    b = ctx.dense_dgrad_act(dy, w, y, mask, rate, L.EPI_RELU)
    # the split-K partial sums are accumulated with f32 atomics: two runs of the SAME GEMM differ in the last bit now and
    # then, so compare as the other dense tests do
    assert rel_err(b, a.float()) < 2e-2
    ref = (dy[:, :N].float() @ w.float()) * (y.float() > 0)
    if drop:
        ref = ref * mask.float() * 2.0
    assert rel_err(b, ref) < 2e-2
    assert bool(((b.float() == 0) | (y.float() > 0)).all())            # exact zeros wherever the unit was off


@pytest.mark.parametrize("quantised", [False, True])
def test_silog_loss_vs_oracle(ctx, quantised):
    g = torch.Generator().manual_seed(45)
    B, n = 8, 4070
    out = torch.rand(B, n, generator=g) * 1.4 - 0.4           # ~30 % negative -> NaN branch
    tar = torch.rand(B, n, generator=g) * 0.95 + 0.05
    if quantised:                                              # depth PNGs are k/255 incl. zeros
        tar = torch.round(torch.rand(B, n, generator=g) * 255) / 255
    o64 = out.double().requires_grad_(True)
    ref = OM.silog_loss(o64, tar.double())
    (gref,) = torch.autograd.grad(ref, o64)
    # the per-element bounds of the float32 arithmetic on the float32 arguments fl(o + eps) (silog_reference); the
    # oracle (float64 arguments) agrees with that reference far inside them
    lon = float(torch.tensor(0.5 / 4070, dtype=torch.float32))
    r = ML.silog_reference(out.to(DEV), tar.to(DEV), lon)
    assert abs(float(r["loss"][0]) - float(ref.detach())) < 1e-7 * abs(float(ref.detach()))
    assert float((r["grad"][0].cpu() - gref).abs().max()) < 1e-7 * float(gref.abs().max())
    loss, lps, dout, _ = ctx.silog_loss(out.to(DEV), tar.to(DEV))
    for got, key in ((loss, "loss"), (lps, "loss_ps"), (dout, "grad")):
        assert ML.within(got, *r[key], key)[0] is None
    assert bool((dout[out.to(DEV) < 0] == 0).all())                # the NaN branch: exactly 0
    _, _, _, db = ctx.silog_loss(out.to(DEV), tar.to(DEV), grad_bf16=True)
    assert ML.rounded(db, *r["grad"], "bf16 grad")[0] is None


@pytest.mark.parametrize("beta2", [1.0, 0.999])
def test_adam_vs_oracle(ctx, beta2):
    g = torch.Generator().manual_seed(46)
    n = 100003                                                 # odd: exercises the scalar tail
    w = torch.randn(n, generator=g)
    gr = torch.randn(n, generator=g) * 1e-2
    m = torch.randn(n, generator=g) * 1e-3
    v = torch.rand(n, generator=g) * 1e-4
    wr, mr, vr = T.tf_adam_update(w.double(), gr.double() * 0.5, m.double(), v.double(), 3, 0.1, 0.9, beta2, 1e-8)
    wd, gd, md, vd = (t.to(DEV).clone() for t in (w, gr, m, v))
    wb = torch.empty(n, dtype=torch.bfloat16, device=DEV)
    ctx.adam_tf(wd, gd, md, vd, wb, 0.1, 0.9, beta2, 1e-8, 3, grad_scale=0.5)
    assert float((wd.cpu().double() - wr).abs().max()) < 1e-5
    assert float((md.cpu().double() - mr).abs().max()) < 1e-7
    assert float((vd.cpu().double() - vr).abs().max()) < 1e-9
    assert torch.equal(wb, wd.to(torch.bfloat16))
    if beta2 == 1.0:                                           # the reference's configuration: weights frozen
        assert torch.equal(wd.cpu(), w)
    w2 = w.to(DEV).clone()
    ctx.sgd(w2, gd, None, 0.1)
    assert float((w2.cpu() - (w - 0.1 * gr)).abs().max()) < 1e-6


def test_cast_and_scatter(ctx):
    x = torch.randn(12345, device=DEV)
    assert torch.equal(ctx.cast_f32_bf16(x), x.to(torch.bfloat16))
    buf = torch.zeros(10, 7, 64, dtype=torch.bfloat16, device=DEV)
    src = torch.randn(70, device=DEV)
    ctx.scatter_channel_bf16(src, buf, 63)
    assert torch.equal(buf[..., 63].reshape(-1), src.to(torch.bfloat16)) and float(buf[..., :63].abs().max()) == 0


# ----------------------------------------------------------------------------- DCNF pieces
def test_crf_vs_oracle(ctx):
    g = torch.Generator().manual_seed(47)
    B, n = 16, 48
    z = torch.rand(B, n, 1, generator=g, dtype=torch.float64)
    y = torch.rand(B, n, 1, generator=g, dtype=torch.float64)
    r = torch.rand(B, 48, 1, generator=g, dtype=torch.float64)
    pl, pr = OD.pair_indices()
    zl = z.clone().requires_grad_(True)
    rl = r.clone().requires_grad_(True)
    A = OD.build_A(rl)
    nll = torch.stack([OD.nll_stable(A[i:i + 1], y[i:i + 1], zl[i:i + 1]) for i in range(B)])
    gz, gr = torch.autograd.grad(nll.sum(), (zl, rl))
    ystar = OD.crf_map(A.detach(), z)
    res = ctx.crf(z.float().reshape(B, n).to(DEV), y.float().reshape(B, n).to(DEV), r.float().reshape(B, 48).to(DEV),
                  torch.tensor(pl, dtype=torch.int32, device=DEV), torch.tensor(pr, dtype=torch.int32, device=DEV),
                  want_dr=True)
    assert int(res["status"].abs().max()) == 0
    assert float((res["ystar"].cpu().double() - ystar.reshape(B, n)).abs().max()) < 1e-5      # north-star: 1e-5
    # per-element bounds of the float32 arithmetic (crf_reference) on the float32 inputs
    ref = ML.crf_reference(z.float().reshape(B, n), y.float().reshape(B, n), r.float().reshape(B, 48), pl, pr, 1.0, False)
    for key in ("ystar", "nll", "logdet", "dz", "dr"):
        assert ML.within(res[key].cpu(), *ref[key], key)[0] is None
    assert ML.crf_solution_checks({}, res["ystar"], ref) is None
    # the float32 inputs are within 1e-7 of the float64 ones: the oracle on those agrees far inside 1e-4
    assert float((ref["nll"][0] - nll.detach()).abs().max()) < 1e-4
    assert float((ref["dz"][0] - gz.reshape(B, n)).abs().max()) < 1e-4
    assert float((ref["dr"][0] - gr.reshape(B, 48)).abs().max()) < 1e-4
    # not SPD -> status, zeros instead of NaNs
    rbad = -torch.ones(2, 48)
    res = ctx.crf(z.float().reshape(B, n)[:2].to(DEV), y.float().reshape(B, n)[:2].to(DEV), rbad.to(DEV),
                  torch.tensor(pl, dtype=torch.int32, device=DEV), torch.tensor(pr, dtype=torch.int32, device=DEV))
    assert int(res["status"].min()) > 0 and bool(torch.isfinite(res["ystar"]).all())


def test_pairwise_features_tile_means_patches(ctx):
    """similarities on tile-wise constant colours with a few pixels moved between histogram bins (exact features,
    test_gpu_model_launches.pairwise_image), spanning (0.05, 0.95) in both features; tile means of dyadic depths, exact"""
    g = torch.Generator().manual_seed(48)
    im = ML.pairwise_image(2, 240, 320, g)
    pl, pr = OD.pair_indices()
    ref = OD.pairwise_features(im.double())
    ML.assert_similarities_span(ref)
    sims = ctx.pairwise_features(im.to(DEV), torch.tensor(pl, dtype=torch.int32, device=DEV),
                                 torch.tensor(pr, dtype=torch.int32, device=DEV))
    ref64, bound = ML.pairwise_reference(im, pl, pr)
    assert torch.equal(ref64, ref)
    assert ML.within(sims.cpu(), ref, bound, "similarities")[0] is None
    dp = torch.randint(0, 4096, (2, 240, 320, 1), generator=g).double() / 4096       # the 1600-term sums are exact
    q = OD.tile_means(dp).reshape(2, 48)
    ML.assert_no_f32_tie(q)
    ym = ctx.tile_means(dp.float().to(DEV))
    assert torch.equal(ym.cpu(), q.float())
    im = torch.rand(2, 240, 320, 3, generator=g)
    pt = ctx.extract_patches(im.to(DEV), dstC=16)
    refp = OD.patches(im).reshape(96, 100, 100, 3).to(torch.bfloat16)
    assert torch.equal(pt[..., :3].cpu(), refp) and float(pt[..., 3:].abs().max()) == 0


@pytest.mark.parametrize("N,H,W,C", [(2, 55, 74, 96), (1, 27, 37, 256), (1, 110, 148, 64)])
def test_maxpool_f32_routing(ctx, N, H, W, C):
    g = torch.Generator().manual_seed(50)
    x = torch.relu(torch.randn(N, H, W, C, generator=g)).to(DEV)
    idx = torch.empty(N, H // 2, W // 2, C, dtype=torch.uint8, device=DEV)
    y = ctx.maxpool2x2_fwd_f32(x, idx=idx)
    xr = x.permute(0, 3, 1, 2).clone().requires_grad_(True)
    yr = F.max_pool2d(xr, 2, 2)
    assert torch.equal(y, yr.permute(0, 2, 3, 1).to(torch.bfloat16))
    dy = bf16_rand(N, H // 2, W // 2, C, seed=51)
    (gx,) = torch.autograd.grad(yr, xr, dy.float().permute(0, 3, 1, 2))
    gx = gx.permute(0, 2, 3, 1) * (x > 0)
    dx = ctx.maxpool2x2_idx_bwd(idx, dy, (N, H, W, C))
    assert torch.equal(dx.float(), gx)


# ----------------------------------------------------------------------------- pool-fused conv, s2d resize, index maps
@pytest.mark.parametrize("impl", ["tc", "simt"])
def test_conv_pool4_fwd_bwd(ctx, impl):
    """conv + bias + ReLU + 2x2 max-pool as one GEMM (a3d_conv2d_pool4_fwd) and its MaxPoolGrad/ReluGrad."""
    N, H, W, Cc = 2, 57, 76, 64
    d = ops.conv_desc(N, H, W, Cc, 256, 3, 3, 1, "valid", ldy=64, impl=L.IMPL_SIMT if impl == "simt" else L.IMPL_AUTO)
    x = bf16_rand(N, H, W, Cc, seed=40)
    w = bf16_rand(256, 3, 3, Cc, seed=41, scale=1.0 / math.sqrt(9 * Cc))
    bias = (torch.rand(64, generator=torch.Generator().manual_seed(42)) - 0.5).to(DEV) * 0.2
    y = torch.full((N, d.P, d.Q, 64), 7.0, dtype=torch.bfloat16, device=DEV)
    idx = torch.full((N, d.P, d.Q, 64), 9, dtype=torch.uint8, device=DEV)
    ctx.conv2d_pool4_fwd(d, x, w, bias, relu=True, out=y, idx=idx)
    acc = torch_conv_ref(x, w, None, 1, 0, 0, d.P, d.Q, False).view(N, d.P, d.Q, 4, 64)
    m, gi = acc.max(3)
    ref = torch.relu(m + bias)
    assert rel_err(y, ref) < 1e-2
    # routing: identical wherever the winner is clear (f32 accumulation order differs in the last bits)
    top2 = acc.topk(2, dim=3).values                # [N,P,Q,2,64]
    clear = (top2[:, :, :, 0] - top2[:, :, :, 1]) > 1e-3
    assert bool((idx.long()[clear] == gi[clear]).all()) and int(idx.max()) <= 3
    # backward: dy routed to the arg-max group where the pooled output is positive
    dy = bf16_rand(N, d.P, d.Q, 64, seed=43)
    big = ctx.pool4_bwd(dy.view(-1, 64), y.view(-1, 64), idx)
    exp = torch.zeros(N * d.P * d.Q, 4, 64, device=DEV)
    exp.scatter_(1, idx.view(-1, 1, 64).long(), (dy.float() * (y.float() > 0)).view(-1, 1, 64))
    assert torch.equal(big.float().view(-1, 4, 64), exp)


@pytest.mark.parametrize("force", ["6", "7"])
def test_conv_pool4_fwd_cta_pair(ctx, monkeypatch, force):
    """pool-fused fine/first GEMM through the CTA-pair kernel (short / deep ring) == one-CTA kernel, bit for bit"""
    N, H, W, Cc = 3, 57, 76, 64
    d = ops.conv_desc(N, H, W, Cc, 256, 3, 3, 1, "valid", ldy=64, impl=L.IMPL_AUTO)
    x = bf16_rand(N, H, W, Cc, seed=40)
    w = bf16_rand(256, 3, 3, Cc, seed=41, scale=1.0 / math.sqrt(9 * Cc))
    bias = (torch.rand(64, generator=torch.Generator().manual_seed(42)) - 0.5).to(DEV) * 0.2
    res = []
    for f in ("0", force):
        monkeypatch.setenv("A3D_POOL4_FORCE", f)
        y = torch.full((N, d.P, d.Q, 64), 7.0, dtype=torch.bfloat16, device=DEV)
        idx = torch.full((N, d.P, d.Q, 64), 9, dtype=torch.uint8, device=DEV)
        ctx.conv2d_pool4_fwd(d, x, w, bias, relu=True, out=y, idx=idx)
        res.append((y, idx))
    monkeypatch.delenv("A3D_POOL4_FORCE")
    assert torch.equal(res[0][0], res[1][0]) and torch.equal(res[0][1], res[1][1])     # same MMA order: bit-exact


def test_resize_s2d_matches_resize_then_space_to_depth(ctx):
    g = torch.Generator().manual_seed(44)
    src = torch.rand(2, 480, 640, 3, generator=g).to(DEV)
    flat = ctx.resize_bilinear_tf1(src, 228, 304, dstC=3, dtype=torch.bfloat16)
    out = torch.full((2, 57, 76, 64), 5.0, dtype=torch.bfloat16, device=DEV)
    ctx.resize_bilinear_tf1_s2d(src, 228, 304, 4, out=out)
    exp = flat.view(2, 57, 4, 76, 4, 3).permute(0, 1, 3, 2, 4, 5).reshape(2, 57, 76, 48)
    assert torch.equal(out[..., :48], exp)
    assert float(out[..., 48:].abs().max()) == 0.0


def test_resize_s2d_uint8_and_pipelined(ctx, monkeypatch):
    """uint8 images (pixel / 255) through the pipelined resize kernel == float path on the same pixels; batch > grid
    so that persistent blocks walk over several rows; ragged width (W*3 % 16 == 0 only)"""
    g = torch.Generator().manual_seed(46)
    for B, H, W in ((5, 480, 640), (1, 50, 64)):
        OH, OW = (228, 304) if H == 480 else (24, 28)
        u8 = torch.randint(0, 256, (B, H, W, 3), generator=g, dtype=torch.uint8).to(DEV)
        f32 = u8.float() / 255.0
        ref = torch.full((B, OH // 4, OW // 4, 64), 5.0, dtype=torch.bfloat16, device=DEV)
        ctx.resize_bilinear_tf1_s2d(f32, OH, OW, 4, out=ref)
        out = torch.full_like(ref, 7.0)
        ctx.resize_bilinear_tf1_s2d(u8, OH, OW, 4, out=out)
        assert float((out.float() - ref.float()).abs().max()) <= 2.0 ** -8      # one bf16 ulp at 1.0 (rounding order)
        assert float(out[..., 48:].abs().max()) == 0.0
        flat = ctx.resize_bilinear_tf1(f32, OH, OW, dstC=3, dtype=torch.bfloat16)
        exp = flat.view(B, OH // 4, 4, OW // 4, 4, 3).permute(0, 1, 3, 2, 4, 5).reshape(B, OH // 4, OW // 4, 48)
        assert torch.equal(ref[..., :48], exp)


def test_gather_sum_and_scatter_cast(ctx):
    g = torch.Generator().manual_seed(45)
    n, G, big = 1000, 4, 5000
    perm = torch.stack([torch.randperm(big, generator=g)[:n] for _ in range(G)]).to(torch.int32)
    perm[1, ::7] = -1
    src = torch.rand(big, generator=g).to(DEV)
    idx = perm.to(DEV)
    dst = torch.empty(n, device=DEV)
    ctx.gather_sum_f32(src, idx, dst)
    exp = torch.zeros(n, device=DEV)
    for k in range(G):
        ok = idx[k] >= 0
        exp[ok] += src[idx[k][ok].long()]
    assert torch.allclose(dst, exp, atol=1e-6)
    w = torch.rand(n, generator=g).to(DEV)
    out = torch.zeros(big, dtype=torch.bfloat16, device=DEV)
    one = idx[:1].contiguous()                       # a single copy: no write conflicts
    ctx.scatter_cast_bf16(w, one, out)
    exp = torch.zeros(big, dtype=torch.bfloat16, device=DEV)
    exp[one[0].long()] = w.bfloat16()
    assert torch.equal(out, exp)


def test_dense_wgrad_adam_fused(ctx):
    """Fused dense wgrad + TF-Adam (mma.sync gradient inside the optimizer pass) against f32 torch math on the same
    bf16 operands."""
    M, N, K = 32, 100, 512
    g = torch.Generator().manual_seed(50)
    x = bf16_rand(M, K, seed=51)
    lddy = (N + 7) // 8 * 8
    dy = bf16_rand(M, lddy, seed=52)
    w0 = torch.rand(N, K, generator=g).to(DEV)
    m0 = (torch.rand(N, K, generator=g) * 0.1).to(DEV)
    v0 = (torch.rand(N, K, generator=g) * 0.01).to(DEV)
    lr, b1, b2, eps, t, gs = 0.1, 0.9, 0.999, 1e-8, 3, 0.5
    grad = dy[:, :N].float().t() @ x.float() * gs
    m1 = b1 * m0 + (1 - b1) * grad
    v1 = b2 * v0 + (1 - b2) * grad * grad
    w1 = w0 - ops.adam_lr_t(lr, b1, b2, t) * m1 / (v1.sqrt() + eps)
    w, m, v = w0.clone(), m0.clone(), v0.clone()
    wb = torch.zeros(N, K, dtype=torch.bfloat16, device=DEV)
    db = torch.zeros(N, device=DEV)
    ctx.dense_wgrad_adam(x, dy, db, w, m, v, wb, lr, b1, b2, eps, t, gs)
    assert torch.allclose(w, w1, rtol=1e-4, atol=1e-5) and torch.allclose(m, m1, rtol=1e-4, atol=1e-6)
    assert torch.allclose(db, dy[:, :N].float().sum(0), rtol=1e-3, atol=1e-3)


def test_bias_grad_bf16_rank_blocks(ctx):
    """a3d_bias_grad_bf16 over a batch stored as rank blocks [x_r | dy_r] (group_rows / group_stride) must give the
    column sums of the plain [M, ld] matrix."""
    n, B, N, K = 4, 16, 96, 256
    lddy = 96
    x = bf16_rand(n * B, K, seed=60)
    dy = bf16_rand(n * B, lddy, seed=61)
    blk = B * (K + lddy)
    gbuf = torch.zeros(n, blk, dtype=torch.bfloat16, device=DEV)
    for r in range(n):
        gbuf[r, :B * K] = x[r * B:(r + 1) * B].reshape(-1)
        gbuf[r, B * K:] = dy[r * B:(r + 1) * B].reshape(-1)
    db = torch.zeros(N, device=DEV)
    ctx.bias_grad_bf16(gbuf.view(-1)[B * K:], N, db, rows=n * B, ld=lddy, group_rows=B, group_stride=blk)
    assert torch.allclose(db, dy[:, :N].float().sum(0), rtol=1e-5, atol=1e-4)


# ---- overlapped-pixel / dilated view (a3d_conv_desc dil_w, pix_pitch): the DCNF first layer ------------------------------
def _view_reference(cells, w, N, Hc, Wc, P, Q, dil):
    """cells f64 flat (with slack), w f64 [K,R,S,64]: out[n,p,q,k] = sum_{r,s} w[k,r,s,:] . cells[(n,p+r,q+s*dil) .. +64)."""
    K, R, S, _ = w.shape
    out = torch.zeros(N, P, Q, K, dtype=torch.float64)
    pix = torch.arange(Hc * Wc * N).view(N, Hc, Wc)
    win = cells.unfold(0, 64, 16)                                   # win[i] = 64 elements starting at cell i
    for r in range(R):
        for s in range(S):
            sel = pix[:, r:r + P, s * dil:s * dil + Q]
            out += win[sel] @ w[:, r, s, :].t()
    return out, win, pix


@pytest.mark.parametrize("fold", [1, 4])
@pytest.mark.parametrize("impl", ["tc", "simt"])
def test_conv_view_pool4_fwd_and_wgrad(ctx, fold, impl):
    """64-channel pixels that are 4 consecutive 16-channel cells (pix_pitch = 16, or materialised for fold = 4), taps 4
    pixels apart (dil_w = 4): pool-fused forward and weight gradient against float64 on the same bf16 values."""
    N, Hc, Wc, R, S, dil = 3, 20, 30, 6, 2, 4
    P, Q = Hc - R + 1, Wc - 6 + 1
    g = torch.Generator().manual_seed(60)
    cells = torch.randn(N * Hc * Wc * 16 + 64, generator=g).to(torch.bfloat16)
    cells[N * Hc * Wc * 16:] = 0
    w = (torch.randn(256, R, S, 64, generator=g) / math.sqrt(R * S * 64)).to(torch.bfloat16)
    bias = (torch.rand(64, generator=g) - 0.5) * 0.2
    ref, win, pix = _view_reference(cells.double(), w.double(), N, Hc, Wc, P, Q, dil)
    if fold == 1:
        x = cells.to(DEV)
        xv = x[:N * Hc * Wc * 16].view(N, Hc, Wc, 16)
    else:
        xv = win[pix].to(torch.bfloat16).to(DEV).contiguous()      # [N,Hc,Wc,64] materialised
        x = xv
    d = ops.conv_desc(N, Hc, Wc, 64, 256, R, S, 1, "valid", ldy=64, impl=L.IMPL_SIMT if impl == "simt" else L.IMPL_AUTO)
    d.P, d.Q, d.dil_w, d.pix_pitch = P, Q, dil, 16 if fold == 1 else 0
    y = torch.full((N, P, Q, 64), 7.0, dtype=torch.bfloat16, device=DEV)
    idx = torch.full((N, P, Q, 64), 9, dtype=torch.uint8, device=DEV)
    ctx.conv2d_pool4_fwd(d, xv, w.to(DEV), bias.to(DEV), relu=True, out=y, idx=idx)
    r4 = ref.view(N, P, Q, 4, 64)
    yref = torch.relu(r4.max(3).values + bias.double())
    assert float((y.cpu().double() - yref).abs().max()) < 2e-2 * float(yref.abs().max())
    # the routing byte names a group whose value is the maximum (ties aside, within accumulation noise)
    picked = r4.gather(3, idx.cpu().long().unsqueeze(3)).squeeze(3)
    assert float((picked - r4.max(3).values).abs().max()) < 1e-3
    # weight gradient over the 4 x 64 columns
    dy = (torch.randn(N, P, Q, 256, generator=g) * 0.1).to(torch.bfloat16)
    dw = torch.empty(256, R, S, 64, dtype=torch.float32, device=DEV)
    db = torch.empty(256, dtype=torch.float32, device=DEV)
    dwd = L.ConvDesc.from_buffer_copy(d)
    dwd.ldy = 256
    ctx.conv2d_wgrad(dwd, xv, dy.to(DEV), dw=dw, db=db)
    dwref = torch.zeros(256, R, S, 64, dtype=torch.float64)
    dyf = dy.double().view(-1, 256)
    for r in range(R):
        for s in range(S):
            sel = pix[:, r:r + P, s * dil:s * dil + Q].reshape(-1)
            dwref[:, r, s, :] = dyf.t() @ win[sel]
    assert float((dw.cpu().double() - dwref).abs().max()) < 1e-3 * float(dwref.abs().max())
    assert float((db.cpu().double() - dyf.sum(0)).abs().max()) < 1e-3 * float(dyf.sum(0).abs().max())
    # every other convolution call rejects the view
    with pytest.raises(L.A3DError):
        ctx.conv2d_fwd(dwd, xv, w.to(DEV), None)


def test_extract_patches_s2d(ctx):
    g = torch.Generator().manual_seed(61)
    im = torch.rand(2, 240, 320, 3, generator=g)
    refp = OD.patches(im).reshape(96, 100, 100, 3).to(torch.bfloat16)
    exp = torch.zeros(96, 50, 50, 16, dtype=torch.bfloat16)
    for a in range(2):
        for b in range(2):
            exp[..., (2 * a + b) * 3:(2 * a + b) * 3 + 3] = refp[:, a::2, b::2, :]
    c1 = torch.full((96, 50, 50, 16), 5.0, dtype=torch.bfloat16, device=DEV)
    ctx.extract_patches_s2d(im.to(DEV), c1, 1)
    assert torch.equal(c1.cpu(), exp)
    c4 = torch.full((96, 50, 50, 64), 5.0, dtype=torch.bfloat16, device=DEV)
    ctx.extract_patches_s2d(im.to(DEV), c4, 4)
    for k in range(4):
        assert torch.equal(c4[:, :, :50 - k, 16 * k:16 * k + 16].cpu(), exp[:, :, k:, :])
        if k:
            assert float(c4[:, :, 50 - k:, 16 * k:16 * k + 16].abs().max()) == 0.0


def test_image_cells_and_window_gather_scatter(ctx):
    g = torch.Generator().manual_seed(62)
    im = torch.rand(2, 240, 320, 3, generator=g)
    cells = torch.full((2, 150, 190, 16), 5.0, dtype=torch.bfloat16, device=DEV)
    ctx.image_cells_s2d(im.to(DEV), 30, cells)
    pad = F.pad(im.permute(0, 3, 1, 2), (30, 30, 30, 30)).permute(0, 2, 3, 1).to(torch.bfloat16)     # [2,300,380,3]
    exp = torch.zeros(2, 150, 190, 16, dtype=torch.bfloat16)
    for a in range(2):
        for b in range(2):
            exp[..., (2 * a + b) * 3:(2 * a + b) * 3 + 3] = pad[:, a::2, b::2, :]
    assert torch.equal(cells.cpu(), exp)
    # the patch-wise cells are windows of it: patch (prow, pcol) = cells[20 prow : +50, 20 pcol : +50]
    pc = torch.empty(96, 50, 50, 16, dtype=torch.bfloat16, device=DEV)
    ctx.extract_patches_s2d(im.to(DEV), pc, 1)
    win = torch.empty(96, 50 * 50 * 16, dtype=torch.bfloat16, device=DEV)
    ctx.window_gather(cells, 6, 8, 50, 20, win)
    assert torch.equal(win.view(96, 50, 50, 16), pc)
    # 7x7 windows at stride 5 and the transpose
    src = bf16_rand(2, 32, 42, 256, seed=63)
    out = torch.empty(96, 7, 7, 256, dtype=torch.bfloat16, device=DEV)
    ctx.window_gather(src, 6, 8, 7, 5, out)
    ref = src.cpu().unfold(1, 7, 5).unfold(2, 7, 5).permute(0, 1, 2, 4, 5, 3).reshape(96, 7, 7, 256)
    assert torch.equal(out.cpu(), ref)
    go = bf16_rand(96, 7, 7, 256, seed=64)
    gs = torch.full((2, 32, 42, 256), 3.0, dtype=torch.bfloat16, device=DEV)
    ctx.window_scatter_sum(go, 6, 8, 7, 5, gs)
    x = src.cpu().double().requires_grad_(True)
    x.unfold(1, 7, 5).unfold(2, 7, 5).permute(0, 1, 2, 4, 5, 3).reshape(96, 7, 7, 256).backward(go.cpu().double())
    assert torch.equal(gs.cpu(), x.grad.to(torch.bfloat16))


def test_dense_bwd_long_batch(ctx):
    """DCNF dense layers: 768 patches.  dgrad with the batch as the GEMM M dimension (a3d_tc_dense_dgrad_rows) and the
    tiny weight gradients (16x128, 1x16) through the sliced CUDA-core kernel, against fp32 on the same bf16 values."""
    M, N, K = 768, 128, 12544
    w = bf16_rand(N, K, seed=70, scale=1.0 / math.sqrt(K))
    dy = bf16_rand(M, N, seed=71)
    n0 = ctx.launches
    dx = ctx.dense_dgrad(dy, w, impl=L.IMPL_TC)
    assert ctx.launches == n0 + 1                                   # one GEMM launch, no memset / finish
    assert rel_err(dx, dy.float() @ w.float()) < 1e-2
    assert rel_err(ctx.dense_dgrad(dy, w, impl=L.IMPL_SIMT), dy.float() @ w.float()) < 1e-2
    for (n, k) in ((16, 128), (1, 16)):
        x = bf16_rand(M, k, seed=72)
        g = bf16_rand(M, n, seed=73)
        db = torch.empty(n, dtype=torch.float32, device=DEV)
        dw, _ = ctx.dense_wgrad(x, g, db=db, N=n, impl=L.IMPL_SIMT)
        assert rel_err(dw, g.float().t() @ x.float()) < 1e-4
        assert rel_err(db, g.float().sum(0)) < 2e-3
