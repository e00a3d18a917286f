"""GPU tests of the FP8 inference mode (E4M3 operands, tcgen05.mma kind::f8f6f4; include/a3d.h "FP8 inference"):
the engine against exact float64 products, every MSDN layer against float64 on its dequantised operands, the quantisers
bit for bit against oracle/fp8.py, the whole forward against oracle/fp8.py, per-image batch invariance, graph replay,
uint8 inputs, weight reloads, the error cases and `evaluate --dtype fp8`."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

from oracle import fp8 as F
from oracle import msdn as OM
from oracle import tf1_ops as T

if torch.cuda.is_available():
    from ann3depth_b200 import models

DEV = "cuda:0"
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def rel_l2(a, b):
    a, b = a.double().cpu(), b.double().cpu()
    return float((a - b).norm() / b.norm())


def params(seed=1):
    p = OM.init_params(seed, torch.float32, bias_range=0.05)
    p["coarse/dense/dense_1/bias"] += 1.0
    p["fine/third/bias"] += 1.0
    return p


def inputs(B, seed=0):
    g = torch.Generator().manual_seed(seed)
    return torch.rand(B, 480, 640, 3, generator=g), torch.rand(B, 55, 73, 1, generator=g) * 0.95 + 0.05


def fp8_net(images, depths, p, dtype="fp8"):
    op = models.msdn(images.to(DEV).contiguous(), depths.to(DEV).contiguous(), train=False, dtype=dtype)
    op.net.load_params(p)
    return op


@pytest.mark.parametrize("M,N,K,bn,kcb,splits", [(200, 96, 512, 96, 128, 1), (130, 40, 256, 64, 64, 1),
                                                 (256, 256, 1024, 256, 128, 3), (129, 200, 384, 192, 128, 1),
                                                 (77, 20, 128, 32, 64, 2)])
def test_engine_matches_exact_products(M, N, K, bn, kcb, splits):
    ctx = models.get_context(0)
    g = torch.Generator().manual_seed(M + N + K)
    A = F.e4m3(torch.randn(M, K, generator=g) * 16).to(DEV)
    B = F.e4m3(torch.randn(N, K, generator=g) * 16).to(DEV)
    ref = A.double() @ B.double().t()
    D = ctx.debug_tc_gemm_fp8(A, B, M, N, K, bn, kcb, splits)
    torch.cuda.synchronize()
    assert float((D.double() - ref).abs().max() / ref.abs().max()) <= 1e-6
    rs = torch.rand(ceil(M, 64), generator=g).to(DEV)
    cs = torch.rand(N, generator=g).to(DEV)
    D = ctx.debug_tc_gemm_fp8(A, B, M, N, K, bn, kcb, splits, rs=rs, rs_div=64, cs=cs)
    refs = ref * rs.double().repeat_interleave(64)[:M, None] * cs.double()[None, :]
    assert float((D.double() - refs).abs().max() / refs.abs().max()) <= 1e-6


def ceil(a, b):
    return (a + b - 1) // b


def test_quantizers_bit_identical():
    ctx = models.get_context(0)
    g = torch.Generator().manual_seed(5)
    w = (torch.randn(300, 3, 3, 64, generator=g) * torch.rand(300, 1, 1, 1, generator=g)).to(torch.bfloat16)
    w[7] = 0
    q, s = ctx.quantize_rows_e4m3(w.to(DEV))
    qr, sr = F.quantize_rows(w.float())
    assert torch.equal(s.cpu(), sr) and torch.equal(q.cpu().view(torch.uint8), qr.view(torch.uint8))
    x = torch.relu(torch.randn(3, 13, 18, 384, generator=g) * torch.tensor([1e-3, 1.0, 300.0]).view(3, 1, 1, 1))
    x = x.to(torch.bfloat16)
    q, s = ctx.quantize_e4m3(x.to(DEV))
    qr, sr = F.quantize_images(x.float())
    assert torch.equal(s.cpu(), sr) and torch.equal(q.cpu().view(torch.uint8), qr.view(torch.uint8))
    x = torch.relu(torch.randn(2, 55, 74, 96, generator=g)).to(torch.bfloat16)
    q, s = ctx.maxpool2x2_quantize_e4m3(x.to(DEV), ldy=128)
    pooled = torch.cat([T.max_pool_2x2(x.float()), torch.zeros(2, 27, 37, 32)], dim=-1)
    qr, sr = F.quantize_images(pooled)
    assert torch.equal(s.cpu(), sr) and torch.equal(q.cpu().view(torch.uint8), qr.view(torch.uint8))


def _s2d(x):
    """[B,228,304,3] -> [B,57,76,48] in the (dy, dx, c) channel order of the space-to-depth image"""
    B = x.shape[0]
    return x.reshape(B, 57, 4, 76, 4, 3).permute(0, 1, 3, 2, 4, 5).reshape(B, 57, 76, 48)


def test_resize_into_e4m3():
    ctx = models.get_context(0)
    images, _ = inputs(2, seed=7)
    got = ctx.resize_bilinear_tf1_s2d_e4m3(images.to(DEV), 228, 304).cpu()
    v = _s2d(T.resize_bilinear_tf1(images.double(), 228, 304)) * 256
    ref = F.e4m3(v.float())
    near = F.e4m3((v * (1 + 1e-6)).float()).view(torch.uint8) != F.e4m3((v * (1 - 1e-6)).float()).view(torch.uint8)
    bad = (got[..., :48].view(torch.uint8) != ref.view(torch.uint8)) & ~near
    assert int(bad.sum()) == 0 and int(near.sum()) < 100
    assert int(got[..., 48:].view(torch.uint8).count_nonzero()) == 0
    u8 = (torch.rand(2, 480, 640, 3, generator=torch.Generator().manual_seed(8)) * 255).round().to(torch.uint8)
    a = ctx.resize_bilinear_tf1_s2d_e4m3(u8.to(DEV), 228, 304)
    b = ctx.resize_bilinear_tf1_s2d_e4m3((u8.float() / 255).to(DEV), 228, 304)
    assert torch.equal(a.view(torch.uint8), b.view(torch.uint8))


def _deq(q, s):
    return q.double() * s.double().reshape((-1,) + (1,) * (q.dim() - 1))


def _excess(got, ref):
    """worst excess over one bf16 rounding of the output (2^-8 of each value) plus the float32 accumulation of up to
    3456 exact products (1e-4 of the output's scale); <= 0 passes"""
    got, ref = got.double(), ref.double()
    tol = ref.abs() * 2.0 ** -8 + ref.abs().max() * 1e-4
    return float(((got - ref).abs() - tol).max() / ref.abs().max())


def _close_bf16(got, ref):
    e = _excess(got, ref)
    assert e <= 0, e


def test_layers_against_dequantised_operands():
    images, depths = inputs(2, seed=1)
    op = fp8_net(images, depths, params())
    net = op.net
    net.forward()
    torch.cuda.synchronize()
    wq = {k: _deq(*v) for k, v in net.wq.items()}
    n = "coarse/conv/conv2d_"

    def conv(x, name, stride, pad, relu=True):
        return T.conv2d(x, wq[name].permute(1, 2, 3, 0), net.bias(name).double(), stride, pad, relu)
    img = _deq(net.img4q, net.s_img)
    d = "coarse/dense/dense_"
    big = T.conv2d(img, wq["fine/first/conv2d"].permute(1, 2, 3, 0), None, 1, "valid", False)
    b1 = net.bias("fine/first/conv2d").double()
    b1 = torch.cat([b1, b1.new_zeros(64 - b1.numel())])[:64]
    pooled = torch.relu(big.reshape(2, 55, 74, 4, 64).amax(3) + b1)
    excess = {
        "conv2d_0": _excess(net.c0, conv(img, n + "0", 1, "valid")),
        "conv2d_1": _excess(net.c1, conv(_deq(net.p0q, net.s_p0), n + "1", 1, "same")),
        "conv2d_2": _excess(net.c2, conv(_deq(net.p1q, net.s_p1), n + "2", 1, "same")),
        "conv2d_3": _excess(net.c3, conv(_deq(net.c2q, net.s_c2), n + "3", 1, "same")),
        "conv2d_4": _excess(net.c4, conv(_deq(net.c3q, net.s_c3), n + "4", 2, "valid")),
        "dense_0": _excess(net.d0, torch.relu(_deq(net.c4q, net.s_c4) @ wq[d + "0"].t() + net.bias(d + "0").double())),
        "fine/first": _excess(net.cat[..., :63], pooled[..., :63]),
        "fine/second": _excess(net.f2, conv(_deq(net.catq, net.s_cat), "fine/second/conv2d", 1, "same")),
    }
    print("fp8 layer excess over the bf16 tolerance:", excess)
    assert all(e <= 0 for e in excess.values()), excess
    ref = _deq(net.d0q, net.s_d0) @ wq[d + "1"].t() + net.bias(d + "1").double()
    assert rel_l2(net.coarse, ref) < 1e-5
    # the storage points: pool + quantise and quantise of the bf16 outputs, bit for bit
    for src, q, s in ((torch.cat([T.max_pool_2x2(net.c0.float()), torch.zeros(2, 27, 37, 32, device=DEV)], -1), net.p0q,
                       net.s_p0), (T.max_pool_2x2(net.c1.float()), net.p1q, net.s_p1), (net.c2, net.c2q, net.s_c2),
                      (net.d0, net.d0q, net.s_d0), (net.cat, net.catq, net.s_cat)):
        qr, sr = F.quantize_images(src.float())
        assert torch.equal(s, sr) and torch.equal(q.view(torch.uint8), qr.view(torch.uint8))
    # split-K of the convolution (scaled partial sums, bias in the finishing pass) against the unsplit tile
    ctx = net.ctx
    os.environ["A3D_FP8_CONV_FORCE"] = "128,1,0"
    try:
        one = ctx.conv2d_fwd_fp8(net.d_c2, net.p1q, net.s_p1, *net.wq[n + "2"], net.bias(n + "2"), relu=True).clone()
        os.environ["A3D_FP8_CONV_FORCE"] = "128,4,0"
        four = ctx.conv2d_fwd_fp8(net.d_c2, net.p1q, net.s_p1, *net.wq[n + "2"], net.bias(n + "2"), relu=True)
    finally:
        del os.environ["A3D_FP8_CONV_FORCE"]
    _close_bf16(four, one.double())
    _close_bf16(one, conv(_deq(net.p1q, net.s_p1), n + "2", 1, "same"))


# relative L2 of these FP8 maps against the unrounded float64 forward and against the bf16 net, measured on a B200 at
# B = 2 and 32 (DESIGN.md 4.5); the asserted bounds are twice these
ERR_F64 = {"coarse": 0.0031, "fine": 0.0083}
ERR_BF16 = {"coarse": 0.0031, "fine": 0.0084}


@pytest.mark.parametrize("B", [2, 32])
def test_forward_matches_oracle(B):
    images, depths = inputs(B, seed=B)
    p = params()
    op = fp8_net(images, depths, p)
    op.net.forward()
    ref = F.forward({k: v.to(DEV) for k, v in p.items()}, images.to(DEV), depths.to(DEV))
    p64 = {k: v.double().to(DEV) for k, v in p.items()}
    im = OM.preprocess(images.double(), depths.double())[0].to(DEV)      # the oracle resize builds CPU index tensors
    f64 = {"coarse": OM.coarse(p64, im, None, False)}
    f64["fine"] = OM.fine(p64, im, f64["coarse"])
    bf = fp8_net(images, depths, p, dtype="bf16")
    bf.net.forward()
    torch.cuda.synchronize()
    got = {"coarse": op.coarse, "fine": op.outputs}
    errs = {}
    for k in ("coarse", "fine"):
        errs[k] = (rel_l2(got[k], ref[k]), rel_l2(got[k], f64[k]), rel_l2(got[k], {"coarse": bf.coarse, "fine": bf.outputs}[k]))
    print(f"fp8 B={B} rel L2 (oracle fp8, float64, bf16 net): {errs}")
    for k, (e_or, e64, ebf) in errs.items():
        assert e_or < 1e-2, (k, e_or)
        assert e64 < 2 * ERR_F64[k] and ebf < 2 * ERR_BF16[k], (k, e64, ebf)
    for name, s in ref["scales"].items():
        got_s = getattr(op.net, "s_" + name)
        assert float(((got_s - s.reshape(-1)).abs() / s.reshape(-1)).max()) < 2.0 ** -6, name


def test_batch_invariance():
    images, depths = inputs(32, seed=11)
    p = params()
    big = fp8_net(images, depths, p)
    big.net.forward()
    one = fp8_net(images[:1], depths[:1], p)
    one.net.forward()
    torch.cuda.synchronize()
    for name in ("img", "p0", "p1", "c2", "c3", "c4", "d0", "cat"):
        a, b = getattr(one.net, "s_" + name)[0], getattr(big.net, "s_" + name)[0]
        # equal up to the order of the split-K float32 sums the tuner chose for each batch size
        assert abs(float(a) - float(b)) <= float(b) * 2.0 ** -7, (name, float(a), float(b))
    assert rel_l2(one.outputs[0], big.outputs[0]) < 1e-2 and rel_l2(one.coarse[0], big.coarse[0]) < 1e-2


def test_graph_replay_uint8_and_reload():
    images, depths = inputs(4, seed=3)
    p = params()
    op = fp8_net(images, depths, p)
    net = op.net
    net.forward()                                       # warm-up: autotuning and workspaces outside the capture
    torch.cuda.synchronize()
    s_first = net.s_c2.clone()
    gr = torch.cuda.CUDAGraph()
    with torch.cuda.graph(gr):
        net.forward()
    images2, depths2 = inputs(4, seed=4)
    net.images.copy_(images2.to(DEV))
    net.depths.copy_(depths2.to(DEV))
    gr.replay()
    torch.cuda.synchronize()
    replayed = (op.outputs.clone(), op.coarse.clone(), net.s_c2.clone())
    net.forward()
    torch.cuda.synchronize()
    assert rel_l2(replayed[0], op.outputs) < 1e-3 and rel_l2(replayed[1], op.coarse) < 1e-3
    assert not torch.equal(replayed[2], s_first)
    assert float(((replayed[2] - net.s_c2).abs() / net.s_c2).max()) <= 2.0 ** -7
    # uint8 images are float32 images of k / 255
    u8 = (images2 * 255).round().to(torch.uint8)
    a = models.msdn(u8.to(DEV).contiguous(), depths2.to(DEV).contiguous(), train=False, dtype="fp8")
    a.net.load_params(p)
    a.net.forward()
    b = fp8_net(u8.float() / 255, depths2, p)
    b.net.forward()
    torch.cuda.synchronize()
    assert torch.equal(a.net.img4q.view(torch.uint8), b.net.img4q.view(torch.uint8))
    assert rel_l2(a.outputs, b.outputs) < 1e-3
    # a second load_params: the E4M3 weights follow
    p2 = params(seed=9)
    net.load_params(p2)
    gr.replay()
    torch.cuda.synchronize()
    fresh = fp8_net(images2, depths2, p2)
    fresh.net.forward()
    torch.cuda.synchronize()
    assert rel_l2(op.outputs, fresh.outputs) < 1e-3 and rel_l2(op.coarse, fresh.coarse) < 1e-3


def test_fp8_is_inference_only():
    from ann3depth_b200.augment import Augment
    im, dp = (t.to(DEV).contiguous() for t in inputs(1))
    with pytest.raises(ValueError, match="inference"):
        models.msdn(im, dp, train=True, dtype="fp8")
    with pytest.raises(ValueError, match="augment"):
        models.msdn(im, dp, train=False, dtype="fp8", augment=Augment())


def test_evaluate_fp8_end_to_end(tmp_path):
    from test_gpu_eval import N_TEST, _assert_close, _run, _test_split
    from oracle import metrics as OMet
    from ann3depth_b200 import data
    from ann3depth_b200.ann3depth import restore_checkpoint
    from ann3depth_b200.evaluate import model_outputs
    _test_split(str(tmp_path))
    ck = tmp_path / "ckpt"
    _run("ann3depth_b200.ann3depth", "nyu", "--model", "msdn", "--steps", "2", "--batchsize", "2", "--ckptdir", str(ck),
         "--datadir", str(tmp_path), "--sumfreq", "1")
    out = tmp_path / "fp8.json"
    _run("ann3depth_b200.evaluate", "nyu", "--model", "msdn", "--ckptdir", str(ck), "--batchsize", "2", "--datadir",
         str(tmp_path), "--dtype", "fp8", "--json", str(out))
    res = json.loads(out.read_text())
    assert res["dtype"] == "fp8" and res["images"] == N_TEST and res["global_step"] == 2
    # the metrics of the FP8 net's own maps through the float64 metric oracle, as tests/test_gpu_eval.py does for bf16
    inp = data.inputs(str(tmp_path), "nyu", 2, "test", epochs=1)
    op = models.msdn(inp.images, inp.depths, train=False, dtype="fp8")
    assert restore_checkpoint(op, str(ck / "msdn"))
    per = {}
    while True:
        n = inp.next_batch()
        if not n:
            break
        op.net.infer()
        for name, t in model_outputs(op).items():
            up = op.net.ctx.resize_bilinear_tf1(t, 480, 640).cpu().numpy()[..., 0]
            gt = inp.depths.cpu().numpy()[..., 0]
            per.setdefault(name, []).extend(OMet.image_sums(up[b], gt[b])[0] for b in range(n))
    inp.close()
    for name, v in per.items():
        _assert_close(res["metrics"][name], OMet.dataset_metrics(np.stack(v)))
    r = subprocess.run([sys.executable, "-m", "ann3depth_b200.evaluate", "nyu", "--model", "dcnf", "--ckptdir", str(ck),
                        "--datadir", str(tmp_path), "--dtype", "fp8"], cwd=ROOT, capture_output=True, text=True,
                       timeout=300)
    assert r.returncode != 0 and "no FP8 mode" in r.stderr
