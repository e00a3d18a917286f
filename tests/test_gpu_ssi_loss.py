"""The scale-and-shift-invariant loss on the GPU: `a3d_ssi_loss` against the storage-point oracle
(oracle/ssi_loss.py `ssi_loss_points`), and `models.msdn(..., loss="ssi")` end to end against the float64 MSDN oracle,
in every precision mode, in the four-stream step and in the train driver."""
import json
import os
import subprocess
import sys
import tempfile

import pytest
import torch

pytestmark = pytest.mark.gpu

from oracle import msdn as OM
from oracle import ssi_loss as S

if torch.cuda.is_available():
    from ann3depth_b200 import _lib as L
    from ann3depth_b200 import models

DEV = "cuda:0"
H, W, N = 55, 74, 55 * 74
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def ctx():
    return models.get_context(0)


def loss_batch(B, seed):
    """k/255 targets with zeros; random predictions, with image b % 5 == 1 of negative slope, == 2 an exact affine fit of
    the target, == 3 constant.  Returns p, t (float32 [B, N]) and the exact-fit rows."""
    g = torch.Generator().manual_seed(seed)
    t = torch.round(torch.rand(B, N, generator=g) * 255) / 255
    t[:, ::17] = 0.0
    p = torch.randn(B, N, generator=g) * 0.3 + 1.0
    exact = []
    for b in range(B):
        if b % 5 == 1:
            p[b] = -0.8 * t[b] + 0.1 * torch.randn(N, generator=g) + 2.0
        elif b % 5 == 2:
            p[b] = 3.0 * t[b] + 1.0
            exact.append(b)
        elif b % 5 == 3:
            p[b] = 0.25
    return p.float(), t.float(), exact


def bits(x):
    return x.view(torch.int32) if x.dtype == torch.float32 else x.view(torch.int16)


@pytest.mark.parametrize("alpha,scales", [(0.0, 1), (0.0, 4), (0.5, 1), (0.5, 4)])
@pytest.mark.parametrize("ld", [4070, 4096])
@pytest.mark.parametrize("B", [1, 5, 32, 130])
def test_kernel_vs_storage_point_oracle(ctx, B, ld, alpha, scales):
    p, t, exact = loss_batch(B, seed=B)
    Lref, Gref = S.ssi_loss_points(p.numpy(), t.numpy(), H, W, alpha, scales)
    Gref = torch.from_numpy(Gref / B)
    pd, td = p.to(DEV), t.to(DEV)
    sentinel = 7.0
    d32 = torch.full((B, ld), sentinel, device=DEV)
    d16 = torch.full((B, ld), sentinel, dtype=torch.bfloat16, device=DEV)
    lps, loss = torch.empty(B, device=DEV), torch.empty(1, device=DEV)
    ctx.ssi_loss(pd, td, H, W, alpha, scales, want_grad=False, loss_ps=lps, loss=loss, dout=d32, dout_ld=ld)
    again = ctx.ssi_loss(pd, td, H, W, alpha, scales)                  # dense rows [B, N]
    l16 = ctx.ssi_loss(pd, td, H, W, alpha, scales, want_grad=False, dout_bf16=d16, dout_ld=ld)
    torch.cuda.synchronize()
    got_l = lps.cpu().double()
    for b in range(B):
        ref = float(Lref[b])
        tol = 1e-6 if b in exact else 1e-6 * abs(ref)
        assert abs(float(got_l[b]) - ref) <= tol, (b, float(got_l[b]), ref)
    assert abs(float(loss) - float(Lref.mean())) <= 1e-6 * abs(float(Lref.mean()))
    g = d32[:, :N].cpu().double()
    for b in range(B):
        if b in exact:
            continue
        m = float(Gref[b].abs().max())
        if m == 0.0:                                          # constant prediction
            assert float(g[b].abs().max()) == 0.0, b
        else:
            assert float((g[b] - Gref[b]).abs().max()) <= 2e-6 * m, (b, float((g[b] - Gref[b]).abs().max()) / m)
    assert torch.all(d32[:, N:] == sentinel) and torch.all(d16[:, N:] == sentinel)        # the row padding untouched
    assert torch.equal(bits(d16[:, :N]), bits(d32[:, :N].to(torch.bfloat16)))
    # the same inputs give the same bits
    assert torch.equal(bits(again[1]), bits(lps)) and torch.equal(bits(again[0]), bits(loss))
    assert torch.equal(bits(again[2]), bits(d32[:, :N].contiguous()))
    assert torch.equal(bits(l16[1]), bits(lps))


def test_argument_errors(ctx):
    p = torch.zeros(2, N, device=DEV)
    for kw, msg in ((dict(alpha=-0.1), "alpha"), (dict(scales=0), "scales"), (dict(scales=5), "scales"),
                    (dict(dout_ld=4000), "dout_ld")):
        with pytest.raises(L.A3DError, match=msg):
            ctx.ssi_loss(p, p, H, W, **kw)
    big = torch.zeros(1, 200 * 200, device=DEV)
    with pytest.raises(L.A3DError, match=r"H\*W = 40000 exceeds"):
        ctx.ssi_loss(big, big, 200, 200)
    import ctypes as C
    ptr = C.c_void_p(p.data_ptr())
    args = dict(out=ptr, tar=ptr, loss_per_sample=ptr, loss=ptr)
    for name in args:
        a = dict(args, **{name: None})
        rc = ctx.lib.a3d_ssi_loss(ctx.h, a["out"], a["tar"], 2, H, W, 0.5, 4, a["loss_per_sample"], a["loss"], None,
                                  None, 0, None)
        with pytest.raises(L.A3DError, match=f"{name} is null"):
            L.check(rc, "ssi_loss")


# ---------------------------------------------------------------------------------------------- the model
def make_inputs(B, seed=0):
    g = torch.Generator().manual_seed(seed)
    images = torch.rand(B, 480, 640, 3, generator=g)
    depths = torch.rand(B, 55, 73, 1, generator=g) * 0.95 + 0.05
    mask = (torch.rand(B, 4096, generator=torch.Generator().manual_seed(2)) < 0.5).float()
    p = OM.init_params(1, torch.float32, bias_range=0.05)
    p["coarse/dense/dense_1/bias"] += 1.0
    p["fine/third/bias"] += 1.0
    return images, depths, mask, p


def build(B, p, mask, images, depths, train=True, **kw):
    op = models.msdn(images.to(DEV).contiguous(), depths.to(DEV).contiguous(), train=train, loss="ssi", **kw)
    op.net.load_params(p)
    if train:
        op.net.set_dropout_mask(mask.to(DEV))
    return op


LOSS_KEYS = {"loss_coarse": "loss/coarse_loss", "loss_fine": "loss/fine_loss"}


def cos(a, b):
    a, b = a.double().cpu().reshape(-1), b.double().cpu().reshape(-1)
    return float((a @ b) / (a.norm() * b.norm() + 1e-300))


def forward_backward(op):
    op.net.forward()
    op.net.backward_coarse()            # the phase-1 gradients
    op.net.backward_fine()              # the phase-2 gradients
    torch.cuda.synchronize()
    return op.net.export_grads()


# The bias of the one-channel fine/third adds the same constant to every pixel of the fine map, and the loss is
# invariant to a shift: its gradient, the sum of dL/dp over all pixels, is exactly 0, so what is computed is rounding
# noise and has no direction.  It is bounded against the sum of |dL/dp| it is summed from instead.
SHIFT_BIAS = "fine/third/bias"


def worst_cosine(op, got, ref):
    g = got[SHIFT_BIAS].double().abs().sum()
    l1 = op.net.g_fine.double().abs().sum()
    print(f"{SHIFT_BIAS}: |gradient| {float(g):.3e} = {float(g / l1):.1e} of sum |dL/dp|")
    assert float(g) <= 1e-2 * float(l1)
    return min((cos(got[n], r), n) for n, r in ref.items() if n != SHIFT_BIAS)


@pytest.mark.parametrize("B", [2, 32])
def test_msdn_ssi_bf16_vs_oracle(B):
    images, depths, mask, p = make_inputs(B)
    op = build(B, p, mask, images, depths)
    got = forward_backward(op)
    p64 = {k: v.double() for k, v in p.items()}
    _, ref = S.msdn_grads(p64, images.double(), depths.double(), mask.double(), "all")
    gq, _ = S.msdn_grads(p64, images.double(), depths.double(), mask.double(), "all", q=OM.bf16_round)
    for key in ("loss_coarse", "loss_fine"):
        lg, lr = float(op.losses[LOSS_KEYS[key]]), float(ref[key])
        print(f"B={B} {key}: {lg:.6f} vs float64 {lr:.6f}")
        assert abs(lg - lr) <= 1e-2 * abs(lr), key
    worst_cosine(op, got, gq)
    # The loss gradient is a sum of signs of pair differences, so bf16 noise in the forward that the oracle's storage
    # points do not follow (split-K sums, the bf16 backward chain) moves it more than silog's smooth gradient.  Measured
    # on the B200: worst cosine 0.9990-0.9991 at B = 2 and 0.9985-0.9988 at B = 32 (coarse convolutions) over two runs;
    # 3xTF32 reaches 0.9999997 against float64 (test below), so the loss kernel is not what limits it.
    for n, r in sorted(gq.items()):
        if n != SHIFT_BIAS:
            c = cos(got[n], r)
            print(f"B={B} {n:34s} cos={c:.6f}")
            assert c >= 0.998, (n, c)


def test_msdn_ssi_tf32_vs_float64():
    B = 2
    images, depths, mask, p = make_inputs(B)
    op = build(B, p, mask, images, depths, dtype="tf32x3")
    got = forward_backward(op)
    p64 = {k: v.double() for k, v in p.items()}
    g64, ref = S.msdn_grads(p64, images.double(), depths.double(), mask.double(), "all")
    for key in ("loss_coarse", "loss_fine"):
        lg, lr = float(op.losses[LOSS_KEYS[key]]), float(ref[key])
        print(f"3xTF32 {key}: {lg:.7f} vs float64 {lr:.7f} ({abs(lg - lr) / abs(lr):.1e})")
        assert abs(lg - lr) <= 1e-4 * abs(lr), key
    worst = worst_cosine(op, got, g64)
    print("worst gradient cosine vs float64:", worst)
    assert worst[0] >= 0.9999, worst


def test_msdn_ssi_fp8_inference_losses(ctx):
    B = 2
    images, depths, mask, p = make_inputs(B)
    op = build(B, p, mask, images, depths, train=False, dtype="fp8")
    op.run()
    torch.cuda.synchronize()
    net = op.net
    for pred, lps, loss in ((net.coarse, net.lps_coarse, net.loss_coarse), (net.fine, net.lps_fine, net.loss_fine)):
        ref_loss, ref_lps, _, _ = ctx.ssi_loss(pred, net.tar, H, W, 0.5, 4, want_grad=False)
        assert torch.equal(bits(ref_lps), bits(lps)) and torch.equal(bits(ref_loss), bits(loss))


def test_msdn_ssi_four_stream_graph_step():
    """The phase-1 step on four streams, eager and as a replayed CUDA graph.  The maps themselves may differ between
    the two in the last bits (split-K partial sums meet in float atomics), so each step's losses and loss gradient are
    checked bit for bit against the loss kernel run again on that step's own maps, and the two steps against each
    other within the overlap tests' bounds."""
    B = 32
    images, depths, mask, p = make_inputs(B)
    op = build(B, p, mask, images, depths)
    net, ctx = op.net, op.net.ctx
    res = []
    for use_graph in (False, True):
        assert op.run(use_graph=use_graph) == 1
        torch.cuda.synchronize()
        g = torch.zeros(B, 4096, dtype=torch.bfloat16, device=DEV)
        loss, lps, _, _ = ctx.ssi_loss(net.coarse, net.tar, H, W, 0.5, 4, want_grad=False, dout_bf16=g, dout_ld=4096)
        torch.cuda.synchronize()
        assert torch.equal(bits(loss), bits(net.loss_coarse)) and torch.equal(bits(lps), bits(net.lps_coarse))
        assert torch.equal(bits(g[:, :N]), bits(net.g_coarse[:, :N]))
        res.append((float(net.loss_coarse), float(net.loss_fine), net.g_coarse[:, :N].float().clone()))
    (a0, a1, ag), (b0, b1, bg) = res
    assert abs(a0 - b0) <= 1e-3 * abs(a0) and abs(a1 - b1) <= 1e-3 * abs(a1)
    assert cos(ag, bg) > 0.999


_RECORD = r"""
import json, sys
sys.path.insert(0, sys.argv[1])
import make_schedule_golden as G
G.install()
out = {}
for loss in ("silog", "ssi"):
    for name, rec in (("overlap B=32", G.single(32, loss=loss)), ("phase 2 B=2", G.single(2, phase=2, loss=loss)),
                      ("inference B=2", G.single(2, train=False, loss=loss)),
                      ("tf32 phase 1 B=2", G.single(2, dtype="tf32", loss=loss))):
        out[f"{name} {loss}"] = rec()
json.dump(out, open(sys.argv[2], "w"))
"""

LOSS_SCALARS = ("lambda_over_n", "H", "W", "alpha", "scales")


def as_silog(ln):
    """A recorded ssi_loss launch read as silog_loss: the method renamed and the loss-specific scalars dropped."""
    ln = json.loads(json.dumps(ln))
    if ln["m"] == "ssi_loss":
        ln["m"] = "silog_loss"
        if ln["args"]["dout_ld"] <= 0:                   # as the recorder normalises silog_loss: 0 means n
            ln["args"]["dout_ld"] = N
    for k in LOSS_SCALARS:
        ln["args"].pop(k, None)
    return ln


def test_ssi_launch_list_equals_silog_launch_list():
    """loss="ssi" changes only the loss kernel: the same launches with the same buffers, streams and ordering."""
    env = {k: v for k, v in os.environ.items() if not k.startswith("A3D_")}
    with tempfile.TemporaryDirectory() as tmp:
        out = os.path.join(tmp, "launches.json")
        r = subprocess.run([sys.executable, "-c", _RECORD, os.path.join(ROOT, "tests", "golden"), out], env=env,
                           capture_output=True, text=True, timeout=1200, cwd=ROOT)
        assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
        rec = json.load(open(out))
    for name in ("overlap B=32", "phase 2 B=2", "inference B=2", "tf32 phase 1 B=2"):
        a, b = rec[f"{name} silog"], rec[f"{name} ssi"]
        assert a["lanes"] == b["lanes"], name
        assert sum(ln["m"] == "ssi_loss" for ln in b["launches"]) == 2, name
        assert not any(ln["m"] == "silog_loss" for ln in b["launches"]), name
        la, lb = [as_silog(x) for x in a["launches"]], [as_silog(x) for x in b["launches"]]
        assert len(la) == len(lb), name
        for i, (x, y) in enumerate(zip(la, lb)):
            assert x == y, f"{name} launch {i}: {json.dumps(x)[:300]} vs {json.dumps(y)[:300]}"


def test_driver_trains_with_ssi_and_resumes(tmp_path):
    def run(*extra):
        cmd = [sys.executable, "-u", "-m", "ann3depth_b200.ann3depth", "nyu", "--batchsize", "2", "--ckptdir",
               str(tmp_path), "--datadir", str(tmp_path / "no_data"), "--sumfreq", "1", "--loss", "ssi", *extra]
        return subprocess.run(cmd, cwd=ROOT, capture_output=True, text=True, timeout=300)
    r = run("--steps", "3")
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
    assert "step 3 losses" in r.stdout and "loss/coarse_loss" in r.stdout
    st = torch.load(os.path.join(tmp_path, "msdn", "model.ckpt"), map_location="cpu")
    assert st["global_step"] == 3
    r2 = run("--steps", "5")
    assert r2.returncode == 0 and "Restored checkpoint at global step 3" in r2.stdout and "step 5 losses" in r2.stdout
