"""GPU parity at the BASELINE configurations themselves (BASELINE.json configs 2 and 4), not at toy batches:

  * MSDN batch 32 (Makefile:37-40, src/models.py:277-367): forward, both losses, all-parameter gradients and one
    general (beta2 = 0.999) TF-Adam phase-1 step -- run AFTER the first-use autotuner has picked its tiles / split-K
    factors for the batch-32 shapes, through the same CUDA-graph multi-stream schedule bench.py times; the same step at
    batch 64, where the dense weight gradients and their TF-Adam update run as separate kernels;
  * DCNF batch 16 (src/models.py:179-200): unary outputs, CRF solve, loss, unary gradients;
  * the device dropout RNG the bench actually runs (`a3d_bernoulli_mask`): keep rate, determinism per (seed, step),
    replay-to-replay change inside the captured graph.

Tolerances (BASELINE.json north_star): forward depth maps + losses 1e-2 relative (BF16); per-parameter gradient cosine
>= 0.999 against the oracle evaluated at the BF16 storage points; the cosine against the unrounded float64 oracle is
printed and, at batch 32 and 64, bounded by the same 0.999 (at batch 2 only >= 0.99: see tests/test_gpu_msdn.py); CRF solve 1e-5.
"""
import pytest
import torch

pytestmark = pytest.mark.gpu

from oracle import dcnf as OD
from oracle import msdn as OM

if torch.cuda.is_available():
    from ann3depth_b200 import models

DEV = "cuda:0"
B32 = 32


def rel(a, b):
    a, b = a.double().cpu(), b.double().cpu()
    return float((a - b).abs().max() / b.abs().max())


def cos(a, b):
    a, b = a.double().cpu().reshape(-1), b.double().cpu().reshape(-1)
    return float((a @ b) / (a.norm() * b.norm() + 1e-300))


def rms(t):
    return float(t.double().pow(2).mean().sqrt())


def msdn_inputs(B):
    """Inputs and conditioned parameters at batch B."""
    g = torch.Generator().manual_seed(0)
    images = torch.rand(B, 480, 640, 3, generator=g)
    depths = torch.rand(B, 55, 73, 1, generator=g) * 0.95 + 0.05
    mask = (torch.rand(B, 4096, generator=torch.Generator().manual_seed(2)) < 0.5).float()
    p = OM.init_params(1, torch.float32, bias_range=0.05)
    p["coarse/dense/dense_1/bias"] += 1.0          # keep predictions away from the log() discontinuity at 0
    p["fine/third/bias"] += 1.0
    return dict(B=B, images=images, depths=depths, mask=mask, p=p, p64={k: v.double() for k, v in p.items()})


@pytest.fixture(scope="module")
def msdn32():
    return msdn_inputs(B32)


def with_oracle(s):
    """s plus the float64 oracle results at its inputs (~15 s of CPU at batch 32, twice that at 64)."""
    i64, d64, m64 = s["images"].double(), s["depths"].double(), s["mask"].double()
    s["gq"], s["fq"] = OM.grads(s["p64"], i64, d64, m64, "all", q=OM.bf16_round)          # BF16 storage points
    s["g64"], s["f64"] = OM.grads(s["p64"], i64, d64, m64, "all")                          # unrounded
    return s


def build_msdn(s, **kw):
    op = models.msdn(s["images"].to(DEV).contiguous(), s["depths"].to(DEV).contiguous(), train=True, **kw)
    op.net.load_params(s["p"])
    op.net.set_dropout_mask(s["mask"].to(DEV))
    return op


def test_msdn_b32_step_forward_gradients_adam(msdn32):
    check_step_forward_gradients_adam(with_oracle(dict(msdn32)))


def test_msdn_b64_step_forward_gradients_adam():
    """The same step and tolerances at batch 64, above the fused dense wgrad + TF-Adam kernel's batch limit: there the
    dense weight gradients and their TF-Adam update run as separate kernels."""
    check_step_forward_gradients_adam(with_oracle(msdn_inputs(64)))


def check_step_forward_gradients_adam(s):
    B = s["B"]
    # ---- 1. one real step exactly as bench.py runs it: first use autotunes every shape of the batch, then the phase-1
    #         CUDA graph (4 streams; fused dense wgrad + Adam at B = 32, separate kernels at 64) is captured and replayed
    op = build_msdn(s, beta2=0.999)
    assert op.run(use_graph=True) == 1
    torch.cuda.synchronize()
    net = op.net
    st = OM.TrainState(s["p64"], beta2=0.999)
    out_q, ph = OM.train_step(st, s["images"].double(), s["depths"].double(), s["mask"].double(), q=OM.bf16_round)
    assert ph == 1
    # forward of that step (the graph's outputs)
    rc, rf = rel(op.coarse, s["f64"]["coarse"]), rel(op.outputs, s["f64"]["fine"])
    print(f"B={B} forward: coarse rel vs f64 {rc:.2e} (vs bf16-point {rel(op.coarse, s['fq']['coarse']):.2e}), "
          f"fine {rf:.2e} (vs bf16-point {rel(op.outputs, s['fq']['fine']):.2e})")
    assert rc < 1e-2 and rf < 1e-2
    lc, lf = float(op.losses["loss/coarse_loss"]), float(op.losses["loss/fine_loss"])
    rlc, rlf = float(s["f64"]["loss_coarse"]), float(s["f64"]["loss_fine"])
    print(f"B={B} losses: coarse {lc:.4f} (f64 {rlc:.4f}), fine {lf:.4f} (f64 {rlf:.4f})")
    assert abs(lc - rlc) < 1e-2 * abs(rlc) and abs(lf - rlf) < 1e-2 * abs(rlf)
    # ---- 2. TF-Adam state after the step, per element.  m = 0.1 g, v = 0.001 g^2 inherit the gradient's BF16 noise
    #         (~1 % rms, measured below), so the bounds are relative to each tensor's scale.
    got_w = net.export_params()
    got_m, got_v = net.arena.export_tf(net.arena.m), net.arena.export_tf(net.arena.v)
    for name in st.p:
        if not name.startswith("coarse/"):
            assert torch.equal(got_w[name], s["p"][name]), name                     # fine stack untouched in phase 1
            continue
        m_ref, v_ref = st.m[name], st.v[name]
        em, ev = (got_m[name].double() - m_ref).abs(), (got_v[name].double() - v_ref).abs()
        dw, dw_ref = got_w[name].double() - s["p64"][name], st.p[name] - s["p64"][name]
        lr = OM.ADAM_GROUPS[OM.group_of(name)][0]
        # first TF-Adam step: dw = -lr_t m / (sqrt(v) + eps) ~ -lr sign(g).  Elements whose gradient is numerically zero
        # have no defined sign; count the others
        sig = m_ref.abs() > 1e-3 * m_ref.abs().max()
        wrong = float(((dw - dw_ref).abs() > 0.05 * lr)[sig].double().mean()) if bool(sig.any()) else 0.0
        print(f"{name:32s} m: max err {float(em.max() / m_ref.abs().max()):.2e} rms err {rms(em) / rms(m_ref):.2e} | "
              f"v: max err {float(ev.max() / v_ref.abs().max()):.2e} rms err {rms(ev) / rms(v_ref):.2e} | "
              f"dw: cos {cos(dw, dw_ref):.5f} wrong-sign fraction {wrong:.2e} max|dw| {float(dw.abs().max()):.4f} "
              f"(oracle {float(dw_ref.abs().max()):.4f})")
        assert float(em.max()) <= 5e-2 * float(m_ref.abs().max()), name
        assert rms(em) <= 2e-2 * rms(m_ref), name
        assert float(ev.max()) <= 1e-1 * float(v_ref.abs().max()), name
        assert rms(ev) <= 4e-2 * rms(v_ref), name
        assert wrong < 2e-2, name
        assert abs(float(dw.abs().max()) / float(dw_ref.abs().max()) - 1) < 0.02, name
    # ---- 3. all-parameter gradients with the tuned kernels (same process: the tuner cache is keyed by shape)
    op2 = build_msdn(s)
    n2 = op2.net
    n2.forward()
    n2.backward_coarse()
    n2.backward_fine()
    torch.cuda.synchronize()
    got = n2.export_grads()
    worst, worst64, bad = 1.0, 1.0, []
    for name, g in s["gq"].items():
        c, c64 = cos(got[name], g), cos(got[name], s["g64"][name])
        nr = float(got[name].double().norm() / (g.norm() + 1e-300))
        print(f"{name:32s} cos={c:.6f} norm ratio={nr:.4f}  (vs unrounded f64: cos={c64:.6f})")
        worst, worst64 = min(worst, c), min(worst64, c64)
        # at batch 32 (and 64) the ReLU-flip noise averages out far enough that even the UNROUNDED float64 oracle is met at
        # the north star's 0.999 (measured on B200 at batch 32: worst 0.99942, profiles/parity_full_r02.log)
        if not (c >= 0.999 and 0.97 < nr < 1.03 and c64 >= 0.999):
            bad.append(name)
    print(f"B={B} worst gradient cosine: bf16-point oracle", worst, "| unrounded float64 oracle", worst64)
    assert not bad, bad


def test_msdn_b32_graph_replays_are_consistent(msdn32):
    """Replays of the captured batch-32 graph with the reference's Adam (beta2 = 1): weights bit-frozen, losses stable."""
    op = build_msdn(msdn32)
    w0 = op.net.arena.w.clone()
    losses = []
    for _ in range(3):
        op.run()
        losses.append((float(op.losses["loss/coarse_loss"]), float(op.losses["loss/fine_loss"])))
    torch.cuda.synchronize()
    assert torch.equal(op.net.arena.w, w0) and op.global_step == 3 and int(op.net.step_dev) == 3
    for lc, lf in losses[1:]:                      # split-K atomics: last-bit differences only
        assert abs(lc - losses[0][0]) <= 1e-4 * abs(losses[0][0]) and abs(lf - losses[0][1]) <= 1e-4 * abs(losses[0][1])


def test_bernoulli_mask_device_rng():
    """`a3d_bernoulli_mask` (the dropout mask bench.py and the train loop use; src/models.py:230 is unseeded TF dropout):
    Bernoulli(0.5) bytes, deterministic in (seed, step counter), different for another seed or step."""
    ctx = models.get_context(0)
    n = 32 * 4096
    step = torch.zeros(1, dtype=torch.int64, device=DEV)

    def draw(seed, t, keep_prob=0.5):
        step.fill_(t)
        k = torch.full((n,), 7, dtype=torch.uint8, device=DEV)
        ctx.bernoulli_mask(k, keep_prob, seed, step)
        return k
    a, a2, b, c = draw(2, 0), draw(2, 0), draw(2, 1), draw(3, 0)
    assert int(a.max()) == 1 and int(a.min()) == 0
    assert torch.equal(a, a2)
    rate = float(a.float().mean())
    assert abs(rate - 0.5) < 5 * 0.5 / n ** 0.5, rate                      # 5 sigma
    for other in (b, c):                                                    # independent draws agree on ~half the bytes
        agree = float((a == other).float().mean())
        assert abs(agree - 0.5) < 5 * 0.5 / n ** 0.5, agree
    assert abs(float(draw(2, 5, 0.8).float().mean()) - 0.8) < 5 * 0.4 / n ** 0.5
    # neighbouring bytes are uncorrelated (a counter-mode hash, not an LCG over the index)
    x = a.float() - 0.5
    assert abs(float((x[:-1] * x[1:]).mean())) < 5 * 0.25 / n ** 0.5


def test_dropout_mask_changes_between_graph_replays(msdn32):
    """Inside the captured graph the mask is a function of the device step counter: every replay draws a new one, and a
    second net with the same seed reproduces the sequence."""
    s = msdn32
    seqs = []
    for _ in range(2):
        op = models.msdn(s["images"].to(DEV).contiguous(), s["depths"].to(DEV).contiguous(), train=True, dropout_seed=11)
        op.net.load_params(s["p"])
        masks = []
        for _ in range(3):
            op.run()
            torch.cuda.synchronize()
            masks.append(op.net.keep_mask.clone())
        seqs.append(masks)
    m = seqs[0]
    assert not torch.equal(m[0], m[1]) and not torch.equal(m[1], m[2])
    assert abs(float(m[1].float().mean()) - 0.5) < 0.01
    for x, y in zip(*seqs):
        assert torch.equal(x, y)


def _bf16(t):
    return t.to(torch.bfloat16).to(t.dtype)


def test_dcnf_b16_forward_crf_gradients():
    """BASELINE config 4: DCNF batch 16 = 768 patches through the unary CNN, 16 CRF graphs."""
    B = 16
    g = torch.Generator().manual_seed(3)
    images = torch.rand(B, 480, 640, 3, generator=g)
    depths = torch.rand(B, 480, 640, 1, generator=g) * 0.95 + 0.05
    p = OD.init_params(5, torch.float32, bias_range=0.05, pairwise_nonneg=True)
    op = models.dcnf(images.to(DEV), depths.to(DEV), train=True, naive_loss=False)
    net = op.net
    net.load_params(p)
    net.forward()
    net.backward()
    torch.cuda.synchronize()
    p64 = {k: v.double() for k, v in p.items()}
    gref, ref = OD.grads(p64, images.double(), depths.double(), q=_bf16, stable=True)
    z, zr = net.z.view(B, 48).cpu().double(), ref["z"].reshape(B, 48)
    print("B=16 z rel", float((z - zr).abs().max() / zr.abs().max()))
    assert float((z - zr).abs().max() / zr.abs().max()) < 1e-2
    assert float((net.r.cpu().double() - ref["r"].reshape(B, 48)).abs().max()) < 1e-5
    assert float((net.y.cpu().double() - ref["y"].reshape(B, 48)).abs().max()) < 1e-6
    assert int(net.status.abs().max()) == 0
    A = OD.build_A(net.r.cpu().double().reshape(B, 48, 1))
    ystar = OD.crf_map(A, z.reshape(B, 48, 1)).reshape(B, 48)
    err = float((net.ystar.cpu().double() - ystar).abs().max())
    print("B=16 CRF solve max err", err)
    assert err < 1e-5
    lref = float(OD.nll_stable(A, ref["y"], z.reshape(B, 48, 1)))
    assert abs(float(net.loss) - lref) < 1e-3 * max(1.0, abs(lref))
    assert abs(float(net.loss) - float(ref["loss"])) < 2e-2 * max(1.0, abs(float(ref["loss"])))
    got = net.export_grads()
    bad = []
    for name, gr in gref.items():
        c = cos(got[name], gr)
        nr = float(got[name].double().norm() / (gr.norm() + 1e-300))
        print(f"{name:36s} cos={c:.6f} norm ratio={nr:.4f}")
        if float(gr.abs().max()) == 0.0:
            assert float(got[name].abs().max()) == 0.0, name               # no gradient reaches the pairwise layer
        elif not (c >= 0.999 and 0.97 < nr < 1.03):
            bad.append(name)
    assert not bad, bad
    # one SGD step at batch 16 (src/models.py:198-200)
    w0 = net.arena.w.clone()
    op.run()
    torch.cuda.synchronize()
    lo, hi = net.arena.group_range("SGD")
    assert torch.allclose(net.arena.w[lo:hi], w0[lo:hi] - 0.1 * net.arena.g[lo:hi], atol=1e-7)
