"""GPU tests of the affine (least-squares scale-and-shift) mode of `a3d_depth_metrics` against the float64 oracle
(oracle/metrics_affine.py) at both models' shapes, its CUDA-graph replay, `evaluate --scale affine` end to end and
`--evalfreq` with `--evalscale affine`."""
import json

import numpy as np
import pytest
import torch

from ann3depth_b200 import data, models
from ann3depth_b200._lib import DM_SLOTS
from oracle import metrics as OM
from oracle import metrics_affine as OA

from test_gpu_eval import COUNTS, LOG, N_TEST, SUMS, _assert_close, _inputs, _read_scalars, _run, _test_split, _tol

pytestmark = pytest.mark.gpu


def _affine_inputs(ctx, B, ph, pw, gh, gw, seed):
    """_inputs (NaN predictions, gt above max_depth, zeros, an image without a valid pixel) plus +-inf predictions, a
    negative-slope image 0 whose ground truth follows its own upsampled prediction, and a constant image 2."""
    pred, gt = _inputs(B, ph, pw, gh, gw, seed)
    g = torch.Generator(device="cuda").manual_seed(seed)
    pred[0] = torch.rand(ph, pw, device="cuda", generator=g) * 0.9 + 0.05
    flat = pred.view(-1)
    idx = torch.randperm(flat.numel(), device="cuda", generator=g)[:8]
    flat[idx[:4]] = float("inf")
    flat[idx[4:]] = float("-inf")
    up0 = ctx.resize_bilinear_tf1(pred[:1].unsqueeze(-1), gh, gw)[0, ..., 0]
    noise = (torch.rand(gh, gw, device="cuda", generator=g) - 0.5) * 0.04
    gt[0] = torch.where(torch.isfinite(up0), 0.95 - 0.8 * up0 + noise, torch.zeros_like(up0))
    gt[0, :3] = 1.5                                                           # > max_depth: invalid
    if B > 2:
        pred[2] = 2.0                                                         # every sample clamped: s = 1
    return pred.contiguous(), gt.contiguous()


CASES = {"msdn": (32, 55, 74, 480, 640), "dcnf": (16, 240, 320, 480, 640), "b1": (1, 55, 74, 480, 640),
         "cluster1": (None, 55, 74, 55, 73)}


@pytest.mark.parametrize("case", list(CASES))
def test_affine_depth_metrics_matches_oracle(case):
    B, ph, pw, gh, gw = CASES[case]
    ctx = models.get_context()
    if B is None:
        B = ctx.sm_count // 2 + 1                                             # B * 2 > SM count: clusters of 1
    pred, gt = _affine_inputs(ctx, B, ph, pw, gh, gw, seed=B * 7 + ph)
    st = torch.full((B, 2), -7.0, device="cuda")
    sums = ctx.depth_metrics(pred, gt, 1e-3, 1.0, affine=True, scale=st)
    up = ctx.resize_bilinear_tf1(pred.unsqueeze(-1), gh, gw)                  # what the kernel samples, bit for bit
    torch.cuda.synchronize()
    sums, st, up, gtc = sums.cpu().numpy(), st.cpu().numpy(), up.cpu().numpy()[..., 0], gt.cpu().numpy()
    exact = 0
    for b in range(B):
        _, (s_ref, t_ref) = OA.image_sums(up[b], gtc[b])
        s, t = st[b]
        assert abs(s - s_ref) <= 1e-5 * abs(s_ref), (b, s, s_ref)
        assert abs(t - t_ref) <= 1e-5 * (abs(t_ref) + abs(s_ref)), (b, t, t_ref)
        exact += s == s_ref and t == t_ref
        # the slots at the kernel's own (s, t): the tolerances of the other modes
        ref, _ = OA.image_sums(up[b], gtc[b], fit=(s, t))
        assert np.array_equal(sums[b][COUNTS], ref[COUNTS]), (b, sums[b][COUNTS], ref[COUNTS])
        np.testing.assert_allclose(sums[b][SUMS], ref[SUMS], rtol=1e-6, atol=0, err_msg=f"image {b}")
        assert abs(sums[b][LOG] - ref[LOG]) <= 1e-6 * max(ref[6] * np.log(10.0), 1e-30), b
    print(f"{case}: B = {B}, (s, t) bit-identical to the oracle's in {exact} of {B} images")
    assert st[0, 0] == pytest.approx(-0.8, abs=0.01) and st[0, 1] == pytest.approx(0.95, abs=0.01)
    assert sums[0][DM_SLOTS.index("delta1")] > 0.9 * sums[0][0]
    if B > 2:
        assert not sums[1].any() and tuple(st[1]) == (1.0, 0.0)
        assert st[2, 0] == 1.0 and sums[2][0] > 0


def test_affine_mode_removes_an_exact_scale_and_shift():
    """A prediction that is an exact negative-slope affine map of the ground truth scores no error in the affine mode,
    and badly without alignment; an image without a valid pixel writes zeros and (s, t) = (1, 0)."""
    ctx = models.get_context()
    g = torch.Generator(device="cuda").manual_seed(3)
    pred = torch.rand(2, 60, 80, device="cuda", generator=g) * 0.8 + 0.1
    gt = (0.9 - 0.7 * pred).contiguous()                                      # same grid: p~ = pred exactly
    gt[1] = 0.0
    st = torch.zeros(2, 2, device="cuda")
    aff = ctx.depth_metrics(pred, gt, 1e-3, 1.0, affine=True, scale=st).cpu()
    st = st.cpu()
    none = ctx.depth_metrics(pred, gt, 1e-3, 1.0).cpu()
    n = 60 * 80
    assert aff[0, 0] == n and aff[0, DM_SLOTS.index("delta1")] == n
    assert aff[0, DM_SLOTS.index("abs_rel")] / n < 1e-5
    assert none[0, DM_SLOTS.index("delta1")] < 0.5 * n
    assert not aff[1].any() and not none[1].any() and tuple(st[1].tolist()) == (1.0, 0.0)
    assert st[0, 0].item() == pytest.approx(-0.7, rel=1e-5) and st[0, 1].item() == pytest.approx(0.9, rel=1e-5)


def test_affine_graph_replay_is_identical():
    ctx = models.get_context()
    pred, gt = _affine_inputs(ctx, 32, 55, 74, 480, 640, seed=11)
    sums = torch.zeros(32, len(DM_SLOTS), dtype=torch.float64, device="cuda")
    st = torch.zeros(32, 2, device="cuda")
    ctx.depth_metrics(pred, gt, 1e-3, 1.0, affine=True, sums=sums, scale=st)
    eager, eager_st = sums.clone(), st.clone()
    gr = torch.cuda.CUDAGraph()
    with torch.cuda.graph(gr):
        ctx.depth_metrics(pred, gt, 1e-3, 1.0, affine=True, sums=sums, scale=st)
    for _ in range(3):
        sums.zero_()
        st.zero_()
        gr.replay()
        torch.cuda.synchronize()
        assert torch.equal(sums, eager) and torch.equal(st, eager_st)


def test_affine_argument_errors():
    ctx = models.get_context()
    pred, gt = _inputs(2, 55, 74, 480, 640, seed=1)
    with pytest.raises(ValueError, match="exclusive"):
        ctx.depth_metrics(pred, gt, 1e-3, 1.0, median=True, affine=True)
    with pytest.raises(ValueError, match=r"\[B, 2\]"):
        ctx.depth_metrics(pred, gt, 1e-3, 1.0, affine=True, scale=torch.zeros(2, device="cuda"))


# ------------------------------------------------------------------------------------------------ end to end
def _affine_oracle_of_checkpoint(model, ckptdir, datadir, B=2):
    """The model's own infer() outputs in this process, upsampled on the GPU, through the float64 affine oracle."""
    from ann3depth_b200.ann3depth import restore_checkpoint
    from ann3depth_b200.evaluate import model_outputs
    inp = data.inputs(datadir, "nyu", B, "test", epochs=1)
    op = getattr(models, model)(inp.images, inp.depths, train=False)
    assert restore_checkpoint(op, ckptdir)
    ctx = op.net.ctx
    per = {}
    while True:
        n = inp.next_batch()
        if not n:
            break
        op.net.infer()
        for name, t in model_outputs(op).items():
            up = ctx.resize_bilinear_tf1(t, 480, 640).cpu().numpy()[..., 0]
            gt = inp.depths.cpu().numpy()[..., 0]
            per.setdefault(name, []).extend(OA.image_sums(up[b], gt[b])[0] for b in range(n))
    inp.close()
    return {name: OM.dataset_metrics(np.stack(v)) for name, v in per.items()}, op.global_step


@pytest.mark.parametrize("model,outputs", [("msdn", ("fine", "coarse")), ("dcnf", ("output",))])
def test_evaluate_affine_end_to_end(tmp_path, model, outputs):
    _test_split(str(tmp_path))
    ck = tmp_path / "ckpt"
    _run("ann3depth_b200.ann3depth", "nyu", "--model", model, "--steps", "2", "--batchsize", "2", "--ckptdir", str(ck),
         "--datadir", str(tmp_path), "--sumfreq", "1")
    out = tmp_path / f"{model}_affine.json"
    r = _run("ann3depth_b200.evaluate", "nyu", "--model", model, "--ckptdir", str(ck), "--batchsize", "2",
             "--datadir", str(tmp_path), "--scale", "affine", "--json", str(out))
    res = json.loads(out.read_text())
    assert res["scale"] == "affine" and res["model"] == model and res["global_step"] == 2 and res["images"] == N_TEST
    assert set(res["metrics"]) == set(outputs)
    ref, step = _affine_oracle_of_checkpoint(model, str(ck / model), str(tmp_path))
    assert step == 2 and res["pixels"] == ref[outputs[0]]["pixels"]
    for name in outputs:
        _assert_close(res["metrics"][name], ref[name])
    assert f"{model}/{outputs[0]} at step 2 on 5 images" in r.stdout


def test_evalfreq_with_affine_scale_writes_eval_scalars(tmp_path):
    _test_split(str(tmp_path))
    ck = tmp_path / "ckpt"
    r = _run("ann3depth_b200.ann3depth", "nyu", "--steps", "2", "--evalfreq", "1", "--evalscale", "affine",
             "--batchsize", "2", "--ckptdir", str(ck), "--datadir", str(tmp_path), "--sumfreq", "1", "--id", "aff")
    assert "step 1 eval" in r.stdout and "step 2 eval" in r.stdout
    sc = _read_scalars(str(ck / "msdn_aff"))
    for step in (1, 2):
        for k in OM.METRICS:
            assert (step, f"eval/fine/{k}") in sc and (step, f"eval/coarse/{k}") in sc, (step, k)
    out = tmp_path / "final.json"
    _run("ann3depth_b200.evaluate", "nyu", "--model", "msdn", "--ckptdir", str(ck), "--id", "aff", "--batchsize", "2",
         "--datadir", str(tmp_path), "--scale", "affine", "--json", str(out))
    res = json.loads(out.read_text())
    assert res["global_step"] == 2
    for name in ("fine", "coarse"):
        for k in OM.METRICS:
            assert sc[(2, f"eval/{name}/{k}")] == pytest.approx(res["metrics"][name][k], **_tol(k)), (name, k)
