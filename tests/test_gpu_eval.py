"""GPU tests of evaluation: `a3d_depth_metrics` against the float64 oracle (oracle/metrics.py) on the output of
`a3d_resize_bilinear_tf1`, its CUDA-graph replay, the `python -m ann3depth_b200.evaluate` command end to end for both
models, and validation during training (`--evalfreq`)."""
import glob
import json
import os
import struct
import subprocess
import sys

import numpy as np
import pytest
import torch

from ann3depth_b200 import data, models
from ann3depth_b200._lib import DM_SLOTS
from oracle import metrics as OM

from test_data_cpu import _example, _write

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
COUNTS = [DM_SLOTS.index(k) for k in ("n", "delta1", "delta2", "delta3", "nonfinite")]
SUMS = [DM_SLOTS.index(k) for k in ("abs_rel", "sq_rel", "sq", "log_sq", "log10")]
LOG = DM_SLOTS.index("log")


def _inputs(B, ph, pw, gh, gw, seed):
    g = torch.Generator().manual_seed(seed)
    gt = torch.randint(0, 256, (B, gh, gw), generator=g).float() / 255.0      # k/255 relative depth: zeros are invalid
    gt[:, :3] = 1.5                                                           # > max_depth: invalid
    pred = gt.new_empty(B, ph, pw)
    pred.copy_(torch.rand(B, ph, pw, generator=g) * 1.3 - 0.1)               # some negative values, some above max_depth
    pred.view(-1)[torch.randperm(pred.numel(), generator=g)[:max(pred.numel() // 200, 1)]] = float("nan")
    if B > 1:
        gt[1] = 0.0                                                           # an image without a valid pixel
    return pred.cuda(), gt.cuda()


SHAPES = [(55, 74, 480, 640), (55, 74, 55, 73), (240, 320, 480, 640), (60, 80, 60, 80)]


@pytest.mark.parametrize("B", [1, 3, 32])
@pytest.mark.parametrize("shape", SHAPES, ids=lambda s: "%dx%d-%dx%d" % s)
@pytest.mark.parametrize("median", [False, True], ids=["none", "median"])
def test_depth_metrics_matches_oracle(shape, B, median):
    ph, pw, gh, gw = shape
    ctx = models.get_context()
    pred, gt = _inputs(B, ph, pw, gh, gw, seed=B * 7 + ph)
    scale = torch.full((B,), -1.0, device="cuda")
    sums = ctx.depth_metrics(pred, gt, 1e-3, 1.0, median=median, scale=scale)
    up = ctx.resize_bilinear_tf1(pred.unsqueeze(-1), gh, gw)                  # what the kernel samples, bit for bit
    torch.cuda.synchronize()
    sums, scale, up, gtc = sums.cpu().numpy(), scale.cpu().numpy(), up.cpu().numpy()[..., 0], gt.cpu().numpy()
    for b in range(B):
        ref, s = OM.image_sums(up[b], gtc[b], 1e-3, 1.0, median)
        assert np.array_equal(sums[b][COUNTS], ref[COUNTS]), (b, sums[b][COUNTS], ref[COUNTS])
        np.testing.assert_allclose(sums[b][SUMS], ref[SUMS], rtol=1e-6, atol=0, err_msg=f"image {b}")
        # the signed sum d can cancel: compare it against the scale of sum |d|
        assert abs(sums[b][LOG] - ref[LOG]) <= 1e-6 * max(ref[6] * np.log(10.0), 1e-30), b
        assert scale[b].view(np.int32) == np.float32(s if median else 1.0).view(np.int32), (b, scale[b], s)
    if B > 1:
        assert not sums[1].any() and scale[1] == 1.0


def test_depth_metrics_graph_replay_is_identical():
    ctx = models.get_context()
    pred, gt = _inputs(32, 55, 74, 480, 640, seed=11)
    sums = torch.zeros(32, len(DM_SLOTS), dtype=torch.float64, device="cuda")
    scale = torch.zeros(32, device="cuda")
    ctx.depth_metrics(pred, gt, 1e-3, 1.0, median=True, sums=sums, scale=scale)
    eager = sums.clone()
    gr = torch.cuda.CUDAGraph()
    with torch.cuda.graph(gr):
        ctx.depth_metrics(pred, gt, 1e-3, 1.0, median=True, sums=sums, scale=scale)
    for _ in range(3):
        sums.zero_()
        gr.replay()
        torch.cuda.synchronize()
        assert torch.equal(sums, eager)


# ------------------------------------------------------------------------------------------------ end to end
N_TEST = 5


def _test_split(root):
    rng = np.random.default_rng(0)
    recs = []
    for i in range(N_TEST):
        img = (rng.integers(0, 256, size=(480, 640, 3)) / 255.0 - 0.5).astype(np.float32)
        dep8 = rng.integers(0, 256, size=(480, 640, 1))
        dep8[: 40 * (i + 1)] = 0                                          # some invalid (zero) depth
        dep = (dep8 / 255.0 - 0.5).astype(np.float32)
        recs.append(_example({"image_height": 480, "image_width": 640, "image_channels": 3, "depth_height": 480,
                              "depth_width": 640, "depth_channels": 1, "image": img.tobytes(), "depth": dep.tobytes()},
                             True))
    os.makedirs(os.path.join(root, "nyu"), exist_ok=True)
    _write(os.path.join(root, "nyu", "test.tfrecords"), recs)


def _run(*args, timeout=900):
    r = subprocess.run([sys.executable, "-u", "-m", *args], cwd=ROOT, capture_output=True, text=True, timeout=timeout)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
    return r


def _oracle_of_checkpoint(model, ckptdir, datadir, B=2, scale="none"):
    """The model's own infer() outputs in this process, upsampled on the GPU, through the float64 oracle."""
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
            per.setdefault(name, []).extend(OM.image_sums(up[b], gt[b], median=scale == "median")[0] for b in range(n))
    inp.close()
    return {name: OM.dataset_metrics(np.stack(v)) for name, v in per.items()}, op.global_step


def _tol(k):
    # the two processes' forward passes differ in the last bits (split-K atomics); a prediction that crosses a ratio
    # threshold flips every ground-truth pixel sampling it (tens of the 1.1 M pixels), so the delta fractions get an
    # absolute margin of that size
    return dict(rel=1e-4, abs=2e-5 if k.startswith("delta") else 1e-6)


def _assert_close(got, ref):
    for k in OM.METRICS:
        assert got[k] == pytest.approx(ref[k], **_tol(k)), (k, got[k], ref[k])


@pytest.mark.parametrize("model,outputs", [("msdn", ("fine", "coarse")), ("dcnf", ("output",))])
def test_evaluate_command_end_to_end(tmp_path, model, outputs):
    _test_split(str(tmp_path))
    ck = tmp_path / "ckpt"
    _run("ann3depth_b200.ann3depth", "nyu", "--model", model, "--steps", "2", "--batchsize", "2", "--ckptdir", str(ck),
         "--datadir", str(tmp_path), "--sumfreq", "1")
    for scale in ("none", "median"):
        out = tmp_path / f"{model}_{scale}.json"
        r = _run("ann3depth_b200.evaluate", "nyu", "--model", model, "--ckptdir", str(ck), "--batchsize", "2",
                 "--datadir", str(tmp_path), "--scale", scale, "--json", str(out))
        res = json.loads(out.read_text())
        assert res["model"] == model and res["global_step"] == 2 and res["images"] == N_TEST, res
        assert set(res["metrics"]) == set(outputs)
        ref, step = _oracle_of_checkpoint(model, str(ck / model), str(tmp_path), scale=scale)
        assert step == 2 and res["pixels"] == ref[outputs[0]]["pixels"]
        for name in outputs:
            _assert_close(res["metrics"][name], ref[name])
        assert f"{model}/{outputs[0]} at step 2 on 5 images" in r.stdout
    # no test split: a clear error, no synthetic evaluation
    r = subprocess.run([sys.executable, "-m", "ann3depth_b200.evaluate", "nyu", "--model", model, "--ckptdir", str(ck),
                        "--datadir", str(tmp_path / "none")], cwd=ROOT, capture_output=True, text=True, timeout=300)
    assert r.returncode != 0 and "test.tfrecords not found" in r.stderr


def _read_scalars(logdir):
    """{(step, tag): value} of the event files in logdir (tf.Event: step = 2, summary = 5 {value = 1 {tag = 1,
    simple_value = 2}})."""
    out = {}
    for path in glob.glob(os.path.join(logdir, "events.out.tfevents.*")):
        for rec in data.tfrecord_iterator(path):
            step, vals = 0, []
            for f, _, v in data._parse_fields(rec):
                if f == 2:
                    step = v
                elif f == 5:
                    for f2, _, val in data._parse_fields(v):
                        tag, x = None, None
                        for f3, _, w in data._parse_fields(val):
                            if f3 == 1:
                                tag = bytes(w).decode()
                            elif f3 == 2:
                                x = struct.unpack("<f", bytes(w))[0]
                        vals.append((tag, x))
            for tag, x in vals:
                out[(step, tag)] = x
    return out


def test_evalfreq_writes_eval_scalars(tmp_path):
    _test_split(str(tmp_path))
    ck = tmp_path / "ckpt"
    r = _run("ann3depth_b200.ann3depth", "nyu", "--steps", "4", "--evalfreq", "2", "--batchsize", "2", "--ckptdir",
             str(ck), "--datadir", str(tmp_path), "--sumfreq", "1", "--id", "ev")
    assert "step 2 eval" in r.stdout and "step 4 eval" in r.stdout
    sc = _read_scalars(str(ck / "msdn_ev"))
    for step in (2, 4):
        for k in OM.METRICS:
            assert (step, f"eval/fine/{k}") in sc and (step, f"eval/coarse/{k}") in sc, (step, k)
    out = tmp_path / "final.json"
    _run("ann3depth_b200.evaluate", "nyu", "--model", "msdn", "--ckptdir", str(ck), "--id", "ev", "--batchsize", "2",
         "--datadir", str(tmp_path), "--json", str(out))
    res = json.loads(out.read_text())
    assert res["global_step"] == 4
    for name in ("fine", "coarse"):
        for k in OM.METRICS:
            assert sc[(4, f"eval/{name}/{k}")] == pytest.approx(res["metrics"][name][k], **_tol(k)), (name, k)
