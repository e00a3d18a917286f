"""Training-time augmentation on the CPU: the oracle's transform contract (identity, known answers), the parameter draw,
the `Augment` config, the `--augment` flag and the C layout of `a3d_augment_desc`."""
import ctypes
import math
import os
import subprocess

import numpy as np
import pytest
import torch

from oracle import augment as OA
from oracle import tf1_ops

SHAPES = [((480, 640, 3), (228, 304)), ((480, 640, 1), (55, 74)), ((55, 73, 1), (55, 74)), ((480, 640, 3), (240, 320))]
EIGEN = dict(scale_lo=1.0, scale_hi=1.5, max_rotation_deg=5.0, crop_fraction=0.95, flip_prob=0.5, color_lo=0.8,
             color_hi=1.2, aspect=0.75)


@pytest.mark.parametrize("dtype", [torch.float32, torch.float64])
@pytest.mark.parametrize("src,dst", SHAPES)
def test_identity_equals_tf1_resize(src, dst, dtype):
    g = torch.Generator().manual_seed(0)
    x = torch.rand(2, *src, generator=g, dtype=torch.float64).to(dtype)
    ref = tf1_ops.resize_bilinear_tf1(x, *dst)
    mode = "color" if src[-1] == 3 else "depth"
    got = OA.resize_affine_tf1(x, *dst, OA.identity_params(2), mode)
    assert torch.equal(got, ref)


def _ramp(h, w, a, b, g):
    yy, xx = torch.meshgrid(torch.arange(h, dtype=torch.float64), torch.arange(w, dtype=torch.float64), indexing="ij")
    return (a * xx + b * yy + g).view(1, h, w, 1)


@pytest.mark.parametrize("src,dst", [((480, 640), (228, 304)), ((55, 73), (55, 74))])
def test_linear_ramp_maps_to_ramp_at_T(src, dst):
    h, w = src
    params = torch.stack([torch.tensor(OA.params_from(1.3, 4.0, 0.52, 0.47, True, (1.0, 1.0, 1.0), 0.95)),
                          torch.tensor(OA.params_from(1.0, -5.0, 0.5, 0.5, False, (1.0, 1.0, 1.0), 0.95))])
    x = _ramp(h, w, 0.37, -1.25, 3.0).expand(2, h, w, 1).contiguous()
    got = OA.resize_affine_tf1(x, *dst, params, "color")[..., 0]
    xs, ys = OA.source_coords(params, h, w, *dst)
    inside = (xs >= 0) & (xs <= w - 1) & (ys >= 0) & (ys <= h - 1)
    assert inside.float().mean() > 0.9
    want = 0.37 * xs + -1.25 * ys + 3.0
    assert float((got - want)[inside].abs().max()) < 1e-12


def test_two_flips_are_identity():
    """The flip is p_x -> 1 - p_x.  On the TF1 legacy grid (position = index * W/OW, no half-pixel offset) that maps
    column ox to W - ox, so column 0 reads the clamped border column W - 1 and the round trip is exact elsewhere."""
    flip = torch.tensor(OA.params_from(1.0, 0.0, 0.5, 0.5, True, (1.0, 1.0, 1.0), 1.0)).view(1, -1)
    m = flip[0, :6].view(2, 3)
    lin, off = m[:, :2], m[:, 2]
    assert torch.equal(lin @ lin, torch.eye(2, dtype=torch.float64)) and torch.equal(lin @ off + off, torch.zeros(2, dtype=torch.float64))
    g = torch.Generator().manual_seed(1)
    x = torch.rand(1, 48, 64, 3, generator=g, dtype=torch.float64)
    once = OA.resize_affine_tf1(x, 48, 64, flip, "color")
    assert torch.equal(once[:, :, 1:], x[:, :, 1:].flip(2))
    assert torch.equal(once[:, :, 0], x[:, :, 63])
    twice = OA.resize_affine_tf1(once, 48, 64, flip, "color")
    assert torch.equal(twice[:, :, 1:], x[:, :, 1:])


def test_constant_image_and_depth():
    params = torch.tensor(OA.params_from(1.4, -3.0, 0.45, 0.55, True, (0.8, 1.1, 1.2), 0.95)).view(1, -1)
    img = torch.full((1, 480, 640, 3), 0.6, dtype=torch.float64)
    got = OA.resize_affine_tf1(img, 228, 304, params, "color")
    want = 0.6 * torch.tensor([0.8, 1.1, 1.2], dtype=torch.float64)
    assert float((got - want).abs().max()) < 1e-15
    dep = torch.full((1, 55, 73, 1), 2.5, dtype=torch.float64)
    got = OA.resize_affine_tf1(dep, 55, 74, params, "depth")
    assert float((got - 2.5 / 1.4).abs().max()) < 1e-15


def test_draw_ranges_flip_rate_and_determinism():
    n = 100_000
    rows = []
    B = 1000
    for counter in range(n // B):
        rows.append(OA.draw(EIGEN, B, seed=7, counter=counter).numpy())
    p = np.concatenate(rows)
    s, th, fl = p[:, OA.SCALE], p[:, OA.THETA], p[:, OA.FLIP]
    assert s.min() >= 1.0 and s.max() <= 1.5
    assert th.min() >= -5.0 and th.max() <= 5.0
    half = 0.5 * (1 - 0.95 / s)
    assert np.all(np.abs(p[:, OA.CX] - 0.5) <= half + 1e-15) and np.all(np.abs(p[:, OA.CY] - 0.5) <= half + 1e-15)
    col = p[:, OA.COLOR:OA.COLOR + 3]
    assert col.min() >= 0.8 and col.max() <= 1.2
    assert set(np.unique(fl)) == {0.0, 1.0}
    assert abs(fl.mean() - 0.5) < 4 * math.sqrt(0.25 / n)
    assert np.allclose(p[:, OA.INV_SCALE] * s, 1.0)
    assert np.all(p[:, OA.CROP] == np.float32(0.95))
    # the unrotated window stays in the frame: T of the four corners of the unit square, theta = 0
    a = OA.draw(EIGEN, 4, seed=3, counter=11)
    assert torch.equal(a, OA.draw(EIGEN, 4, seed=3, counter=11))
    assert not torch.equal(a, OA.draw(EIGEN, 4, seed=3, counter=12))
    assert not torch.equal(a, OA.draw(EIGEN, 4, seed=4, counter=11))
    assert not torch.equal(a[0], a[1])


def test_window_inside_frame_without_rotation():
    r = dict(EIGEN, max_rotation_deg=0.0)
    p = OA.draw(r, 64, seed=5, counter=0)
    xs, ys = OA.source_coords(p, 480, 640, 228, 304)
    assert float(xs.min()) >= -1e-9 and float(xs.max()) <= 640 and float(ys.min()) >= -1e-9 and float(ys.max()) <= 480


def test_augment_config_validation():
    from ann3depth_b200.augment import Augment, from_flag
    a = Augment.eigen_nyu()
    assert (a.scale_lo, a.scale_hi, a.max_rotation_deg, a.crop_fraction, a.flip_prob, a.color_lo, a.color_hi) == \
        (1.0, 1.5, 5.0, 0.95, 0.5, 0.8, 1.2)
    assert a.crop_fraction == pytest.approx(304 / 320)
    for bad in (dict(scale_lo=0.0), dict(scale_lo=1.2, scale_hi=1.1), dict(crop_fraction=0.0),
                dict(crop_fraction=1.01), dict(flip_prob=-0.1), dict(flip_prob=1.5), dict(color_lo=1.3, color_hi=1.2),
                dict(max_rotation_deg=-1.0), dict(aspect=0.0), dict(scale_hi=float("nan"))):
        with pytest.raises(ValueError):
            Augment(**bad)
    d = a.desc()
    assert d.scale_hi == 1.5 and d.flip_prob == 0.5 and d.aspect == 0.75
    assert from_flag("none") is None and from_flag("eigen") == a
    with pytest.raises(ValueError):
        from_flag("strong")


def test_augment_flag():
    from ann3depth_b200 import ann3depth
    assert ann3depth.parse_args([]).augment == "none"
    assert ann3depth.parse_args(["nyu", "--augment", "eigen"]).augment == "eigen"
    with pytest.raises(SystemExit):
        ann3depth.parse_args(["--augment", "bogus"])


def test_augment_desc_layout_matches_header(repo_root, tmp_path):
    """The ctypes mirror of a3d_augment_desc and the packed-row constants must match include/a3d.h."""
    from ann3depth_b200 import _lib
    fields = [n for n, _ in _lib.AugmentDesc._fields_]
    consts = ["A3D_AUG_PARAMS", "A3D_AUG_M00", "A3D_AUG_M12", "A3D_AUG_COLOR", "A3D_AUG_INV_SCALE", "A3D_AUG_SCALE",
              "A3D_AUG_THETA", "A3D_AUG_FLIP", "A3D_AUG_CX", "A3D_AUG_CY", "A3D_AUG_CROP", "A3D_AUG_VALUE_COLOR",
              "A3D_AUG_VALUE_DEPTH", "A3D_U8"]
    src = tmp_path / "layout.c"
    src.write_text("#include <stdio.h>\n#include <stddef.h>\n#include \"a3d.h\"\nint main(void) {\n"
                   "  printf(\"%zu\\n\", sizeof(a3d_augment_desc));\n" +
                   "".join(f"  printf(\"%zu\\n\", offsetof(a3d_augment_desc, {f}));\n" for f in fields) +
                   "".join(f"  printf(\"%d\\n\", (int){c});\n" for c in consts) + "  return 0;\n}\n")
    exe = tmp_path / "layout"
    subprocess.run(["gcc", "-I", os.path.join(repo_root, "include"), "-o", str(exe), str(src)], check=True)
    out = [int(x) for x in subprocess.run([str(exe)], check=True, capture_output=True, text=True).stdout.split()]
    nf = len(fields)
    assert out[0] == ctypes.sizeof(_lib.AugmentDesc)
    assert out[1:1 + nf] == [getattr(_lib.AugmentDesc, f).offset for f in fields]
    want = [_lib.AUG_PARAMS, OA.M00, OA.M12, OA.COLOR, OA.INV_SCALE, OA.SCALE, OA.THETA, OA.FLIP, OA.CX, OA.CY, OA.CROP,
            _lib.AUG_VALUE_COLOR, _lib.AUG_VALUE_DEPTH, _lib.A3D_U8]
    assert out[1 + nf:] == want
    assert OA.NPARAMS == _lib.AUG_PARAMS
