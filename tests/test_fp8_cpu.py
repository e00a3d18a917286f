"""CPU tests of the FP8 inference mode's numerics contract (oracle/fp8.py): the E4M3 quantiser on known answers, the
scale formula against a plain float32 restatement, an exactly representable MSDN forward, per-image batch invariance and
the evaluate command's --dtype flag."""
import numpy as np
import torch

from ann3depth_b200.evaluate import parse_args
from oracle import fp8 as F
from oracle import msdn as OM


def test_e4m3_rounding_known_answers():
    x = torch.tensor([1.0625, 1.1875, 1.125, 448.0, 460.0, 1e6, -1e6, 2.0 ** -9, 2.0 ** -10, 3 * 2.0 ** -10, 0.0, -1.0625])
    got = F.e4m3(x).float().tolist()
    # RNE ties (1.0625 -> 1.0, 1.1875 -> 1.25), exact values, saturation at 448, subnormals (2^-10 is a tie between 0
    # and 2^-9 and goes to the even 0; 3 * 2^-10 ties between 2^-9 and 2^-8 and goes to 2^-8)
    assert got == [1.0, 1.25, 1.125, 448.0, 448.0, 448.0, -448.0, 2.0 ** -9, 0.0, 2.0 ** -8, 0.0, -1.0]


def test_quantize_zero_tensor():
    q, s = F.quantize_images(torch.zeros(2, 5, 8))
    assert torch.equal(s, torch.zeros(2)) and torch.equal(q.float(), torch.zeros(2, 5, 8))


def test_scale_formula_matches_float32_restatement():
    g = torch.Generator().manual_seed(0)
    x = (torch.randn(4, 3, 64, generator=g) * torch.tensor([1e-3, 1.0, 37.0, 1e4]).view(4, 1, 1)).to(torch.bfloat16).float()
    q, s = F.quantize_images(x)
    xn = x.numpy().reshape(4, -1).astype(np.float32)
    for b in range(4):
        amax = np.float32(np.abs(xn[b]).max())
        assert s[b].item() == float(np.float32(amax / np.float32(448.0)))
        inv = np.float32(np.float32(448.0) / amax)
        prod = (xn[b] * inv).astype(np.float32)
        ref = F.e4m3(torch.from_numpy(prod)).float().numpy()
        assert np.array_equal(q[b].float().numpy().reshape(-1), ref)
        assert q[b].float().abs().max().item() == 448.0      # the amax element lands on the top code


def test_quantize_rows_is_per_output_channel():
    g = torch.Generator().manual_seed(1)
    k = torch.randn(3, 3, 16, 8, generator=g, dtype=torch.float64)
    w = F.weight(k)
    for co in range(8):
        amax = float(F.bf16_round(k[..., co].float()).abs().max())
        # the largest entry of each channel lands on the top code: 448 * f32(amax / 448) is amax to float32 precision
        assert abs(float(w[..., co].abs().max()) - amax) <= amax * 2.0 ** -23


def _representable_params():
    """Zero kernels except fine/third, power-of-two biases: every storage point holds exactly representable values, so
    the FP8 forward equals the float64 forward bit for bit."""
    p = OM.init_params(1, torch.float64)
    for n in list(p):
        if n.endswith("/kernel") and not n.startswith("fine/third"):
            p[n] = torch.zeros_like(p[n])
        if n.endswith("/bias"):
            c = p[n].numel()
            p[n] = 2.0 ** -(torch.arange(c, dtype=torch.float64) % 3)          # 1, 1/2, 1/4, ...
    p["fine/third/kernel"] = OM.bf16_round(p["fine/third/kernel"])
    return p


def test_oracle_fp8_forward_exact_on_representable_case():
    p = _representable_params()
    g = torch.Generator().manual_seed(2)
    images = torch.rand(1, 240, 320, 3, generator=g, dtype=torch.float64)
    depths = torch.rand(1, 55, 73, 1, generator=g, dtype=torch.float64) + 0.1
    got = F.forward(p, images, depths)
    ref = OM.forward(p, images, depths, None, False)
    assert torch.equal(got["coarse"], ref["coarse"]) and torch.equal(got["fine"], ref["fine"])
    assert float(got["scales"]["c2"][0]) == float(torch.tensor(1.0) / 448.0)      # amax of relu(bias) = 1, float32


def test_oracle_fp8_batch_permutation():
    p = OM.init_params(3, torch.float64, bias_range=0.05)
    g = torch.Generator().manual_seed(4)
    images = torch.rand(2, 240, 320, 3, generator=g, dtype=torch.float64)
    depths = torch.rand(2, 55, 73, 1, generator=g, dtype=torch.float64) + 0.1
    a = F.forward(p, images, depths)
    b = F.forward(p, images.flip(0), depths.flip(0))
    assert torch.equal(a["coarse"], b["coarse"].flip(0)) and torch.equal(a["fine"], b["fine"].flip(0))
    for k, s in a["scales"].items():
        assert torch.equal(s, b["scales"][k].flip(0)), k


def test_evaluate_dtype_flag():
    assert parse_args(["nyu"]).dtype == "bf16"
    assert parse_args(["nyu", "--dtype", "fp8"]).dtype == "fp8"
