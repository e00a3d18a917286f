"""Every autotuner candidate of the tcgen05 GEMMs and convolutions, at the shapes the models tune, against an exact
reference.

`autotune()` (tc_gemm.cu) times every candidate configuration of a shape on its first eager launch and the CUDA graphs
replay the winner, so any candidate can ship on the day it happens to be fastest.  Here the models run once in a
subprocess with an empty `A3D_TUNE_CACHE` file, which then lists every tuned key (16 ints), its candidate count and the
choice.  Each key is rebuilt into a call and run once per candidate through `A3D_TUNE_PICK`.

The operands are sparse small integers (bf16, or E4M3 codes with power-of-two scales), with every reduction bounded by
2^24, so every float32 accumulation order is exact, split-K atomics included.  Outputs are therefore compared bit for
bit (up to the sign of zero) with a float64 reference rounded to integers: f32 outputs exactly, bf16 outputs as the
round-to-nearest-even of the exact value, plus bias, ReLU, the dropout mask, the pool-fused max and its first arg-max,
and the untouched channels between K and ldy.
"""
import json
import math
import os
import re
import subprocess
import sys
import tempfile

import pytest
import torch
import torch.nn.functional as F

if torch.cuda.is_available():
    import ctypes as C

    from ann3depth_b200 import _lib as L
    from ann3depth_b200 import ops

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
DEV = "cuda:0"
L_F32, L_BF16 = 0, 1                   # include/a3d.h A3D_F32 / A3D_BF16 (the key stores the code)
KINDS = {1: "conv wgrad", 2: "conv fwd", 3: "dense fwd", 4: "dense dgrad", 5: "pool-fused conv fwd",
         6: "fp8 conv fwd", 7: "fp8 pool-fused conv fwd", 8: "fp8 dense fwd"}
CONV_KINDS = (1, 2, 5, 6, 7)
SENTINEL = -1.0e30                     # never a result: the operands keep every output below 2^24
IDX_SENTINEL = 9


# ----------------------------------------------------------------------------- tuner keys (tc_gemm.cu)
def decode(key):
    """A tuner key (16 ints) -> the arguments of the call that produces it."""
    k = [int(v) for v in key]
    kind = k[0]
    if kind in CONV_KINDS:
        a = dict(zip(("N", "H", "W", "C", "K", "R", "S", "sh", "sw", "pt", "pl", "P", "Q"), k[1:14]))
        a.update(kind=kind, ldy=k[14], dil=0, pp=0)
        if kind == 1:                                  # d->dil_w * 4096 + d->pix_pitch
            a.update(dil=k[15] // 4096, pp=k[15] % 4096)
        elif kind == 5:                                # ldy + 4096 dil_w + 65536 pix_pitch, idx requested
            a.update(ldy=k[14] % 4096, dil=k[14] // 4096 % 16, pp=k[14] // 65536, idx=bool(k[15]))
        elif kind in (2, 6):                           # y_dtype * 2 + can_split (+ 4: output not TMA-stored, kind 2)
            a.update(y_f32=(k[15] >> 1 & 1) == L_F32, can_split=bool(k[15] & 1), out_tma=not (k[15] & 4))
        return a
    if kind == 3:
        return dict(kind=3, M=k[1], N=k[2], K=k[3], ldx=k[4], y_f32=k[5] == L_F32, flags=k[6], mask=bool(k[7]),
                    s_ok=bool(k[8]))
    if kind == 4:
        return dict(kind=4, M=k[1], N=k[2], K=k[3], lddy=k[4], s_ok=bool(k[5]))
    if kind == 8:
        return dict(kind=8, M=k[1], N=k[2], K=k[3], ldx=k[4], y_f32=k[5] == L_F32, flags=k[6])
    raise ValueError(f"unknown tuner kind {kind}")


def encode(a):
    """Inverse of decode()."""
    kind = a["kind"]
    k = [kind] + [0] * 15
    if kind in CONV_KINDS:
        k[1:14] = [a[n] for n in ("N", "H", "W", "C", "K", "R", "S", "sh", "sw", "pt", "pl", "P", "Q")]
        k[14] = a["ldy"]
        if kind == 1:
            k[15] = a["dil"] * 4096 + a["pp"]
        elif kind == 5:
            k[14] = a["ldy"] + 4096 * a["dil"] + 65536 * a["pp"]
            k[15] = int(a["idx"])
        elif kind in (2, 6):
            k[15] = (L_F32 if a["y_f32"] else L_BF16) * 2 + int(a["can_split"]) + (0 if a["out_tma"] else 4)
    elif kind == 3:
        k[1:9] = [a["M"], a["N"], a["K"], a["ldx"], L_F32 if a["y_f32"] else L_BF16, a["flags"], int(a["mask"]),
                  int(a["s_ok"])]
    elif kind == 4:
        k[1:6] = [a["M"], a["N"], a["K"], a["lddy"], int(a["s_ok"])]
    elif kind == 8:
        k[1:7] = [a["M"], a["N"], a["K"], a["ldx"], L_F32 if a["y_f32"] else L_BF16, a["flags"]]
    return k


def parse_cache(text):
    """A3D_TUNE_CACHE lines -> [(key tuple, ncand, choice)]"""
    out = []
    for line in text.splitlines():
        v = [int(t) for t in line.split()]
        if v:
            assert len(v) == 18, line
            out.append((tuple(v[:16]), v[16], v[17]))
    return out


def output_dims_ok(a):
    """P and Q follow from the input, the filter, the strides and the pads: the far pad is the near one (VALID, or SAME
    with an even total) or one more (SAME, odd total).  A dilated / overlapped view (DCNF's first layer) keeps the Q of
    the convolution it stands for, so there only the bound every tap of the row must respect is checked."""
    def fits(n, pad, f, s, p, dil=1):
        return any(p == (n + pad + far - dil * (f - 1) - 1) // s + 1 for far in (pad, pad + 1))
    rows = fits(a["H"], a["pt"], a["R"], a["sh"], a["P"])
    if a["dil"] > 1 or a["pp"] not in (0, a["C"]):
        return rows and a["pl"] == 0 and (a["Q"] - 1) * a["sw"] + (a["S"] - 1) * max(a["dil"], 1) < a["W"]
    return rows and fits(a["W"], a["pl"], a["S"], a["sw"], a["Q"])


def test_tune_cache_keys_decode():
    """Every line of the recorded MSDN (B = 32) and DCNF (B = 16) tuner caches decodes into call arguments that encode
    back to the same key, with consistent output dims and a choice inside the candidate list."""
    for name, kinds in (("tune_cache_r02.txt", {1, 2, 3, 4, 5}), ("tune_cache_dcnf_r02.txt", {1, 2, 3, 5})):
        with open(os.path.join(ROOT, "profiles", name)) as f:
            entries = parse_cache(f.read())
        assert len(entries) >= 15
        assert {k[0] for k, _, _ in entries} == kinds
        for key, ncand, choice in entries:
            a = decode(key)
            assert encode(a) == list(key), (name, key)
            assert 1 <= ncand and 0 <= choice < ncand, (name, key)
            if key[0] in CONV_KINDS:
                assert output_dims_ok(a), (name, key)
                assert a["ldy"] >= (64 if key[0] in (5, 7) else a["K"]), (name, key)
            if key[0] == 1 and a["pp"]:
                assert a["C"] % a["pp"] == 0 and a["dil"] > 1, (name, key)
    dcnf_view = decode([1, 16, 150, 190, 64, 256, 6, 2, 1, 1, 0, 0, 145, 185, 256, 16400])
    assert (dcnf_view["dil"], dcnf_view["pp"]) == (4, 16)
    pool = decode([5, 16, 150, 190, 64, 256, 6, 2, 1, 1, 0, 0, 145, 185, 1065024, 1])
    assert (pool["ldy"], pool["dil"], pool["pp"], pool["idx"]) == (64, 4, 16, True)


# ----------------------------------------------------------------------------- the models' inventory
INVENTORY_SCRIPT = r"""
import sys
sys.path.insert(0, sys.argv[1])
import torch
from ann3depth_b200 import models
from ann3depth_b200.init import glorot_params

def msdn(B, train, dtype="bf16"):
    g = torch.Generator().manual_seed(B)
    images = torch.rand(B, 480, 640, 3, generator=g).cuda()
    depths = (torch.rand(B, 55, 73, 1, generator=g) + 0.05).cuda()
    op = models.msdn(images, depths, train=train, dtype=dtype)
    op.net.load_params(glorot_params(1))
    return op

def train(B, use_graph):
    op = msdn(B, True)
    op.run(use_graph=use_graph)           # phase 1 (with the graph: eager warm-up (tunes), capture, replay)
    op.net.global_step = 2000000 // B     # first step of phase 2 (msdn.phase_of)
    op.run(use_graph=use_graph)

train(32, True)
# one batch per batch-dependent GEMM configuration (test_gpu_model_launches.py RECORD_SCRIPT, DESIGN section 2)
for B in (1, 5, 33, 100, 130):
    train(B, False)
for B in (1, 7, 32, 100, 300, 512):       # inference as tools/fp8_infer_bench.py, and the dense tiles past it
    for dtype in ("bf16", "fp8"):
        op = msdn(B, False, dtype)
        op.run()
        del op
for B in (16, 6):
    g = torch.Generator().manual_seed(B)
    images = torch.rand(B, 480, 640, 3, generator=g).cuda()
    depths = (torch.rand(B, 480, 640, 1, generator=g) * 0.95 + 0.05).cuda()
    models.dcnf(images, depths, train=True).run()
    models.dcnf(images, depths, train=False).run()
torch.cuda.synchronize()
"""


def clean_env(**extra):
    """The environment without any A3D_* setting (every tuner default applies), plus `extra`."""
    env = {k: v for k, v in os.environ.items() if not k.startswith("A3D_")}
    env.update(extra)
    return env


@pytest.fixture(scope="module")
def inventory():
    with tempfile.TemporaryDirectory() as tmp:
        cache = os.path.join(tmp, "tune_cache.txt")
        open(cache, "w").close()
        r = subprocess.run([sys.executable, "-c", INVENTORY_SCRIPT, ROOT], env=clean_env(A3D_TUNE_CACHE=cache),
                           capture_output=True, text=True, timeout=1200)
        assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
        with open(cache) as f:
            entries = parse_cache(f.read())
    keys = [k for k, _, _ in entries]
    assert len(keys) == len(set(keys)), "a key was tuned twice in one process"
    return entries


@pytest.fixture(scope="module")
def ctx():
    saved = {k: os.environ.pop(k) for k in list(os.environ) if k.startswith("A3D_") and k != "A3D_LIB"}
    c = ops.Context(0)
    yield c
    torch.cuda.synchronize()
    c.close()
    os.environ.pop("A3D_TUNE_PICK", None)
    os.environ.update(saved)


@pytest.mark.gpu
def test_inventory_covers_every_kind(inventory, capsys):
    by_kind = {}
    for key, ncand, choice in inventory:
        by_kind.setdefault(key[0], []).append((key, ncand, choice))
    with capsys.disabled():
        print(f"\ntuned keys of the MSDN / DCNF training and inference runs: {len(inventory)} keys, "
              f"{sum(n for _, n, _ in inventory)} candidates")
        for kind in sorted(by_kind):
            rows = by_kind[kind]
            print(f"  kind {kind} ({KINDS[kind]}): {len(rows)} keys, {sum(n for _, n, _ in rows)} candidates")
            for key, ncand, choice in rows:
                print(f"    {' '.join(map(str, key))}  ncand={ncand} choice={choice}")
    assert set(by_kind) == set(KINDS), sorted(by_kind)
    # at least as many shapes as the recorded batch-32 MSDN and batch-16 DCNF training caches list
    recorded = 0
    for name in ("tune_cache_r02.txt", "tune_cache_dcnf_r02.txt"):
        with open(os.path.join(ROOT, "profiles", name)) as f:
            keys = {k for k, _, _ in parse_cache(f.read())}
        recorded += len(keys)
        with capsys.disabled():
            print(f"  {name}: {len(keys - {k for k, _, _ in inventory})} of its {len(keys)} keys not tuned now")
    assert len(inventory) >= recorded


# ----------------------------------------------------------------------------- exact operands and references
def _ptr(t):
    return None if t is None else C.c_void_p(t.data_ptr())


def _stream():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def int_range(kred, scale2=1):
    """Largest r <= 8 with kred * r^2 * scale2 < 2^24: every partial sum of +-r integer products (times the
    power-of-two scales) is an integer below 2^24, so float32 adds it exactly in any order."""
    return max(1, min(8, int(math.isqrt((2 ** 24 - 1) // (kred * scale2)))))


def sparse_ints(shape, r, g):
    """float64 integers in [-r, r], about half of them zero."""
    v = torch.randint(-r, r + 1, shape, generator=g, device=DEV, dtype=torch.int32).double()
    return v * (torch.rand(shape, generator=g, device=DEV) < 0.55)


def pow2(n, g, lo=0, hi=2):
    return torch.pow(2.0, torch.randint(lo, hi + 1, (n,), generator=g, device=DEV).float())


def exact(t, what):
    """Round a float64 reference of integer operands to integers; it must already be one."""
    r = t.round()
    assert float((t - r).abs().max()) < 1e-6, f"{what}: the float64 reference is not integral"
    return r


def to_fp8(t):
    return t.float().to(torch.float8_e4m3fn)


def conv_input(a, r, g):
    """The input as the kernel reads it: a plain NHWC tensor, or for an overlapped view (pix_pitch < C) a flat buffer whose
    pixel w starts pix_pitch elements after pixel w - 1.  Returns (float64 [N,H,W,C] as read, flat float64 buffer)."""
    N, H, W, Cc, pp = a["N"], a["H"], a["W"], a["C"], a["pp"] or a["C"]
    flat = sparse_ints((N * H * W * pp + Cc - pp,), r, g)
    return flat.as_strided((N, H, W, Cc), (H * W * pp, W * pp, pp, 1)), flat


def _cols(xm, a, n0, n1):
    """im2col rows [(n, p, q)] x [(r, s, c)] of images n0..n1 (float64), taps dil_w pixels apart."""
    R, S, sh, sw, pt, pl, P, Q = (a[n] for n in ("R", "S", "sh", "sw", "pt", "pl", "P", "Q"))
    dil = max(a["dil"], 1)
    x = xm[n0:n1].permute(0, 3, 1, 2)
    hn, wn = (P - 1) * sh + R, (Q - 1) * sw + (S - 1) * dil + 1
    x = F.pad(x, (pl, wn - a["W"] - pl, pt, hn - a["H"] - pt))       # negative = crop
    cols = F.unfold(x, (R, S), dilation=(1, dil), stride=(sh, sw))     # [n, C*R*S, P*Q]
    n = n1 - n0
    return cols.view(n, a["C"], R, S, P * Q).permute(0, 4, 2, 3, 1).reshape(n * P * Q, R * S * a["C"])


def _chunks(a):
    per = max(1, (1 << 27) // (a["P"] * a["Q"] * a["R"] * a["S"] * a["C"]))
    return [(n0, min(a["N"], n0 + per)) for n0 in range(0, a["N"], per)]


def conv_ref(xm, w, a):
    """[N*P*Q, K] = conv(x, w) in float64, w [K, R, S, C]"""
    wm = w.reshape(a["K"], -1).t()
    return exact(torch.cat([_cols(xm, a, n0, n1) @ wm for n0, n1 in _chunks(a)]), "conv")


def wgrad_ref(xm, dy, a):
    """[K, R*S*C] = dy^T im2col(x) in float64, dy [N*P*Q, K]"""
    PQ = a["P"] * a["Q"]
    dw = torch.zeros(a["K"], a["R"] * a["S"] * a["C"], dtype=torch.float64, device=DEV)
    for n0, n1 in _chunks(a):
        dw += dy[n0 * PQ:n1 * PQ].t() @ _cols(xm, a, n0, n1)
    return exact(dw, "wgrad")


def pool_ref(v, bias, relu):
    """v [rows, 256] exact, the four window positions in groups of 64 columns: (max + bias, ReLU) and the first arg-max"""
    g4 = v.view(-1, 4, 64)
    m, idx = g4[:, 0].clone(), torch.zeros_like(g4[:, 0], dtype=torch.uint8)
    for j in (1, 2, 3):
        gt = g4[:, j] > m                                  # strict: the FIRST maximum wins
        m = torch.where(gt, g4[:, j], m)
        idx[gt] = j
    m = m + bias
    return (m.clamp(min=0) if relu else m), idx


def cast(v, f32):
    return v.float() if f32 else v.float().to(torch.bfloat16)


def filled(shape, dtype, value=SENTINEL, offset=0):
    """A sentinel-filled output, `offset` elements past a 256-byte aligned allocation."""
    n = math.prod(shape)
    buf = torch.full((n + 64,), value, dtype=dtype, device=DEV)
    return buf[offset:offset + n].view(shape)


def untouched(t):
    """every element still holds the sentinel filled() wrote"""
    return t.numel() == 0 or bool((t == torch.full((), SENTINEL, dtype=t.dtype, device=DEV)).all())


def bits(t):
    t = t + 0                                              # -0 -> +0: the sign of an exact zero is not a result
    return t.view(torch.int32 if t.element_size() == 4 else torch.int16)


def mismatch(got, exp, what):
    """None if got == exp bit for bit (up to the sign of zero), else a description of the first difference."""
    got, exp = got.reshape(exp.shape), exp
    if got.dtype == exp.dtype and torch.equal(bits(got), bits(exp)):
        return None
    bad = (bits(got) != bits(exp)) if got.dtype == exp.dtype else torch.ones_like(exp, dtype=torch.bool)
    i = tuple(int(v) for v in bad.nonzero()[0])
    return f"{what}: {int(bad.sum())} of {exp.numel()} differ, first at {i}: got {float(got[i])} expected {float(exp[i])}"


class Case:
    """One tuner key rebuilt into a call with exact operands.  `calls` maps a variant name to a function that runs the call
    (with whatever A3D_TUNE_PICK is set) and returns a list of mismatch descriptions (empty when everything is exact)."""

    def __init__(self, ctx, key, seed=0):
        self.ctx, self.key, self.a = ctx, tuple(key), decode(key)
        g = torch.Generator(device=DEV).manual_seed(1000 + seed)
        self.calls = {}
        getattr(self, f"_kind{key[0]}")(g)

    # -- conv wgrad: dw (starts as NaN garbage) = dy^T im2col(x); dy rows carry ldy - K channels that are never read
    def _kind1(self, g):
        a, ctx = self.a, self.ctx
        r = int_range(a["N"] * a["P"] * a["Q"])
        xm, flat = conv_input(a, r, g)
        rows = a["N"] * a["P"] * a["Q"]
        dyf = sparse_ints((rows, a["ldy"]), r, g)
        dyf[:, a["K"]:] = 99.0
        x, dy = flat.to(torch.bfloat16), dyf.to(torch.bfloat16)
        exp = wgrad_ref(xm, dyf[:, :a["K"]], a).float()
        d = self.desc()

        def call(offset):
            def run():
                dw = filled((a["K"], a["R"] * a["S"] * a["C"]), torch.float32, float("nan"), offset)
                ctx.conv2d_wgrad(d, x, dy, dw=dw)
                return [m for m in [mismatch(dw, exp, "dw")] if m]
            return run
        self.calls = {"recorded": call(0), "offset dw": call(1)}

    def desc(self):
        a = self.a
        d = ops.conv_desc(a["N"], a["H"], a["W"], a["C"], a["K"], a["R"], a["S"], (a["sh"], a["sw"]), (a["pt"], a["pl"]),
                          ldy=a["ldy"])
        d.P, d.Q, d.dil_w, d.pix_pitch = a["P"], a["Q"], a["dil"], a["pp"]
        return d

    def _conv_common(self, g, fp8):
        a = self.a
        kred = a["R"] * a["S"] * a["C"]
        r = int_range(kred, 16 if fp8 else 1)
        xm, flat = conv_input(a, r, g)
        w = sparse_ints((a["K"], a["R"], a["S"], a["C"]), r, g)
        bias = torch.randint(-40, 41, (a["K"] if a["kind"] in (2, 6) else 64,), generator=g, device=DEV).float()
        S = conv_ref(xm, w, a)                                  # [N*P*Q, K]
        if fp8:
            xs, ws = pow2(a["N"], g), pow2(a["K"], g)
            S = S * xs.double().repeat_interleave(a["P"] * a["Q"])[:, None] * ws.double()[None, :]
            return dict(x=to_fp8(flat), w=to_fp8(w), xs=xs, ws=ws, bias=bias, S=S)
        return dict(x=flat.to(torch.bfloat16), w=w.to(torch.bfloat16), bias=bias, S=S)

    # -- conv fwd (bf16 / E4M3): y = act(S + bias) into [N,P,Q,ldy]; split-K candidates only with the key's workspace
    def _conv_fwd(self, g, fp8):
        a, ctx = self.a, self.ctx
        o = self._conv_common(g, fp8)
        rows, K, ldy, f32 = a["N"] * a["P"] * a["Q"], a["K"], a["ldy"], a["y_f32"]
        ws = torch.empty(rows * K * 4, dtype=torch.uint8, device=DEV) if a["can_split"] else None
        d = self.desc()
        v = o["S"] + o["bias"].double()
        exp = {False: cast(v, f32), True: cast(v.clamp(min=0), f32)}
        dtype = torch.float32 if f32 else torch.bfloat16
        code = L.A3D_F32 if f32 else L.A3D_BF16

        def call(offset, relu):
            def run():
                y = filled((a["N"], a["P"], a["Q"], ldy), dtype, offset=offset)
                flags = L.EPI_RELU if relu else 0
                if fp8:
                    rc = ctx.lib.a3d_conv2d_fwd_fp8(ctx.h, C.byref(d), _ptr(o["x"]), _ptr(o["xs"]), _ptr(o["w"]),
                                                    _ptr(o["ws"]), _ptr(o["bias"]), _ptr(y), code, flags, _ptr(ws),
                                                    0 if ws is None else ws.numel(), _stream())
                else:
                    rc = ctx.lib.a3d_conv2d_fwd(ctx.h, C.byref(d), _ptr(o["x"]), _ptr(o["w"]), _ptr(o["bias"]), _ptr(y),
                                                code, flags, _ptr(ws), 0 if ws is None else ws.numel(), _stream())
                L.check(rc, "conv2d_fwd_fp8" if fp8 else "conv2d_fwd")
                y2 = y.view(rows, ldy)
                out = [mismatch(y2[:, :K], exp[relu], "y"),
                       None if untouched(y2[:, K:]) else "y: channels K..ldy overwritten"]
                return [m for m in out if m]
            return run
        # one element off alignment: the register epilogue instead of the TMA store (kind 2 keys record which one)
        off = 0 if a.get("out_tma", True) else 1
        self.calls = {"recorded": call(off, False), ("aligned y, relu" if off else "offset y, relu"): call(1 - off, True)}

    def _kind2(self, g):
        self._conv_fwd(g, False)

    def _kind6(self, g):
        self._conv_fwd(g, True)

    # -- pool-fused conv fwd: y [N,P,Q,ldy] = act(max over the 4 groups of 64 columns + bias), idx = first arg-max
    def _conv_pool(self, g, fp8):
        a, ctx = self.a, self.ctx
        o = self._conv_common(g, fp8)
        rows, ldy = a["N"] * a["P"] * a["Q"], a["ldy"]
        want_idx = (not fp8) and a.get("idx", False)
        refs = {relu: pool_ref(o["S"], o["bias"].double(), relu) for relu in (False, True)}
        d = self.desc()

        def call(relu):
            def run():
                y = filled((a["N"], a["P"], a["Q"], ldy), torch.bfloat16)
                if fp8:
                    ctx.conv2d_pool4_fwd_fp8(d, o["x"], o["xs"], o["w"], o["ws"], o["bias"], relu=relu, out=y)
                    idx = None
                else:
                    idx = torch.full((a["N"], a["P"], a["Q"], 64), IDX_SENTINEL, dtype=torch.uint8, device=DEV) \
                        if want_idx else None
                    ctx.conv2d_pool4_fwd(d, o["x"], o["w"], o["bias"], relu=relu, out=y, idx=idx)
                m, gi = refs[relu]
                y2 = y.view(rows, ldy)
                out = [mismatch(y2[:, :64], m.float().to(torch.bfloat16), "pooled y"),
                       None if untouched(y2[:, 64:]) else "y: channels 64..ldy overwritten"]
                if idx is not None and not torch.equal(idx.view(rows, 64), gi):
                    bad = idx.view(rows, 64) != gi
                    out.append(f"idx: {int(bad.sum())} of {gi.numel()} are not the first arg-max")
                return [m for m in out if m]
            return run
        self.calls = {"relu": call(True), "no relu": call(False)}

    def _kind5(self, g):
        self._conv_pool(g, False)

    def _kind7(self, g):
        self._conv_pool(g, True)

    # -- dense fwd (bf16): y = act(x w^T + bias) * mask * 2 (drop rate 0.5); x rows carry ldx - K unread columns
    def _kind3(self, g):
        a, ctx = self.a, self.ctx
        M, N, K, ldx, f32, flags = a["M"], a["N"], a["K"], a["ldx"], a["y_f32"], a["flags"]
        assert flags & ~L.EPI_RELU == 0, f"key {self.key}: only ReLU has an exact reference"
        r = int_range(K)
        xf = sparse_ints((M, ldx), r, g)
        xf[:, K:] = 99.0
        w = sparse_ints((N, K), r, g)
        bias = torch.randint(-40, 41, (N,), generator=g, device=DEV).float()
        mask = (torch.rand(M, N, generator=g, device=DEV) < 0.5).to(torch.uint8) if a["mask"] else None
        v = exact(xf[:, :K] @ w.t(), "dense") + bias.double()
        if flags & L.EPI_RELU:
            v = v.clamp(min=0)
        if mask is not None:
            v = v * mask.double() * 2
        exp = cast(v, f32)
        x, wb = xf.to(torch.bfloat16), w.to(torch.bfloat16)

        def run():
            y = filled((M, N), torch.float32 if f32 else torch.bfloat16)
            ctx.dense_fwd(x, wb, bias, flags=flags, keep_mask=mask, drop_rate=0.5 if mask is not None else 0.0, out=y)
            return [m for m in [mismatch(y, exp, "y")] if m]
        self.calls = {"recorded": run}

    # -- dense dgrad: dx (bf16) = dy[:, :N] w; dy rows carry lddy - N unread columns
    def _kind4(self, g):
        a, ctx = self.a, self.ctx
        M, N, K, lddy = a["M"], a["N"], a["K"], a["lddy"]
        r = int_range(N)
        dyf = sparse_ints((M, lddy), r, g)
        dyf[:, N:] = 99.0
        w = sparse_ints((N, K), r, g)
        exp = cast(exact(dyf[:, :N] @ w, "dense dgrad"), False)
        dy, wb = dyf.to(torch.bfloat16), w.to(torch.bfloat16)

        def run():
            dx = filled((M, K), torch.bfloat16)
            ctx.dense_dgrad(dy, wb, out=dx)
            return [m for m in [mismatch(dx, exp, "dx")] if m]
        self.calls = {"recorded": run}

    # -- fp8 dense fwd: y = act(S * x_scale[m] * w_scale[n] + bias)
    def _kind8(self, g):
        a, ctx = self.a, self.ctx
        M, N, K, ldx, f32, flags = a["M"], a["N"], a["K"], a["ldx"], a["y_f32"], a["flags"]
        assert flags & ~L.EPI_RELU == 0, f"key {self.key}: only ReLU has an exact reference"
        r = int_range(K, 16)
        xf = sparse_ints((M, ldx), r, g)
        xf[:, K:] = 8.0
        w = sparse_ints((N, K), r, g)
        xs, ws = pow2(M, g), pow2(N, g)
        bias = torch.randint(-40, 41, (N,), generator=g, device=DEV).float()
        v = exact(xf[:, :K] @ w.t(), "fp8 dense") * xs.double()[:, None] * ws.double()[None, :] + bias.double()
        if flags & L.EPI_RELU:
            v = v.clamp(min=0)
        exp = cast(v, f32)
        xq, wq = to_fp8(xf), to_fp8(w)

        def run():
            y = filled((M, N), torch.float32 if f32 else torch.bfloat16)
            ctx.dense_fwd_fp8(xq[:, :K], xs, wq, ws, bias, flags=flags, out=y)
            return [m for m in [mismatch(y, exp, "y")] if m]
        self.calls = {"recorded": run}


class pick:
    """A3D_TUNE_PICK=i around a block"""

    def __init__(self, i):
        self.i = i

    def __enter__(self):
        os.environ["A3D_TUNE_PICK"] = str(self.i)

    def __exit__(self, *exc):
        os.environ.pop("A3D_TUNE_PICK", None)


PICK_ERROR = re.compile(r"A3D_TUNE_PICK=(\d+) out of range: tuner kind (\d+) has (\d+) candidates")


def candidate_count(run):
    """(kind, number of candidates) of the key a call tunes, from the error of an out-of-range pick"""
    with pick(10 ** 6):
        try:
            run()
        except L.A3DError as e:
            m = PICK_ERROR.search(str(e))
            assert m, str(e)
            return int(m.group(2)), int(m.group(3))
    raise AssertionError("A3D_TUNE_PICK=1000000 did not fail the call")


@pytest.mark.gpu
@pytest.mark.parametrize("kind", sorted(KINDS))
def test_every_candidate_is_exact(ctx, inventory, kind):
    """For every key of `kind` the models tune: each candidate gives the exact result (every variant of the call), and
    the pick one past the last candidate fails naming the kind, the index and the count."""
    entries = [(k, n, c) for k, n, c in inventory if k[0] == kind]
    assert entries, f"the models tune no key of kind {kind}"
    failures, runs = [], 0
    for seed, (key, ncand, choice) in enumerate(entries):
        case = Case(ctx, key, seed)
        for variant, run in case.calls.items():
            where = f"kind {kind} ({KINDS[kind]}) key {' '.join(map(str, key))} [{variant}]"
            try:
                k, n = candidate_count(run)
            except AssertionError as e:
                failures.append(f"{where}: {e}")
                continue
            if variant == "recorded" or kind != 2:
                # the rebuilt call has the recorded key: same kind and candidate list
                if (k, n) != (kind, ncand):
                    failures.append(f"{where}: the rebuilt call tunes kind {k} with {n} candidates, recorded {ncand}")
                    continue
            for i in range(n):
                with pick(i):
                    try:
                        bad = run()
                    except L.A3DError as e:
                        bad = [f"error: {e}"]
                runs += 1
                failures += [f"{where} candidate {i} of {n}: {b}" for b in bad]
            with pick(n):
                try:
                    run()
                    failures.append(f"{where}: A3D_TUNE_PICK={n} (one past the last candidate) did not fail")
                except L.A3DError as e:
                    m = PICK_ERROR.search(str(e))
                    if not (m and m.groups() == (str(n), str(kind), str(n))):
                        failures.append(f"{where}: A3D_TUNE_PICK={n} failed with an unexpected message: {e}")
        del case
        torch.cuda.empty_cache()
    print(f"kind {kind}: {len(entries)} keys, {runs} candidate runs")
    assert not failures, f"{len(failures)} failures:\n" + "\n".join(failures[:40])


# ----------------------------------------------------------------------------- tuning has no side effects
def check_tuning_side_effects(keys):
    """In a process where none of `keys` has been tuned: the first call of each key tunes (running every candidate on the
    same, sentinel-filled outputs) and must still return exactly the reference, and a second call the identical result.
    The conv fwd / wgrad keys are then called with an output one element off alignment (the register epilogue) after
    tuning on an aligned one."""
    c = ops.Context(0)
    failures = []
    for seed, key in enumerate(keys):
        case = Case(c, key, seed)
        for variant, run in case.calls.items():
            for attempt in ("first (tuning) call", "second call"):
                try:
                    bad = run()
                except L.A3DError as e:
                    bad = [f"error: {e}"]
                failures += [f"kind {key[0]} key {' '.join(map(str, key))} [{variant}] {attempt}: {b}" for b in bad]
    torch.cuda.synchronize()
    c.close()
    assert not failures, "\n".join(failures)


def _smallest(entries, kind):
    def work(k):
        return math.prod(max(v, 1) for v in k[1:8])
    return min((k for k, _, _ in entries if k[0] == kind), key=work)


@pytest.mark.gpu
def test_tuning_has_no_side_effects(inventory):
    keys = [list(_smallest(inventory, kind)) for kind in sorted(KINDS)]
    code = ("import json, sys; sys.path[:0] = [sys.argv[1], sys.argv[2]]; import test_gpu_tuner_candidates as T; "
            "T.check_tuning_side_effects(json.loads(sys.argv[3]))")
    r = subprocess.run([sys.executable, "-c", code, ROOT, os.path.join(ROOT, "tests"), json.dumps(keys)],
                       env=clean_env(), capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-5000:]


@pytest.mark.gpu
def test_pick_out_of_range_fails_at_single_candidate_sites(ctx):
    """A3D_TUNE_PICK past the end fails the call instead of running candidate 0 -- also where the candidate list is
    short: the FP8 pool-fused forward has two candidates, a dense forward key at least one."""
    key = [7, 1, 10, 12, 64, 256, 3, 3, 1, 1, 0, 0, 8, 10, 64, 0]
    case = Case(ctx, key)
    run = case.calls["relu"]
    assert candidate_count(run) == (7, 2)
    for i in (0, 1):
        with pick(i):
            assert run() == []
    with pick(2), pytest.raises(L.A3DError, match="A3D_TUNE_PICK=2 out of range: tuner kind 7 has 2 candidates"):
        run()
    with pick(-1), pytest.raises(L.A3DError, match="out of range"):
        run()
