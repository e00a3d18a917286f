"""Every kernel call the models make, recorded and replayed with exact operands.

A subprocess runs MSDN (bf16, TF32 and 3xTF32; training phases 1 and 2, the sequential step, inference) and DCNF
(training with both pairwise graphs, inference) with every public `ops.Context` method wrapped by a recorder.  Each
outermost call is recorded as its method, its scalars, its `ConvDesc`, `ctx.tf32x3`, and for each tensor the shape,
dtype, strides, `data_ptr() % 256` and which arguments share storage at which relative offsets.  The pointer alignment
matters: the TMA epilogue is chosen from it (DESIGN §4.1).  The calls are deduplicated by that signature.

Every recorded method is either replayed here or excluded with a reason (`EXCLUDED`); an unclassified method fails
`test_inventory_is_classified`.  A replay rebuilds the call's buffers with the recorded geometry (shared storage
included), fills the inputs with values whose results are exact in float32 and compares every output bit for bit with a
float64 reference:

- bf16 and TF32 contractions: sparse integers bounded by `int_range`, so every summation order is exact and the TF32
  conversion (at most 11 significant bits) is the identity.
- 3xTF32 contractions: operands hi + lo with integer hi and lo = +-2^-13, so the TF32 hi/lo split is exact and tie-free;
  the reference is hi.hi + hi.lo + lo.hi (lo.lo is dropped by design) and every partial sum stays on the 2^-13 grid below
  2^11, hence exact.
- Selections (max-pools, routing records, ReluGrad, scatters) use small integers with many ties and zeros, so "the first
  arg-max wins" and "4 = no route when the window max is not positive" are exercised.
- TF-Adam runs with beta1 = beta2 = 0 and m = v = 0: m must be the exact gradient and v its square, bit for bit; w is
  checked within 1 ulp of the float64 step.  The sigmoid epilogue (DCNF dense_1) is the one other inexact result and is
  checked within 1 ulp of its output type.

Bytes of a call's buffers outside its outputs (channels between K and ldy, rows past the end, the rest of a parameter
arena) must not change.
"""
import inspect
import json
import math
import os
import subprocess
import sys
import tempfile

import pytest
import torch
import torch.nn.functional as F

from test_gpu_tuner_candidates import (_chunks, _cols, clean_env, conv_ref, int_range, mismatch, pool_ref, sparse_ints,
                                       wgrad_ref)

if torch.cuda.is_available():
    from ann3depth_b200 import _lib as L
    from ann3depth_b200 import ops
    from oracle import tf1_ops as T

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
DEV = "cuda:0"
SENTINEL = -1.0e30
IDX_SENTINEL = 251
X3_LO = 2.0 ** -13         # the lo part of a 3xTF32 operand
X3_BOUND = 1900.0          # sum |x||w| per output: every partial sum on the 2^-13 grid stays below 2^11

# ----------------------------------------------------------------------------- recording
RECORD_SCRIPT = r"""
import functools, json, sys
sys.path.insert(0, sys.argv[1])
import torch
from ann3depth_b200 import _lib as L, models, ops
from ann3depth_b200.init import glorot_params

out = open(sys.argv[2], "w")
config, depth = [None], [0]


def enc(v, groups):
    if isinstance(v, torch.Tensor):
        gid = groups.setdefault(v.untyped_storage().data_ptr(), len(groups))
        return {"T": list(v.shape), "dt": str(v.dtype)[6:], "st": list(v.stride()), "ptr": v.data_ptr(), "g": gid}
    if isinstance(v, L.ConvDesc):
        return {"D": {f: getattr(v, f) for f, _ in v._fields_}}
    if isinstance(v, (tuple, list)):
        return [enc(x, groups) for x in v]
    if v is None or isinstance(v, (bool, int, float, str)):
        return v
    return {"obj": type(v).__name__}


def tensors(v):
    if isinstance(v, dict) and "T" in v:
        yield v
    elif isinstance(v, list):
        for x in v:
            yield from tensors(x)


def wrap(name, fn):
    @functools.wraps(fn)
    def recorded(self, *a, **k):
        if depth[0] == 0:
            groups = {}
            rec = {"m": name, "a": [enc(x, groups) for x in a], "k": {n: enc(x, groups) for n, x in sorted(k.items())},
                   "x3": bool(self.tf32x3)}
            ts = list(tensors(rec["a"])) + list(tensors(list(rec["k"].values())))
            for g in set(t["g"] for t in ts):
                lo = min(t["ptr"] for t in ts if t["g"] == g)
                for t in ts:
                    if t["g"] == g:
                        t["off"] = t["ptr"] - lo
            for t in ts:
                t["al"] = t.pop("ptr") % 256
            out.write(json.dumps({"config": config[0], "rec": rec}) + "\n")
        depth[0] += 1
        try:
            return fn(self, *a, **k)
        finally:
            depth[0] -= 1
    return recorded


for name, fn in list(vars(ops.Context).items()):
    if callable(fn) and not name.startswith("_") and name not in ("close", "workspace", "conv_ws"):
        setattr(ops.Context, name, wrap(name, fn))


def msdn(label, B, train, dtype="bf16", **kw):
    config[0] = label
    g = torch.Generator().manual_seed(B)
    images = torch.rand(B, 480, 640, 3, generator=g).cuda()
    depths = (torch.rand(B, 55, 73, 1, generator=g) + 0.05).cuda()
    op = models.msdn(images, depths, train=train, dtype=dtype, **kw)
    op.net.load_params(glorot_params(1))
    return op


def train(label, B, dtype="bf16", phases=(1, 2), **kw):
    op = msdn(f"{label} phase 1", B, True, dtype, **kw)
    op.run(use_graph=False)
    if 2 in phases:
        config[0] = f"{label} phase 2"
        op.net.global_step = 2000000 // B                # first step of phase 2 (msdn.phase_of)
        op.run(use_graph=False)
    torch.cuda.synchronize()


def infer(label, B, dtype="bf16"):
    msdn(label, B, False, dtype).run()
    torch.cuda.synchronize()


train("msdn bf16 B=32", 32)
train("msdn bf16 B=32 sequential", 32, phases=(1,), overlap=False, fuse_dense_adam=False)
for B in (1, 32, 512):
    infer(f"msdn bf16 inference B={B}", B)
for dtype in ("tf32", "tf32x3"):
    for B in (2, 32):
        train(f"msdn {dtype} B={B}", B, dtype)
        infer(f"msdn {dtype} inference B={B}", B, dtype)
g = torch.Generator().manual_seed(16)
images = torch.rand(16, 480, 640, 3, generator=g).cuda()
depths = (torch.rand(16, 480, 640, 1, generator=g) * 0.95 + 0.05).cuda()
for label, train_, kw in (("dcnf B=16", True, {}),
                          ("dcnf B=16 grid4", True, dict(graph="grid4", r_nonneg=True, train_pairwise=True, predict="map")),
                          ("dcnf inference B=16", False, {})):
    config[0] = label
    models.dcnf(images, depths, train=train_, **kw).run()
    torch.cuda.synchronize()
out.close()
"""


def signature(rec):
    return json.dumps(rec, sort_keys=True)


def record_inventory():
    """[(sorted config labels, record)] of the distinct calls, and {config: (recorded calls, distinct signatures)}"""
    with tempfile.TemporaryDirectory() as tmp:
        path = os.path.join(tmp, "calls.jsonl")
        r = subprocess.run([sys.executable, "-c", RECORD_SCRIPT, ROOT, path], env=clean_env(), capture_output=True,
                           text=True, timeout=1500)
        assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
        with open(path) as f:
            lines = [json.loads(s) for s in f]
    calls, per_config = {}, {}
    for ln in lines:
        s = signature(ln["rec"])
        calls.setdefault(s, (set(), ln["rec"]))[0].add(ln["config"])
        n, sigs = per_config.setdefault(ln["config"], (0, set()))
        per_config[ln["config"]] = (n + 1, sigs | {s})
    return ([(sorted(c), rec) for c, rec in calls.values()],
            {c: (n, len(sigs)) for c, (n, sigs) in per_config.items()})


@pytest.fixture(scope="module")
def inventory():
    return record_inventory()


@pytest.fixture(scope="module")
def ctx():
    saved = {k: os.environ.pop(k) for k in list(os.environ) if k.startswith("A3D_") and k != "A3D_LIB"}
    c = ops.Context(0)
    yield c
    torch.cuda.synchronize()
    c.close()
    os.environ.update(saved)


# ----------------------------------------------------------------------------- classification
EXCLUDED = {
    "resize_bilinear_tf1": "bilinear interpolation: checked against the TF1 oracle (test_gpu_kernels)",
    "resize_bilinear_tf1_s2d": "interpolation: checked against the TF1 oracle (test_gpu_kernels)",
    "resize_affine_tf1": "augmentation resize: checked against oracle/augment.py (test_gpu_augment)",
    "resize_affine_tf1_s2d": "augmentation resize: checked against oracle/augment.py (test_gpu_augment)",
    "augment_draw": "random draw: checked against oracle/augment.py (test_gpu_augment)",
    "silog_loss": "logarithms: checked against the oracle (test_silog_loss_vs_oracle)",
    "crf": "Cholesky solve: checked against the oracle at 1e-5 (test_crf_vs_oracle)",
    "pairwise_features": "exp() of colour distances: checked against the DCNF oracle (test_gpu_kernels)",
    "tile_means": "divisions by tile areas: checked against the DCNF oracle (test_gpu_kernels)",
    "extract_patches_s2d": "data movement checked against extract_patches (test_gpu_kernels)",
    "image_cells_s2d": "data movement checked against the DCNF oracle (test_gpu_kernels)",
    "conv2d_fwd_fp8": "FP8 GEMM: every tuner candidate is exact in test_gpu_tuner_candidates",
    "conv2d_pool4_fwd_fp8": "FP8 GEMM: every tuner candidate is exact in test_gpu_tuner_candidates",
    "dense_fwd_fp8": "FP8 GEMM: every tuner candidate is exact in test_gpu_tuner_candidates",
    "quantize_rows_e4m3": "quantiser: bit-tested in test_gpu_fp8",
    "quantize_e4m3": "quantiser: bit-tested in test_gpu_fp8",
    "maxpool2x2_quantize_e4m3": "quantiser: bit-tested in test_gpu_fp8",
    "resize_bilinear_tf1_s2d_e4m3": "quantising resize: bit-tested in test_gpu_fp8",
    "stamp": "timeline mark, no arithmetic",
    "increment_i64": "step counter, no arithmetic",
    "bernoulli_mask": "random mask: its rate and independence are tested in test_gpu_parity_full",
    "adam_tf_bf16g": "data parallel only (not recorded on one GPU): test_adam_tf_bf16g_* check it directly",
}


# ----------------------------------------------------------------------------- rebuilding a call
def _tensors(v):
    if isinstance(v, dict) and "T" in v:
        yield v
    elif isinstance(v, list):
        for x in v:
            yield from _tensors(x)


def _int_dtype(esize):
    return {1: torch.uint8, 2: torch.int16, 4: torch.int32, 8: torch.int64}[esize]


def _view(storage, dtype, offset_bytes, shape, stride):
    esize = torch.empty(0, dtype=dtype).element_size()
    assert offset_bytes % esize == 0
    return torch.empty(0, dtype=dtype, device=DEV).set_(storage, offset_bytes // esize, shape, stride)


def desc_dict(d):
    return dict(N=d.N, H=d.H, W=d.W, C=d.C, K=d.K, R=d.R, S=d.S, sh=d.stride_h, sw=d.stride_w, pt=d.pad_t, pl=d.pad_l,
                P=d.P, Q=d.Q, ldy=d.ldy, dil=d.dil_w, pp=d.pix_pitch)


def ulps(got, ref, dtype):
    """|got - ref| in units of the last place of `dtype` at ref (float64 tensors)"""
    mant = {torch.float32: 23, torch.bfloat16: 7}[dtype]
    _, e = torch.frexp(ref)
    unit = torch.ldexp(torch.ones_like(ref), (e - 1 - mant).clamp(min=-126 - mant))
    return ((got - ref).abs() / unit)


class Call:
    """One recorded call rebuilt on fresh buffers: one allocation per storage group, every tensor at its recorded
    offset, strides and pointer alignment.  A replay builder fills the inputs, then declares each output with its
    expected value (`expect`), which fills it with the sentinel first unless it is also an input."""

    def __init__(self, ctx, rec, seed):
        self.ctx, self.rec, self.m = ctx, rec, rec["m"]
        self.g = torch.Generator(device=DEV).manual_seed(seed)
        self.checks, self.marks, self.mirror = [], {}, None
        descs = list(_tensors(rec["a"])) + list(_tensors(list(rec["k"].values())))
        self.bufs = {}
        for gid in sorted(set(t["g"] for t in descs)):
            ts = [t for t in descs if t["g"] == gid]
            need = max(t["off"] + self._extent(t) for t in ts)
            first = min(ts, key=lambda t: t["off"])
            buf = torch.zeros(need + 1024, dtype=torch.uint8, device=DEV)
            start = 256 + (first["al"] - buf.data_ptr()) % 256        # 256 bytes before the first tensor, none touched
            self.bufs[gid] = (buf, start)
        args = [self._mat(v) for v in rec["a"]]
        kw = {k: self._mat(v) for k, v in rec["k"].items()}
        bound = inspect.signature(getattr(ops.Context, self.m)).bind(ctx, *args, **kw)
        bound.apply_defaults()
        self.v = dict(bound.arguments)
        del self.v["self"]
        self.x3 = rec["x3"]
        self.a = desc_dict(self.v["d"]) if isinstance(self.v.get("d"), L.ConvDesc) else None

    @staticmethod
    def _extent(t):
        esize = torch.empty(0, dtype=getattr(torch, t["dt"])).element_size()
        if 0 in t["T"]:
            return 0
        return (sum((n - 1) * s for n, s in zip(t["T"], t["st"])) + 1) * esize

    def _mat(self, v):
        if isinstance(v, dict) and "T" in v:
            buf, start = self.bufs[v["g"]]
            return _view(buf.untyped_storage(), getattr(torch, v["dt"]), start + v["off"], v["T"], v["st"])
        if isinstance(v, dict) and "D" in v:
            d = L.ConvDesc()
            for f, x in v["D"].items():
                setattr(d, f, x)
            return d
        if isinstance(v, list):
            return tuple(self._mat(x) for x in v)
        return v

    # -- views and values
    def flat(self, t, n):
        """n elements from t's first element on, whatever t's own shape"""
        return torch.empty(0, dtype=t.dtype, device=DEV).set_(t.untyped_storage(), t.storage_offset(), (n,), (1,))

    def strided(self, t, shape, stride):
        return torch.empty(0, dtype=t.dtype, device=DEV).set_(t.untyped_storage(), t.storage_offset(), shape, stride)

    def ints(self, shape, r):
        return sparse_ints(shape, r, self.g)

    def nonneg(self, shape, r=3):
        """a ReLU output: small integers >= 0, about half of them zero"""
        return sparse_ints(shape, r, self.g).abs()

    def bits01(self, shape):
        return (torch.rand(shape, generator=self.g, device=DEV) < 0.5).double()

    def uniform(self, shape, lo, hi):
        return torch.rand(shape, generator=self.g, device=DEV, dtype=torch.float64) * (hi - lo) + lo

    def operand(self, shape, kred, x3):
        """(values, parts): parts = (hi, lo) for 3xTF32, else (values, None)"""
        if not x3:
            v = self.ints(shape, int_range(kred))
            return v, (v, None)
        p = min(0.5, math.sqrt(400.0 / kred))
        on = torch.rand(shape, generator=self.g, device=DEV) < p
        hi = torch.where(torch.rand(shape, generator=self.g, device=DEV) < 0.5, 1.0, -1.0).double() * on
        lo = torch.randint(-1, 2, shape, generator=self.g, device=DEV).double() * X3_LO * on
        return hi + lo, (hi, lo)

    def product(self, f, pa, pb, what):
        """f bilinear: f(a, b) for exact operands, hi.hi + hi.lo + lo.hi for 3xTF32 ones (bounded so it is exact)"""
        (ah, al), (bh, bl) = pa, pb
        if al is None:
            return f(ah, bh)
        bound = float(f(ah.abs() + al.abs(), bh.abs() + bl.abs()).max())
        assert bound < X3_BOUND, f"{what}: 3xTF32 operands too dense for an exact reference ({bound})"
        return f(ah, bh) + f(ah, bl) + f(al, bh)

    def put(self, t, vals):
        t.copy_(vals.reshape(t.shape).to(t.dtype))

    # -- outputs
    def expect(self, name, t, exp, prefill=True):
        """t must end up equal to exp (same shape, t's dtype) bit for bit"""
        if prefill:
            t.fill_(IDX_SENTINEL if not t.dtype.is_floating_point else SENTINEL)
        self._mark(t)
        self.checks.append((name, t, exp, None))

    def expect_ulps(self, name, t, ref, n, prefill=True, ftz=False):
        """t within n units in the last place of its dtype of the float64 ref; ftz: a result below the smallest normal
        float32 may also be flushed to zero"""
        if prefill:
            t.fill_(SENTINEL)
        self._mark(t)
        self.checks.append((name, t, ref, (n, ftz)))

    def sentinel_like(self, t):
        return torch.full_like(t, IDX_SENTINEL if not t.dtype.is_floating_point else SENTINEL)

    def _mark(self, t):
        key = t.untyped_storage().data_ptr()
        mark = self.marks.setdefault(key, torch.zeros(t.untyped_storage().nbytes(), dtype=torch.uint8, device=DEV))
        _view(mark.untyped_storage(), _int_dtype(t.element_size()), t.storage_offset() * t.element_size(), t.shape,
              t.stride()).fill_(-1 if t.element_size() > 1 else 255)

    # -- run
    def run(self, overrides=None):
        for k, x in (overrides or {}).items():
            self.v[k] = x
        before = {k: b.clone() for k, (b, _) in self.bufs.items()}
        saved = self.ctx.tf32x3
        self.ctx.tf32x3 = self.x3
        try:
            getattr(self.ctx, self.m)(**self.v)
        except L.A3DError as e:
            return [f"error: {e}"]
        finally:
            self.ctx.tf32x3 = saved
        torch.cuda.synchronize()
        bad = []
        for name, t, exp, n in self.checks:
            if n is None and t.element_size() == 1:       # mismatch() compares 2- and 4-byte words
                diff = (t != exp).nonzero()
                m = None if not len(diff) else f"{name}: {len(diff)} of {t.numel()} differ, first at " \
                    f"{tuple(int(i) for i in diff[0])}: got {int(t[tuple(diff[0])])} expected {int(exp[tuple(diff[0])])}"
            elif n is None:
                m = mismatch(t, exp, name)
            else:
                n, ftz = n
                u = ulps(t.double(), exp, t.dtype)
                if ftz:
                    u = torch.where((exp.abs() < 2.0 ** -126) & (t == 0), 0.0, u)
                worst = float(u.max()) if u.numel() else 0.0
                m = None if worst <= n else \
                    f"{name}: {int((u > n).sum())} of {u.numel()} beyond {n} ulp, worst {worst:.3g} at " \
                    f"{tuple(int(i) for i in (u == u.max()).nonzero()[0])}"
            if m:
                bad.append(m)
        if self.mirror is not None:
            wb, w = self.mirror
            if not torch.equal(wb, w.to(torch.bfloat16)):
                bad.append("w_bf16 is not the bf16 rounding of the updated w")
        for k, (buf, _) in self.bufs.items():
            mark = self.marks.get(buf.untyped_storage().data_ptr())
            changed = buf != before[k]
            if mark is not None:
                changed &= mark == 0
            if bool(changed.any()):
                bad.append(f"wrote {int(changed.sum())} bytes outside its outputs (storage {k}, first at byte "
                           f"{int(changed.nonzero()[0]) - self.bufs[k][1]} from the first tensor)")
        return bad


# ----------------------------------------------------------------------------- references
def conv_x3(xm, w, a):
    """conv_ref without the integrality check (3xTF32 operands are on the 2^-13 grid)"""
    wm = w.reshape(a["K"], -1).t()
    return torch.cat([_cols(xm, a, n0, n1) @ wm for n0, n1 in _chunks(a)])


def conv_any(xm, w, a):
    return conv_ref(xm, w, a) if bool((xm == xm.round()).all() and (w == w.round()).all()) else conv_x3(xm, w, a)


def dgrad_ref(dy, w, a):
    """dx [N,H,W,C] of dy [N,P,Q,K] through w [K,R,S,C]: the transposed convolution, cropped by the pads"""
    assert a["dil"] <= 1 and a["pp"] in (0, a["C"])
    wt = w.permute(0, 3, 1, 2)                                   # [K, C, R, S] = conv_transpose2d's [in, out, kh, kw]
    out = []
    for n0, n1 in _chunks(a):
        full = F.conv_transpose2d(dy[n0:n1].permute(0, 3, 1, 2), wt, stride=(a["sh"], a["sw"]))
        hh, ww = full.shape[2], full.shape[3]
        full = F.pad(full, (0, max(0, a["pl"] + a["W"] - ww), 0, max(0, a["pt"] + a["H"] - hh)))
        out.append(full[:, :, a["pt"]:a["pt"] + a["H"], a["pl"]:a["pl"] + a["W"]].permute(0, 2, 3, 1))
    return torch.cat(out)


def conv_input_view(c, x, a):
    """x as the kernel reads it: pixel w starts pix_pitch elements after pixel w - 1 (C when no overlapped view)"""
    N, H, W, Cc, pp = a["N"], a["H"], a["W"], a["C"], a["pp"] or a["C"]
    return c.flat(x, N * H * W * pp + Cc - pp), (N, H, W, Cc), (H * W * pp, W * pp, pp, 1)


def fill_conv_input(c, x, a, x3):
    flat, shape, stride = conv_input_view(c, x, a)
    v, (h, lo) = c.operand(flat.shape, a["R"] * a["S"] * a["C"], x3)
    c.put(flat, v)
    st = (lambda t: None if t is None else t.as_strided(shape, stride))
    return (st(h), st(lo))


def cast_to(v, t):
    return v.to(t.dtype) if t.dtype != torch.bfloat16 else v.float().to(torch.bfloat16)


def with_columns(c, t, cols, vals):
    """t's expected value: the sentinel everywhere, vals in the first `cols` channels"""
    exp = c.sentinel_like(t)
    exp[..., :cols] = cast_to(vals, t).reshape(exp[..., :cols].shape)
    return exp


# ----------------------------------------------------------------------------- replay builders
def r_conv2d_fwd(c):
    a, v = c.a, c.v
    f32 = v["x"].dtype == torch.float32
    x3 = f32 and c.x3 and a["K"] != 1
    px = fill_conv_input(c, v["x"], a, x3)
    w, pw = c.operand(v["w"].shape, a["R"] * a["S"] * a["C"], x3)
    c.put(v["w"], w)
    S = c.product(lambda xm, wm: conv_any(xm, wm, a), px, pw, "conv")
    if v["bias"] is not None:
        b = torch.randint(-40, 41, v["bias"].shape, generator=c.g, device=DEV).double()
        c.put(v["bias"], b)
        S = S + b
    if v["relu"]:
        S = S.clamp(min=0)
    c.expect("y", v["out"], with_columns(c, v["out"], a["K"], S.view(a["N"], a["P"], a["Q"], a["K"])))


def r_conv2d_pool4_fwd(c):
    a, v = c.a, c.v
    x3 = v["x"].dtype == torch.float32 and c.x3
    px = fill_conv_input(c, v["x"], a, x3)
    w, pw = c.operand(v["w"].shape, a["R"] * a["S"] * a["C"], x3)
    c.put(v["w"], w)
    S = c.product(lambda xm, wm: conv_any(xm, wm, a), px, pw, "pool4 conv")
    b = torch.randint(-40, 41, v["bias"].shape, generator=c.g, device=DEV).double()
    c.put(v["bias"], b)
    m, gi = pool_ref(S, b, v["relu"])
    out = v["out"]
    c.expect("pooled y", out, with_columns(c, out, 64, m.view(*out.shape[:-1], 64)))
    if v["idx"] is not None:
        c.expect("idx", v["idx"], gi.view(v["idx"].shape))


def r_conv2d_dgrad(c):
    a, v = c.a, c.v
    f32 = v["dy"].dtype == torch.float32
    N, P, Q, K, ldy = a["N"], a["P"], a["Q"], a["K"], a["ldy"]
    dyf = c.flat(v["dy"], (N * P * Q - 1) * ldy + K)
    kred = a["R"] * a["S"] * K
    dyv, _ = c.operand(dyf.shape, kred, False)
    c.put(dyf, dyv)
    dy = dyv.as_strided((N, P, Q, K), (P * Q * ldy, Q * ldy, ldy, 1))
    w = c.ints(v["w"].shape, int_range(kred))
    c.put(v["w"], w)
    if v["wflip"] is not None:
        assert not f32
        c.ctx.conv2d_dgrad_prepare(v["d"], v["w"], out=v["wflip"])
    dx = dgrad_ref(dy, w, a)
    if v["relu_src"] is not None:
        src = c.nonneg(v["relu_src"].shape)
        c.put(v["relu_src"], src)
        dx = dx * (src.view(dx.shape) > 0)
    c.expect("dx", v["out"], cast_to(dx, v["out"]).view(v["out"].shape))


def r_conv2d_dgrad_prepare(c):
    a, v = c.a, c.v
    w = c.ints(v["w"].shape, 8)
    c.put(v["w"], w)
    exp = w.view(a["K"], a["R"], a["S"], a["C"]).flip(1, 2).permute(3, 1, 2, 0)      # [C, R, S, K]
    if v["out"] is None:                                   # the first call allocates the filter the later ones refresh
        v["out"] = torch.empty(a["C"], a["R"], a["S"], a["K"], dtype=torch.bfloat16, device=DEV)
    if c.ctx.conv2d_dgrad_prepare(v["d"], v["w"], out=torch.empty_like(v["out"])) is None:
        c.expect("wflip (unused shape)", v["out"], c.sentinel_like(v["out"]))
    else:
        c.expect("wflip", v["out"], cast_to(exp, v["out"]).view(v["out"].shape))


def r_conv2d_wgrad(c):
    a, v = c.a, c.v
    N, P, Q, K, ldy = a["N"], a["P"], a["Q"], a["K"], a["ldy"]
    rows = N * P * Q
    r = int_range(rows)
    flat, shape, stride = conv_input_view(c, v["x"], a)
    xv = c.ints(flat.shape, r)
    c.put(flat, xv)
    dyf = c.flat(v["dy"], (rows - 1) * ldy + K)
    dyv = c.ints(dyf.shape, r)
    c.put(dyf, dyv)
    dy = dyv.as_strided((rows, K), (ldy, 1))
    dw = wgrad_ref(xv.as_strided(shape, stride), dy, a)
    c.expect("dw", v["dw"], dw.float().view(v["dw"].shape))
    if v["db"] is not None:
        c.expect("db", v["db"], dy.sum(0).float().view(v["db"].shape))


def _dense_x(c, x, M, K, ldx, x3, kred):
    xf = c.strided(x, (M, ldx), (ldx, 1))
    xv, px = c.operand((M, ldx), kred, x3)
    c.put(xf, xv)
    return tuple(None if t is None else t[:, :K] for t in px)


def _mask(c, t):
    m = c.bits01(t.shape)
    c.put(t, m)
    return m


def r_dense_fwd(c):
    v = c.v
    x, w = v["x"], v["w"]
    M, (N, K) = x.shape[0], w.shape
    ldx = v["ldx"] or x.shape[1]
    x3 = x.dtype == torch.float32 and c.x3
    px = _dense_x(c, x, M, K, ldx, x3, K)
    wv, pw = c.operand((N, K), K, x3)
    c.put(w, wv)
    y = c.product(lambda p, q: p @ q.t(), px, pw, "dense")
    if v["bias"] is not None:
        b = torch.randint(-40, 41, (N,), generator=c.g, device=DEV).double()
        c.put(v["bias"], b)
        y = y + b
    flags = v["flags"]
    if flags & L.EPI_RELU:
        y = y.clamp(min=0)
    if v["keep_mask"] is not None:
        assert v["drop_rate"] == 0.5
        y = y * _mask(c, v["keep_mask"]).view(M, N) * 2
    if flags & L.EPI_SIGMOID:
        # the one inexact epilogue: expf and a division, within 1 ulp of the output type (outputs below 2^-126, at
        # pre-activations under -87, may be flushed to zero)
        c.expect_ulps("sigmoid y", v["out"], torch.sigmoid(y).view(v["out"].shape), 1, ftz=True)
    else:
        c.expect("y", v["out"], cast_to(y, v["out"]).view(v["out"].shape))


def _dense_dgrad_common(c):
    v = c.v
    dy, w = v["dy"], v["w"]
    M, lddy = dy.shape
    N, K = w.shape
    dyv = c.ints((M, lddy), int_range(N))
    c.put(dy, dyv)
    wv = c.ints((N, K), int_range(N))
    c.put(w, wv)
    return dyv[:, :N] @ wv, M, K


def r_dense_dgrad(c):
    dx, M, K = _dense_dgrad_common(c)
    c.expect("dx", c.v["out"], cast_to(dx, c.v["out"]).view(c.v["out"].shape))


def _act_bwd(c, g, y_t, mask_t, drop_rate, flags, shape):
    """DropoutGrad then ReluGrad / SigmoidGrad of g (float64) with fresh y (and mask) inputs"""
    if mask_t is not None:
        assert drop_rate == 0.5
        g = g * _mask(c, mask_t).view(shape) * 2
    if flags & L.EPI_SIGMOID:
        y = torch.randint(0, 17, shape, generator=c.g, device=DEV).double() / 16       # dyadic: g y (1 - y) is exact
        c.put(y_t, y)
        return g * y * (1 - y)
    y = c.ints(shape, 2)                                  # ReLU outputs and (to test "> 0") zeros and negatives
    c.put(y_t, y)
    return g * (y > 0) if flags & L.EPI_RELU else g


def r_dense_dgrad_act(c):
    v = c.v
    dx, M, K = _dense_dgrad_common(c)
    g = _act_bwd(c, dx, v["y_act"], v["keep_mask"], v["drop_rate"], v["flags"], (M, K))
    c.expect("dx", v["out"], cast_to(g, v["out"]).view(v["out"].shape))


def r_dense_wgrad(c):
    v = c.v
    x, dy = v["x"], v["dy"]
    M, lddy, ldx, K = dy.shape[0], dy.stride(0), x.stride(0), x.shape[1]
    N = v["N"] if v["N"] is not None else (v["dw"].shape[0] if v["dw"] is not None else dy.shape[1])
    r = int_range(M)
    xv = c.ints((M, ldx), r)
    c.put(c.strided(x, (M, ldx), (ldx, 1)), xv)
    dyv = c.ints(dy.shape, r)
    c.put(dy, dyv)
    g = dyv[:, :N]
    c.expect("dw", v["dw"], (g.t() @ xv[:, :K]).float().view(v["dw"].shape))
    if v["db"] is not None:
        c.expect("db", v["db"], g.sum(0).float().view(v["db"].shape))


LR_T = 2.0 ** -10


def _adam_state(c, n_shape, w_t, m_t, v_t, wb_t, lr_t_dev, g, gs):
    """w in [1, 2), m = v = 0, beta1 = beta2 = 0: m = g gs and v = (g gs)^2 exactly, w within 1 ulp"""
    w0 = c.uniform(n_shape, 1, 2).float().double()
    c.put(w_t, w0)
    c.put(m_t, torch.zeros(n_shape, dtype=torch.float64, device=DEV))
    c.put(v_t, torch.zeros(n_shape, dtype=torch.float64, device=DEV))
    if lr_t_dev is not None:
        lr_t_dev.fill_(LR_T)
    gg = g * gs
    assert float(gg.abs().max()) < 2 ** 12
    c.expect("m", m_t, gg.float().view(m_t.shape), prefill=False)
    c.expect("v", v_t, (gg * gg).float().view(v_t.shape), prefill=False)
    w1 = w0 - LR_T * gg / (gg.abs() + 1e-8)
    c.expect_ulps("w", w_t, w1.view(w_t.shape), 1, prefill=False)
    if wb_t is not None:                               # checked against the w the call wrote (Call.run)
        wb_t.fill_(SENTINEL)
        c._mark(wb_t)
        c.mirror = (wb_t, w_t)
    return dict(beta1=0.0, beta2=0.0, lr=LR_T)        # adam_lr_t(lr, 0, 0, t) = lr


def r_dense_wgrad_adam(c):
    v = c.v
    x, dy, w = v["x"], v["dy"], v["w"]
    M, lddy = dy.shape
    N, K = w.shape
    r = int_range(M)
    xv = c.ints(x.shape, r)
    c.put(x, xv)
    dyv = c.ints(dy.shape, r)
    c.put(dy, dyv)
    g = dyv[:, :N].t() @ xv[:, :K]
    if v["db"] is not None:
        c.expect("db", v["db"], dyv[:, :N].sum(0).float().view(v["db"].shape))
    return _adam_state(c, (N, K), w, v["m"], v["v"], v["w_bf16"], v["lr_t_dev"], g, v["grad_scale"])


def r_adam_tf(c):
    v = c.v
    n = v["n"] if v["n"] is not None else v["w"].numel()
    sl = (lambda t: None if t is None else c.flat(t, n))
    g = c.ints((n,), 8)
    c.put(sl(v["g"]), g)
    return _adam_state(c, (n,), sl(v["w"]), sl(v["m"]), sl(v["v"]), sl(v["w_bf16"]), v["lr_t_dev"], g, v["grad_scale"])


def r_sgd(c):
    v = c.v
    n = v["n"] if v["n"] is not None else v["w"].numel()
    w_t, g_t = c.flat(v["w"], n), c.flat(v["g"], n)
    w0 = torch.randint(-256, 257, (n,), generator=c.g, device=DEV).double() / 64
    g = c.ints((n,), 8)
    c.put(w_t, w0)
    c.put(g_t, g)
    p = (g.float() * torch.tensor(v["grad_scale"], dtype=torch.float32)).double()   # the one product that may round
    w1 = (w0 - LR_T * p).float()
    c.expect("w", w_t, w1, prefill=False)
    if v["w_bf16"] is not None:
        wb = c.flat(v["w_bf16"], n)
        c.expect("w_bf16", wb, w1.to(torch.bfloat16))
    return dict(lr=LR_T)


def r_apply_mask_f32(c):
    v = c.v
    n = v["n"] if v["n"] is not None else v["g"].numel()
    g_t, k_t = c.flat(v["g"], n), c.flat(v["keep"], n)
    g = c.ints((n,), 8)
    c.put(g_t, g)
    keep = torch.randint(0, 3, (n,), generator=c.g, device=DEV).double()           # any non-zero byte keeps
    c.put(k_t, keep)
    c.expect("g", g_t, (g * (keep != 0)).float(), prefill=False)


def r_bias_grad_bf16(c):
    v = c.v
    dy, C_ = v["dy"], v["C_"]
    assert v["group_rows"] == 0
    rows, ld = (v["rows"], v["ld"]) if v["rows"] is not None else dy.shape
    dyf = c.flat(dy, (rows - 1) * ld + C_)
    dyv = c.ints(dyf.shape, int_range(rows))
    c.put(dyf, dyv)
    c.expect("db", c.flat(v["db"], C_), dyv.as_strided((rows, C_), (ld, 1)).sum(0).float())


def _pool_windows(x, N, H, W, Cc):
    """[N, OH, OW, Cc, 4] windows of a 2x2/2 pool (the odd edge dropped), positions in the kernels' order"""
    OH, OW = H // 2, W // 2
    x = x.view(N, H, W, Cc)[:, :2 * OH, :2 * OW].reshape(N, OH, 2, OW, 2, Cc)
    return x.permute(0, 1, 3, 5, 2, 4).reshape(N, OH, OW, Cc, 4)


def _first_argmax(win):
    m, idx = win[..., 0].clone(), torch.zeros(win.shape[:-1], dtype=torch.uint8, device=DEV)
    for j in (1, 2, 3):
        gt = win[..., j] > m                              # strict: the FIRST maximum wins
        m = torch.where(gt, win[..., j], m)
        idx[gt] = j
    return m, idx


def _maxpool(c, routed):
    v = c.v
    x, out = v["x"], v["out"]
    N, H, W, Cc = x.shape
    xv = c.ints(x.shape, 3)
    c.put(x, xv)
    m, idx = _first_argmax(_pool_windows(xv, N, H, W, Cc))
    c.expect("y", out, with_columns(c, out, Cc, m))
    if routed and v["idx"] is not None:
        c.expect("idx", v["idx"], torch.where(m > 0, idx, 4).to(torch.uint8).view(v["idx"].shape))


def r_maxpool2x2_fwd(c):
    _maxpool(c, False)


def r_maxpool2x2_fwd_f32(c):
    _maxpool(c, True)


def r_maxpool2x2_idx_bwd(c):
    v = c.v
    N, H, W, Cc = v["shape"]
    OH, OW = H // 2, W // 2
    dy = v["dy"]
    lddy = v["lddy"] or dy.shape[-1]
    idx = torch.randint(0, 5, (N, OH, OW, Cc), generator=c.g, device=DEV)
    c.put(v["idx"], idx)
    dyf = c.flat(dy, (N * OH * OW - 1) * lddy + Cc)
    dyv = c.ints(dyf.shape, 8)
    c.put(dyf, dyv)
    g = dyv.as_strided((N, OH, OW, Cc), (OH * OW * lddy, OW * lddy, lddy, 1))
    full = torch.zeros(N, OH, 2, OW, 2, Cc, dtype=torch.float64, device=DEV)
    for j in range(4):
        full[:, :, j // 2, :, j % 2] = g * (idx == j)
    dx = torch.zeros(N, H, W, Cc, dtype=torch.float64, device=DEV)
    dx[:, :2 * OH, :2 * OW] = full.reshape(N, 2 * OH, 2 * OW, Cc)
    c.expect("dx", v["out"], cast_to(dx, v["out"]).view(v["out"].shape))


def r_pool4_bwd(c):
    v = c.v
    dy, y, idx_t = v["dy"], v["y"], v["idx"]
    rows = idx_t.numel() // 64
    lddy, ldy = dy.shape[-1], y.shape[-1]
    dyf = c.flat(dy, (rows - 1) * lddy + 64)
    dyv = c.ints(dyf.shape, 8)
    c.put(dyf, dyv)
    yf = c.flat(y, (rows - 1) * ldy + 64)
    yv = c.ints(yf.shape, 2)
    c.put(yf, yv)
    idx = torch.randint(0, 5, (rows, 64), generator=c.g, device=DEV)
    c.put(idx_t, idx)
    g = dyv.as_strided((rows, 64), (lddy, 1)) * (yv.as_strided((rows, 64), (ldy, 1)) > 0)
    big = torch.cat([g * (idx == j) for j in range(4)], 1)
    c.expect("dybig", v["out"], cast_to(big, v["out"]).view(v["out"].shape))


def r_gather_sum_f32(c):
    v = c.v
    G, n = v["idx"].shape
    src_n = v["src"].numel()
    src = c.ints((src_n,), 8)
    c.put(v["src"], src)
    idx = torch.randint(-1, src_n, (G, n), generator=c.g, device=DEV)
    c.put(v["idx"], idx)
    got = torch.where(idx >= 0, src[idx.clamp(min=0)], 0.0).sum(0)
    c.expect("dst", v["dst"], got.float().view(v["dst"].shape))


def r_scatter_cast_bf16(c):
    v = c.v
    G, n = v["idx"].shape
    dst = v["dst"]
    src = torch.randn(n, generator=c.g, device=DEV, dtype=torch.float64).float()   # the cast rounds: RNE
    c.put(v["src"], src.double())
    k = min(G * n, dst.numel()) * 9 // 10                 # distinct targets for k of the G x n slots, -1 elsewhere
    pos = torch.full((G * n,), -1, dtype=torch.int64, device=DEV)
    pos[torch.randperm(G * n, generator=c.g, device=DEV)[:k]] = torch.randperm(dst.numel(), generator=c.g,
                                                                               device=DEV)[:k]
    pos = pos.view(G, n)
    c.put(v["idx"], pos)
    exp = c.sentinel_like(dst).view(-1)
    for gi in range(G):
        ok = pos[gi] >= 0
        exp[pos[gi][ok]] = src[ok].to(dst.dtype)
    c.expect("dst", dst, exp.view(dst.shape))


def r_scatter_channel_bf16(c):
    v = c.v
    src, dst, ch = v["src"], v["dst"], v["ch"]
    s = torch.randn(src.shape, generator=c.g, device=DEV, dtype=torch.float64).float()
    c.put(src, s.double())
    exp = c.sentinel_like(dst)
    exp.view(-1, dst.shape[-1])[:, ch] = s.reshape(-1).to(dst.dtype)
    c.expect("dst", dst, exp)


def r_dense_epilogue_bwd(c):
    v = c.v
    gp = v["g_post"]
    g = c.ints(gp.shape, 8)
    c.put(gp, g)
    r = _act_bwd(c, g, v["y"], v["keep_mask"], v["drop_rate"], v["flags"], gp.shape)
    c.expect("g_pre", v["out"], cast_to(r, v["out"]).view(v["out"].shape))


def r_window_gather(c):
    v = c.v
    src, out = v["src"], v["out"]
    B, Hs, Ws, Cc = src.shape
    rows, cols, win, st = v["rows"], v["cols"], v["win"], v["stride"]
    s = c.ints(src.shape, 8)
    c.put(src, s)
    u = s.unfold(1, win, st).unfold(2, win, st)[:, :rows, :cols]       # [B, rows, cols, C, win, win]
    c.expect("out", out, cast_to(u.permute(0, 1, 2, 4, 5, 3), out).reshape(out.shape))


def r_window_scatter_sum(c):
    v = c.v
    go, gs = v["g_out"], v["g_src"]
    B, Hs, Ws, Cc = gs.shape
    rows, cols, win, st = v["rows"], v["cols"], v["win"], v["stride"]
    n = B * rows * cols * win * win * Cc
    gf = c.flat(go, n)
    g = c.ints((n,), 8)
    c.put(gf, g)
    g = g.view(B, rows, cols, win, win, Cc)
    acc = torch.zeros(B, Hs, Ws, Cc, dtype=torch.float64, device=DEV)
    for pr in range(rows):
        for pc in range(cols):
            acc[:, pr * st:pr * st + win, pc * st:pc * st + win] += g[:, pr, pc]
    c.expect("g_src", gs, cast_to(acc, gs))


def _pairwise_inputs(c):
    v = c.v
    sims, w2, b1 = v["sims"], v["w2"], v["b1"]
    s = torch.randint(-64, 65, sims.shape, generator=c.g, device=DEV).double() / 64   # dyadic: every product is exact
    c.put(sims, s)
    w = torch.randint(-8, 9, (2,), generator=c.g, device=DEV).double() / 8
    c.put(c.flat(w2, 2), w)
    b = torch.randint(-8, 9, (1,), generator=c.g, device=DEV).double() / 8
    c.put(c.flat(b1, 1), b)
    s2 = s.view(-1, 2)
    return s2[:, 0] * w[0] + s2[:, 1] * w[1] + b[0]


def r_pairwise_dense(c):
    r = _pairwise_inputs(c)
    c.expect("r", c.v["out"], r.float().view(c.v["out"].shape))


def r_pairwise_dense_act(c):
    r = _pairwise_inputs(c)
    if c.v["flags"] & L.EPI_RELU:
        r = r.clamp(min=0)
    c.expect("r", c.v["out"], r.float().view(c.v["out"].shape))


def r_pairwise_dense_bwd(c):
    v = c.v
    n = v["r"].numel()
    s = torch.randint(-64, 65, (n, 2), generator=c.g, device=DEV).double() / 64
    c.put(v["sims"], s)
    r = c.ints((n,), 2)                                 # the forward's output: zeros and negatives test act'(r)
    c.put(v["r"], r)
    dr = c.ints((n,), 8)
    c.put(v["dr"], dr)
    g = dr * (r > 0) if v["flags"] & L.EPI_RELU else dr
    c.expect("dw2", c.flat(v["dw2"], 2), (g[:, None] * s).sum(0).float())
    c.expect("db1", c.flat(v["db1"], 1), g.sum().view(1).float())


def r_mean_f32(c):
    v = c.v
    n = v["v"].numel()
    assert n & (n - 1) == 0, "a power-of-two count makes the mean exact"
    x = c.ints((n,), 64)
    c.put(v["v"], x)
    c.expect("mean", c.flat(v["out"], 1), (x.sum() / n).view(1).float())


def r_scale_cast_bf16(c):
    v = c.v
    s = torch.randn(v["src"].shape, generator=c.g, device=DEV, dtype=torch.float64).float()
    c.put(v["src"], s.double())
    scale = torch.tensor(v["scale"], dtype=torch.float32)
    c.expect("dst", v["dst"], (s * scale.to(DEV)).to(torch.bfloat16).view(v["dst"].shape))


REPLAY = {name[2:]: fn for name, fn in list(globals().items()) if name.startswith("r_") and callable(fn)}


def replay(ctx, rec, seed):
    """mismatch descriptions of one rebuilt call (empty when every output is exact)"""
    c = Call(ctx, rec, seed)
    return c.run(REPLAY[rec["m"]](c))


def describe(configs, rec):
    def short(x):
        if isinstance(x, dict) and "T" in x:
            s = f"{x['dt']}{x['T']}"
            return s + (f"@{x['al']}" if x["al"] else "") + (f"+{x['off']}" if x.get("off") else "")
        if isinstance(x, dict) and "D" in x:
            d = x["D"]
            return "conv(N=%d %dx%dx%d -> K=%d %dx%d s%d pad %d,%d P=%d Q=%d ldy=%d)" % (
                d["N"], d["H"], d["W"], d["C"], d["K"], d["R"], d["S"], d["stride_h"], d["pad_t"], d["pad_l"], d["P"],
                d["Q"], d["ldy"])
        if isinstance(x, list):
            return "(" + ", ".join(short(y) for y in x) + ")"
        return repr(x)
    args = [short(x) for x in rec["a"]] + [f"{k}={short(x)}" for k, x in rec["k"].items()]
    return f"{rec['m']}({', '.join(args)}){' [3xTF32]' if rec['x3'] else ''} <- {configs[0]}"


def _tensor_arg(rec, i, name):
    if len(rec["a"]) > i:
        return rec["a"][i]
    return rec["k"].get(name)


# ----------------------------------------------------------------------------- tests
def required_signatures():
    """predicates (name -> test on a record) that some recorded call must satisfy"""
    def f32(rec, i, name):
        t = _tensor_arg(rec, i, name)
        return isinstance(t, dict) and t.get("dt") == "float32"

    def bf16(rec, i, name):
        t = _tensor_arg(rec, i, name)
        return isinstance(t, dict) and t.get("dt") == "bfloat16"

    def desc(rec):
        return rec["a"][0]["D"]

    def rows(rec, i, name):
        return _tensor_arg(rec, i, name)["T"][0]

    return {
        "tf32 strided dgrad of conv2d_4 at B = 32": lambda r: r["m"] == "conv2d_dgrad" and f32(r, 1, "dy") and
        desc(r)["stride_h"] == 2 and desc(r)["N"] == 32,
        "tf32 dense wgrad at M = 2": lambda r: r["m"] == "dense_wgrad" and f32(r, 0, "x") and rows(r, 1, "dy") == 2,
        "tf32 dense wgrad at M = 32": lambda r: r["m"] == "dense_wgrad" and f32(r, 0, "x") and rows(r, 1, "dy") == 32,
        "3xTF32 dense fwd": lambda r: r["m"] == "dense_fwd" and f32(r, 0, "x") and r["x3"],
        "3xTF32 conv fwd": lambda r: r["m"] == "conv2d_fwd" and f32(r, 1, "x") and r["x3"] and desc(r)["K"] > 1,
        "conv_k1_fwd_f32": lambda r: r["m"] == "conv2d_fwd" and f32(r, 1, "x") and desc(r)["K"] == 1,
        "conv_k1_dgrad_f32": lambda r: r["m"] == "conv2d_dgrad" and f32(r, 1, "dy") and desc(r)["K"] == 1,
        "conv_k1_wgrad_f32": lambda r: r["m"] == "conv2d_wgrad" and f32(r, 1, "x") and desc(r)["K"] == 1,
        "pool4_reduce_f32": lambda r: r["m"] == "conv2d_pool4_fwd" and f32(r, 1, "x"),
        "pool4_bwd_f32": lambda r: r["m"] == "pool4_bwd" and f32(r, 0, "dy"),
        "bf16 dense_wgrad": lambda r: r["m"] == "dense_wgrad" and bf16(r, 0, "x"),
        "fused dense wgrad + Adam at M = 32": lambda r: r["m"] == "dense_wgrad_adam" and rows(r, 1, "dy") == 32,
        "DCNF dense_dgrad at M = 768": lambda r: r["m"] == "dense_dgrad" and bf16(r, 0, "dy") and rows(r, 0, "dy") == 768,
        "pairwise_dense_bwd": lambda r: r["m"] == "pairwise_dense_bwd",
        "mean_f32 over B = 16": lambda r: r["m"] == "mean_f32" and math.prod(_tensor_arg(r, 0, "v")["T"]) == 16,
        "bias_grad_f32 past 4096 rows": lambda r: r["m"] == "bias_grad_bf16" and f32(r, 0, "dy") and
        rows(r, 0, "dy") > 4096,
        "scale_cast_bf16": lambda r: r["m"] == "scale_cast_bf16",
    }


def test_inventory_is_classified(inventory, capsys):
    calls, per_config = inventory
    methods = {}
    for configs, rec in calls:
        methods.setdefault(rec["m"], []).append(rec)
    with capsys.disabled():
        print(f"\nrecorded calls per configuration (calls, distinct signatures):")
        for cfg, (n, d) in per_config.items():
            print(f"  {cfg}: {n} calls, {d} signatures")
        n_rep = sum(len(r) for m, r in methods.items() if m in REPLAY)
        print(f"distinct signatures: {len(calls)}; replayed {n_rep} in {len(set(methods) & set(REPLAY))} methods, "
              f"excluded {len(calls) - n_rep}:")
        for m in sorted(set(methods) - set(REPLAY)):
            print(f"  {m}: {len(methods[m])} ({EXCLUDED.get(m, 'UNCLASSIFIED')})")
    unclassified = sorted(m for m in methods if m not in REPLAY and m not in EXCLUDED)
    assert not unclassified, f"recorded methods with neither a replay nor an exclusion: {unclassified}"
    assert not set(REPLAY) & set(EXCLUDED)
    missing = [name for name, ok in required_signatures().items() if not any(ok(rec) for _, rec in calls)]
    assert not missing, f"signatures the models no longer record: {missing}"


@pytest.mark.parametrize("method", sorted(REPLAY))
def test_replay_is_exact(ctx, inventory, method):
    calls = [(cfg, rec) for cfg, rec in inventory[0] if rec["m"] == method]
    assert calls, f"no recorded configuration calls {method}"
    failures = []
    for i, (cfg, rec) in enumerate(calls):
        try:
            bad = replay(ctx, rec, i)
        except AssertionError as e:
            bad = [f"replay: {e}"]
        failures += [f"{describe(cfg, rec)}: {b}" for b in bad]
        torch.cuda.empty_cache()
    print(f"{method}: {len(calls)} signatures replayed")
    assert not failures, f"{len(failures)} failures:\n" + "\n".join(failures[:30])


# ----------------------------------------------------------------------------- adam_tf_bf16g (data-parallel optimizer)
def test_adam_tf_bf16g_exact_moments(ctx):
    """beta1 = beta2 = 0, m = v = 0: m is the bf16 gradient times grad_scale and v its square, bit for bit; w within
    1 ulp of the float64 step and the bf16 mirror its rounding."""
    g0 = torch.Generator(device=DEV).manual_seed(7)
    n = 4 * 100003
    g = (torch.randint(-255, 256, (n,), generator=g0, device=DEV).double() / 4)
    g[::7] = 0
    w = (torch.rand(n, generator=g0, device=DEV, dtype=torch.float64) + 1).float()
    m, v = torch.zeros(n, device=DEV), torch.zeros(n, device=DEV)
    wb = torch.empty(n, dtype=torch.bfloat16, device=DEV)
    w0 = w.double()
    ctx.adam_tf_bf16g(w, g.to(torch.bfloat16), m, v, wb, LR_T, 0.0, 0.0, 1e-8, 1, grad_scale=0.5)
    gg = g * 0.5
    assert mismatch(m, gg.float(), "m") is None
    assert mismatch(v, (gg * gg).float(), "v") is None
    assert float(ulps(w.double(), w0 - LR_T * gg / (gg.abs() + 1e-8), torch.float32).max()) <= 1
    assert torch.equal(wb, w.to(torch.bfloat16))


def test_adam_tf_bf16g_vs_oracle(ctx):
    """As test_adam_vs_oracle for adam_tf; the bf16-gradient entry point takes segments of a multiple of 4 elements
    (DataParallel shards are) and rejects any other length instead of skipping its tail."""
    gen = torch.Generator().manual_seed(47)
    n = 100004
    w = torch.randn(n, generator=gen)
    gr = (torch.randn(n, generator=gen) * 1e-2).to(torch.bfloat16)
    m = torch.randn(n, generator=gen) * 1e-3
    v = torch.rand(n, generator=gen) * 1e-4
    wr, mr, vr = T.tf_adam_update(w.double(), gr.double() * 0.5, m.double(), v.double(), 3, 0.1, 0.9, 0.999, 1e-8)
    wd, gd, md, vd = (t.to(DEV).clone() for t in (w, gr, m, v))
    wb = torch.empty(n, dtype=torch.bfloat16, device=DEV)
    ctx.adam_tf_bf16g(wd, gd, md, vd, wb, 0.1, 0.9, 0.999, 1e-8, 3, grad_scale=0.5)
    assert float((wd.cpu().double() - wr).abs().max()) < 1e-5
    assert float((md.cpu().double() - mr).abs().max()) < 1e-7
    assert float((vd.cpu().double() - vr).abs().max()) < 1e-9
    assert torch.equal(wb, wd.to(torch.bfloat16))
    for odd in (n - 1, n - 2, n - 3):
        with pytest.raises(L.A3DError, match="multiple of 4"):
            ctx.adam_tf_bf16g(wd[:odd], gd[:odd], md[:odd], vd[:odd], wb[:odd], 0.1, 0.9, 0.999, 1e-8, 3)
