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
  checked within 1 ulp of the float64 step.  The sigmoid epilogue (DCNF dense_1) is checked within 1 ulp of its output
  type.
- Data movement (DCNF patches and cells), tile means of dyadic depths and the FP8 quantisers: bit for bit.
- Results that cannot be exact (bilinear resize, SILog loss, pairwise similarities, the CRF) are checked against a
  float64 reference within a per-element bound derived from the kernel's float32 arithmetic (`within`); a bf16 or E4M3
  output must be the round-to-nearest-even of the reference wherever that reference is farther than the bound from a
  rounding midpoint (`rounded`).  Each replay prints its worst error as a share of its bound.

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

from oracle import dcnf as OD
from oracle import fp8 as OF
from oracle import tf1_ops as T

if torch.cuda.is_available():
    from ann3depth_b200 import _lib as L
    from ann3depth_b200 import dcnf as dcnf_mod
    from ann3depth_b200 import ops

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
    if isinstance(v, dict):
        return {"O": {k: enc(x, groups) for k, x in sorted(v.items())}}
    if v is None or isinstance(v, (bool, int, float, str)):
        return v
    return {"obj": type(v).__name__}


def tensors(v):
    if isinstance(v, dict) and "T" in v:
        yield v
    elif isinstance(v, dict) and "O" in v:
        yield from tensors(list(v["O"].values()))
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


def dcnf(label, B, train, **kw):
    config[0] = label
    g = torch.Generator().manual_seed(B)
    images = torch.rand(B, 480, 640, 3, generator=g).cuda()
    depths = (torch.rand(B, 480, 640, 1, generator=g) * 0.95 + 0.05).cuda()
    models.dcnf(images, depths, train=train, **kw).run()
    torch.cuda.synchronize()


# Besides the benchmark's batches, one batch per batch-dependent code path (DESIGN section 2): the dense layers' batch is
# their GEMM's M, and the tile width, the chunking above 256 rows and the kernel choice above 32 / 128 rows follow it.
train("msdn bf16 B=32", 32)
train("msdn bf16 B=32 sequential", 32, phases=(1,), overlap=False, fuse_dense_adam=False)
for B in (1, 5, 33, 100, 130):
    train(f"msdn bf16 B={B}", B)
for B in (1, 7, 32, 100, 300, 512):
    infer(f"msdn bf16 inference B={B}", B)
for B in (7, 300):
    infer(f"msdn fp8 inference B={B}", B, "fp8")
for dtype in ("tf32", "tf32x3"):
    for B in (2, 32, 33):
        train(f"msdn {dtype} B={B}", B, dtype)
        infer(f"msdn {dtype} inference B={B}", B, dtype)
dcnf("dcnf B=16", 16, True)
dcnf("dcnf B=16 grid4", 16, True, graph="grid4", r_nonneg=True, train_pairwise=True, predict="map")
dcnf("dcnf inference B=16", 16, False)
for B in (1, 3, 6):
    dcnf(f"dcnf B={B}", B, True)
dcnf("dcnf inference B=6", 6, False)
dcnf("dcnf B=3 patches", 3, True, unary="patches")            # the literal B*48-patch unary batch
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
    "resize_affine_tf1": "augmentation resize: checked against oracle/augment.py (test_gpu_augment)",
    "resize_affine_tf1_s2d": "augmentation resize: checked against oracle/augment.py (test_gpu_augment)",
    "augment_draw": "random draw: checked against oracle/augment.py (test_gpu_augment)",
    "conv2d_fwd_fp8": "FP8 GEMM: every tuner candidate is exact in test_gpu_tuner_candidates",
    "conv2d_pool4_fwd_fp8": "FP8 GEMM: every tuner candidate is exact in test_gpu_tuner_candidates",
    "dense_fwd_fp8": "FP8 GEMM: every tuner candidate is exact in test_gpu_tuner_candidates",
    "stamp": "timeline mark, no arithmetic",
    "increment_i64": "step counter, no arithmetic",
    "bernoulli_mask": "random mask: its rate and independence are tested in test_gpu_parity_full",
    "adam_tf_bf16g": "data parallel only (not recorded on one GPU): test_adam_tf_bf16g_* check it directly",
}


# ----------------------------------------------------------------------------- rebuilding a call
def _tensors(v):
    if isinstance(v, dict) and "T" in v:
        yield v
    elif isinstance(v, dict) and "O" in v:
        yield from _tensors(list(v["O"].values()))
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
        self.checks, self.marks, self.mirror, self.stats, self.post = [], {}, None, {}, []
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
        if isinstance(v, dict) and "O" in v:
            return {k: self._mat(x) for k, x in v["O"].items()}
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
        self.checks.append((name, t, ref, ("ulps", n, ftz)))

    def expect_within(self, name, t, ref, bound, prefill=True):
        """t (float32) within the per-element float64 `bound` of the float64 ref"""
        if prefill:
            t.fill_(SENTINEL)
        self._mark(t)
        self.checks.append((name, t, ref, ("within", bound)))

    def expect_rounded(self, name, t, ref, bound, prefill=True):
        """t (bf16 or E4M3) is the round-to-nearest-even of a float32 value within `bound` of the float64 ref
        (`rounded`)"""
        if prefill:
            t.view(_int_dtype(t.element_size())).fill_(0x7F if t.element_size() == 1 else -1)     # NaN either way
        self._mark(t)
        self.checks.append((name, t, ref, ("rounded", bound)))

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
            elif n[0] == "within":
                m, self.stats[name] = within(t, exp, n[1], name)
            elif n[0] == "rounded":
                m, self.stats[name] = rounded(t, exp, n[1], name)
            else:
                _, n, ftz = n
                u = ulps(t.double(), exp, t.dtype)
                if ftz:
                    u = torch.where((exp.abs() < 2.0 ** -126) & (t == 0), 0.0, u)
                worst = float(u.max()) if u.numel() else 0.0
                m = None if worst <= n else \
                    f"{name}: {int((u > n).sum())} of {u.numel()} beyond {n} ulp, worst {worst:.3g} at " \
                    f"{tuple(int(i) for i in (u == u.max()).nonzero()[0])}"
            if m:
                bad.append(m)
        for check in self.post:                            # checks that need the results, not only a reference
            m = check()
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
    x = c.ints((n,), 64)
    c.put(v["v"], x)
    # the integer sum is exact and the kernel's division rounds to nearest; so does float64 -> float32 of the quotient,
    # which for a count this small never lies within a float64 ulp of a float32 tie (a batch of 3 or 6 is not a power of 2)
    assert n < 2 ** 16
    c.expect("mean", c.flat(v["out"], 1), (x.sum() / n).view(1).float())


def r_scale_cast_bf16(c):
    v = c.v
    s = torch.randn(v["src"].shape, generator=c.g, device=DEV, dtype=torch.float64).float()
    c.put(v["src"], s.double())
    scale = torch.tensor(v["scale"], dtype=torch.float32)
    c.expect("dst", v["dst"], (s * scale.to(DEV)).to(torch.bfloat16).view(v["dst"].shape))


# ----------------------------------------------------------------------------- inexact results: derived bounds
# u is the unit roundoff of float32 and gamma(k) = k u / (1 - k u) bounds the relative error of k float32 roundings in a
# row (Higham, Accuracy and Stability of Numerical Algorithms, 2nd ed., Lemma 3.1).  The CUDA maths functions the
# kernels call are used with their documented worst cases (CUDA C++ Programming Guide, "Mathematical Functions",
# liba3d builds with the defaults -prec-div=true -prec-sqrt=true -ftz=false): sqrtf and the division correctly rounded,
# logf <= 1 ulp, expf <= 2 ulp, powf <= 4 ulp; 1 ulp of a float32 x is at most 2u|x|.
U = 2.0 ** -24


def gamma(k):
    return k * U / (1 - k * U)


def ulp32(x):
    """the spacing of float32 at |x| (float64 tensor; 2^-149 among the subnormals)"""
    _, e = torch.frexp(x.abs())
    return torch.where(x == 0, 2.0 ** -149, torch.ldexp(torch.ones_like(x), (e - 24).clamp(min=-149)))


def within(got, ref, bound, name):
    """(mismatch or None, worst |got - ref| / bound): got must lie within the per-element bound of ref"""
    err = (got.double() - ref).abs()
    bad = ~(err <= bound)                                        # NaN fails
    frac = float(torch.where(err == 0, 0.0, err / bound).max()) if err.numel() else 0.0
    if not bool(bad.any()):
        return None, frac
    i = tuple(int(j) for j in bad.nonzero()[0])
    return (f"{name}: {int(bad.sum())} of {err.numel()} beyond their bound, first at {i}: got {float(got[i]):.9g} "
            f"expected {float(ref[i]):.9g} +- {float(bound[i]):.3g}"), frac


def _round_to(x, dtype):
    """x (float64) rounded to nearest even in float32, then in dtype (E4M3 saturating as the kernels' cvt .satfinite):
    monotone in x, so every float32 value in [a, b] rounds to a value in [_round_to(a), _round_to(b)]"""
    x = x.float()
    if dtype == torch.float8_e4m3fn:
        x = x.clamp(-448.0, 448.0)
    return x.to(dtype).double()


def rounded(got, ref, bound, name):
    """The RNE rule of a bf16 / E4M3 output whose float32 value lies within `bound` of ref: got must be the rounding of
    ref wherever [ref - bound, ref + bound] holds no rounding midpoint, and one of the two neighbours elsewhere.
    Returns (mismatch or None, share of the elements where either neighbour is accepted)."""
    lo, hi = _round_to(ref - bound, got.dtype), _round_to(ref + bound, got.dtype)
    g = got.double()
    bad = ~((g >= lo) & (g <= hi))
    share = float((lo != hi).double().mean()) if g.numel() else 0.0
    if not bool(bad.any()):
        return None, share
    i = tuple(int(j) for j in bad.nonzero()[0])
    return (f"{name}: {int(bad.sum())} of {g.numel()} not the rounding of the reference, first at {i}: got "
            f"{float(g[i]):.9g} expected {float(lo[i]):.9g} .. {float(hi[i]):.9g} (ref {float(ref[i]):.9g})"), share


# -- bilinear resize
def resize_ref(x, OH, OW, chunk=32):
    """TF1 bilinear resize of x (float64 [B,H,W,C] on the device) with oracle/tf1_ops's float32 coordinates, which the
    kernels reproduce bit for bit, and the lerp in float64: (value, largest |corner| of each output)."""
    B, H, W, C = x.shape
    ylo, yhi, yl = (t.to(x.device) for t in T.resize_axis(H, OH))
    xlo, xhi, xl = (t.to(x.device) for t in T.resize_axis(W, OW))
    yl, xl = yl.double().view(1, OH, 1, 1), xl.double().view(1, 1, OW, 1)
    vals, mags = [], []
    for b0 in range(0, B, chunk):
        top, bot = x[b0:b0 + chunk, ylo], x[b0:b0 + chunk, yhi]
        tl, tr, bl, br = top[:, :, xlo], top[:, :, xhi], bot[:, :, xlo], bot[:, :, xhi]
        t = tl + (tr - tl) * xl
        vals.append(t + (bl + (br - bl) * xl - t) * yl)
        mags.append(torch.maximum(torch.maximum(tl.abs(), tr.abs()), torch.maximum(bl.abs(), br.abs())))
    return torch.cat(vals), torch.cat(mags)


# The kernels' lerp, top = tl + (tr - tl) lx, bot likewise, r = top + (bot - top) ly, in float32 with the fused
# multiply-adds nvcc contracts these lines into (its default, --fmad=true): the differences round once (2uM each), each
# fma once (uM), so |top - exact| <= 2uM lx + uM <= 3uM and |r - exact| <= (1 - ly) 3uM + ly 3uM + 2uM ly + uM <= 6uM,
# M the largest |corner|.
LERP_U = 6


def s2d(v, s):
    """[B, OH, OW, C] -> the space-to-depth(s) image [B, OH/s, OW/s, s*s*C], channel (dy*s + dx)*C + c"""
    B, OH, OW, C = v.shape
    return v.reshape(B, OH // s, s, OW // s, s, C).permute(0, 1, 3, 2, 4, 5).reshape(B, OH // s, OW // s, s * s * C)


def resize_s2d_kernel(src, W, C, s, dstC):
    """the kernel a3d_resize_bilinear_tf1_s2d (elementwise.cu) dispatches to for a float32 source"""
    if s == 4 and C == 3 and (W * 3) % 4 == 0 and W * 3 * 4 * 4 <= 100 * 1024 and dstC % 4 == 0 and src % 16 == 0:
        return "pipelined"
    return "s2d4c3" if s == 4 and C == 3 else "generic"


def source_image(c, t):
    """random pixels of t's dtype: float32 in [0, 1) with every mantissa bit in use, or uint8; returns float64 values"""
    if t.dtype == torch.uint8:
        v = torch.randint(0, 256, t.shape, generator=c.g, device=DEV, dtype=torch.uint8)
        t.copy_(v)
        return v.double()
    v = torch.rand(t.shape, generator=c.g, device=DEV)
    t.copy_(v)
    return v.double()


def expect_resized(c, name, out, ref, mag, scale=1.0):
    """out[..., :real] is ref (lerp bound LERP_U u M; `scale` a float32 factor applied after the lerp, one more
    rounding), out[..., real:] zero"""
    real = ref.shape[-1]
    bound = (LERP_U + (scale != 1.0)) * U * mag * scale
    ref = ref * scale
    if out.dtype == torch.float32:
        c.expect_within(name, out[..., :real], ref, bound)
    else:
        c.expect_rounded(name, out[..., :real], ref, bound)
    if out.shape[-1] > real:
        c.expect(name + " padding", out[..., real:], torch.zeros_like(out[..., real:]))


def r_resize_bilinear_tf1(c):
    v = c.v
    x = source_image(c, v["src"])
    ref, mag = resize_ref(x, v["OH"], v["OW"])
    expect_resized(c, "resized", v["out"], ref, mag)


def r_resize_bilinear_tf1_s2d(c):
    v = c.v
    src, s, out = v["src"], v["s"], v["out"]
    x = source_image(c, src)
    ref, mag = resize_ref(x, v["OH"], v["OW"])
    # uint8 pixels: the float32 lerp of the integers, then times fl(1/255) (one more rounding)
    scale = float(torch.tensor(1 / 255, dtype=torch.float32)) if src.dtype == torch.uint8 else 1.0
    expect_resized(c, "resized s2d", out, s2d(ref, s), s2d(mag, s), scale)


def r_resize_bilinear_tf1_s2d_e4m3(c):
    v = c.v
    src, out = v["src"], v["out"]
    x = source_image(c, src)
    if src.dtype == torch.uint8:              # each tap is the correctly rounded float32 quotient k / 255
        x = (x / 255).float().double()
    ref, mag = resize_ref(x, v["OH"], v["OW"])
    # codes of 256 x the float32 lerp (the scaling by 2^8 is exact)
    c.expect_rounded("codes", out[..., :48], s2d(ref, 4) * 256, LERP_U * U * s2d(mag, 4) * 256)
    c.expect("code padding", out[..., 48:].view(torch.uint8), torch.zeros_like(out[..., 48:].view(torch.uint8)))


# -- FP8 quantisers: every step is one float32 operation, restated bit for bit by oracle/fp8.py
def _fp8_source(c, t, relu):
    """bf16 values over six binades, a different magnitude per leading index and one all-zero image or row"""
    lead = t.shape[0]
    mag = torch.pow(2.0, torch.randint(-6, 7, (lead,) + (1,) * (t.dim() - 1), generator=c.g, device=DEV)).float()
    x = torch.randn(t.shape, generator=c.g, device=DEV) * mag
    if relu:
        x = x.clamp(min=0)
    if lead > 1:
        x[lead // 2] = 0
    t.copy_(x.to(torch.bfloat16))
    return t.float()


def _expect_codes(c, q, s, qr, sr):
    c.expect("codes", q.view(torch.uint8), qr.view(torch.uint8).reshape(q.shape))
    c.expect("scales", s, sr.reshape(s.shape))


def r_quantize_rows_e4m3(c):
    v = c.v
    x = _fp8_source(c, v["x"], False)
    qr, sr = OF.quantize_rows(x)
    _expect_codes(c, v["q"], v["scale"], qr, sr)


def r_quantize_e4m3(c):
    v = c.v
    x = _fp8_source(c, v["x"], True)
    qr, sr = OF.quantize_images(x)
    _expect_codes(c, v["out"], v["scale"], qr, sr)


def r_maxpool2x2_quantize_e4m3(c):
    v = c.v
    x = _fp8_source(c, v["x"], True)
    out = v["out"]
    ldy = v["ldy"] or out.shape[-1]
    B, H, W, C = x.shape
    pooled = _first_argmax(_pool_windows(x, B, H, W, C))[0]
    pooled = torch.cat([pooled, torch.zeros(B, H // 2, W // 2, ldy - C, device=DEV)], -1)
    qr, sr = OF.quantize_images(pooled)
    _expect_codes(c, out, v["scale"], qr, sr)


# -- DCNF data movement: bit-exact (the bf16 cast of float32 pixels is RNE in the kernels and in torch)
def _padded_windows(im, pad, size, stride, rows, cols):
    """[B, rows, cols, size, size, 3] windows of the zero-padded image"""
    B, H, W, _ = im.shape
    ph, pw = max(0, (rows - 1) * stride + size - pad - H), max(0, (cols - 1) * stride + size - pad - W)
    p = F.pad(im.permute(0, 3, 1, 2), (pad, pw, pad, ph))
    return p.unfold(2, size, stride).unfold(3, size, stride)[:, :, :rows, :cols].permute(0, 2, 3, 4, 5, 1)


def cells_s2d(p):
    """[..., 2Y, 2X, 3] -> [..., Y, X, 16]: channel (2a + b)*3 + c = pixel (2Y + a, 2X + b, c), channels 12..15 zero"""
    *lead, H2, W2, _ = p.shape
    q = p.reshape(*lead, H2 // 2, 2, W2 // 2, 2, 3).movedim(-4, -3).reshape(*lead, H2 // 2, W2 // 2, 12)
    return torch.cat([q, torch.zeros_like(q[..., :4])], -1)


def r_extract_patches_s2d(c):
    v = c.v
    im, out, fold = v["images"], v["out"], v["fold"]
    B, H, W, _ = im.shape
    x = torch.randn(im.shape, generator=c.g, device=DEV)
    im.copy_(x)
    rows, cols = -(-H // 40), -(-W // 40)
    cells = cells_s2d(_padded_windows(x, 30, 100, 40, rows, cols)).reshape(B * rows * cols, 50, 50, 16)
    if fold == 4:                         # position X holds cells X .. X+3, zeros past the row end
        cells = torch.cat([F.pad(cells[:, :, k:], (0, 0, 0, k)) for k in range(4)], -1)
    c.expect("cells", out, cells.to(torch.bfloat16).view(out.shape))


def r_image_cells_s2d(c):
    v = c.v
    im, out, pad = v["images"], v["out"], v["pad"]
    x = torch.randn(im.shape, generator=c.g, device=DEV)
    im.copy_(x)
    p = F.pad(x.permute(0, 3, 1, 2), (pad, pad, pad, pad)).permute(0, 2, 3, 1)
    c.expect("cells", out, cells_s2d(p).to(torch.bfloat16).view(out.shape))


def r_tile_means(c):
    v = c.v
    dp = v["depth"]
    B, H, W = dp.shape[:3]
    # multiples of 2^-12 in [0, 1): any order of the 1600-term sum is exact (< 2^23 units), so the one IEEE division
    # by 1600 is the only rounding
    d = torch.randint(0, 4096, dp.shape, generator=c.g, device=DEV).double() / 4096
    dp.copy_(d)
    rows, cols = -(-H // 40), -(-W // 40)
    s = _padded_windows(d.expand(*d.shape[:3], 3), 0, 40, 40, rows, cols)[..., 0].sum((-1, -2)).reshape(B, -1)
    q = s / 1600
    assert_no_f32_tie(q)
    c.expect("tile means", v["out"], q.float().view(v["out"].shape))


def assert_no_f32_tie(q):
    """the float64 quotients q round to the same float32 as the exact ones: none within a float64 ulp of a float32 tie"""
    f = q.float()
    up, dn = torch.nextafter(f, torch.full_like(f, math.inf)), torch.nextafter(f, torch.full_like(f, -math.inf))
    mid = torch.minimum((q - (f.double() + up.double()) / 2).abs(), (q - (f.double() + dn.double()) / 2).abs())
    assert bool((mid > q.abs() * 2.0 ** -52).all()), "a quotient lies at a float32 tie"


# -- scale-invariant log loss (elementwise.cu silog_loss_kernel)
def silog_reference(o, t, lon):
    """float64 reference of a3d_silog_loss on float32 o, t [B, n] (device) with the float32 lambda/n `lon`, and the
    first-order bound of each float32 result: dict of (value, bound) for loss_ps [B], loss [1] and the gradient [B, n].

    d_i = log(fl(o_i + eps)) - log(fl(t_i + eps)) (0 for a NaN logarithm): two logf (<= 1 ulp each) and a subtraction,
    |e_d| <= 2u(|lo| + |lt|) + u|d|.  Sum d and sum d^2 are per-thread runs of ceil(n/512) terms, then two 5-level
    shuffle trees (32 lanes, then the 16 warps): every term goes through at most k = ceil(n/512) + 10 additions, so
    their rounding is below gamma(k) sum |term| (plus one rounding of d^2).  loss_ps = s2 - lon s1^2 adds two roundings
    of lon s1^2 and one of the difference; the loss is the mean over B (per-lane runs of ceil(B/32), a 5-level tree,
    one division).  The gradient (2 d_i - 2 lon s1) / fl(o_i + eps) * fl(1/B) rounds the numerator twice and then
    three times more relatively."""
    B, n = o.shape
    eps = float(torch.tensor(1e-8, dtype=torch.float32))
    ao = (o + torch.tensor(1e-8, dtype=torch.float32, device=o.device)).double()      # fl(o + eps)
    at = (t + torch.tensor(1e-8, dtype=torch.float32, device=o.device)).double()
    lo, lt = torch.log(ao).nan_to_num(0.0), torch.log(at).nan_to_num(0.0)
    live = ~torch.isnan(torch.log(ao))
    lo = torch.where(live, lo, 0.0)
    d = lo - lt
    ed = 2 * U * (lo.abs() + lt.abs()) + U * d.abs()
    k = -(-n // 512) + 10
    s1, s2 = d.sum(1), (d * d).sum(1)
    e1 = ed.sum(1) + gamma(k) * d.abs().sum(1)
    e2 = (2 * d.abs() * ed).sum(1) + gamma(k + 1) * (d * d).sum(1)
    lps = s2 - lon * s1 * s1
    elps = e2 + 2 * lon * s1.abs() * e1 + 2 * U * lon * s1 * s1 + U * lps.abs()
    kb = -(-B // 32) + 5
    loss = lps.mean().view(1)
    eloss = (elps.sum() / B + gamma(kb) * lps.abs().sum() / B + U * loss.abs()).view(1)
    num = 2 * d - 2 * lon * s1[:, None]
    enum = 2 * ed + 2 * lon * e1[:, None] + U * 2 * lon * s1.abs()[:, None] + U * num.abs()
    g = torch.where(live, num / ao / B, 0.0)
    eg = torch.where(live, enum / ao.abs() / B + 4 * U * g.abs(), 0.0)
    return dict(loss_ps=(lps, elps), loss=(loss, eloss), grad=(g, eg))


def r_silog_loss(c):
    v = c.v
    o_t, t_t = v["out"], v["tar"]
    B = o_t.shape[0]
    n = o_t.numel() // B
    # predictions in [-0.4, 1.2): a quarter negative (the NaN branch, gradient exactly 0), none within 1e-3 of -eps;
    # targets k/255 with zeros (quantised depth maps)
    o = torch.rand(B, n, generator=c.g, device=DEV) * 1.6 - 0.4
    o = torch.where(o.abs() < 1e-3, 0.5, o)
    t = torch.randint(0, 256, (B, n), generator=c.g, device=DEV).float() / 255
    c.put(o_t, o)
    c.put(t_t, t)
    lon = float(torch.tensor(v["lambda_over_n"], dtype=torch.float32))
    ref = silog_reference(o, t, lon)
    assert v["loss_ps"] is not None and v["loss"] is not None, "the models pass their loss buffers"
    c.expect_within("loss_ps", v["loss_ps"], *ref["loss_ps"])
    c.expect_within("loss", v["loss"], *ref["loss"])
    ld = v["dout_ld"] or n
    for key, dt in (("dout", torch.float32), ("dout_bf16", torch.bfloat16)):
        if v[key] is not None:
            gv = c.strided(v[key], (B, n), (ld, 1))          # columns [n, ld) stay untouched
            g, eg = ref["grad"]
            (c.expect_within if dt == torch.float32 else c.expect_rounded)(f"{key} (ld {ld})", gv, g, eg)


# -- DCNF pairwise features (crf.cu tile_features_kernel, pair_similarity_kernel)
def pairwise_image(B, H, W, gen, device="cpu"):
    """float32 images whose pairwise similarities are exact up to sqrtf and expf: every pixel r = g = b = k/64 with
    1 <= k <= 63, so the colour code k (2^16 + 2^8 + 1) 2^2 and its bin 4k + floor(k/64 + k/2^14) = 4k are exact in
    float32 and at least 0.011 of a bin away from both bin edges, (r + g + b) / 3 = k/64 is exact, and every sum of
    squares of differences is exact (multiples of 2^-12 below 2^12, integers below 2^23).  Each 40x40 tile has one of
    the levels 20, 21, 26 by column (a neighbour differs by 0, 1 or 5 levels: colour similarities near 1, 0.54, 0.04)
    and 0..3 of its pixels moved one level up (similarities between 0.98 and 1, histograms equal or a few counts
    apart)."""
    rows, cols = -(-H // 40), -(-W // 40)
    level = torch.tensor([20, 21, 20, 26])[torch.arange(cols) % 4].view(1, 1, cols).expand(B, rows, cols)
    k = level.repeat_interleave(40, 1).repeat_interleave(40, 2).clone()[:, :H, :W]
    moved = torch.randint(0, 4, (B, rows, cols), generator=gen)
    for b, r, cc in zip(*torch.nonzero(moved, as_tuple=True)):
        m = int(moved[b, r, cc])
        pos = torch.randperm(1600, generator=gen)[:m]
        ys, xs = r * 40 + pos // 40, cc * 40 + pos % 40
        ok = (ys < H) & (xs < W)
        k[b, ys[ok], xs[ok]] += 1
    return (k.float() / 64).unsqueeze(-1).expand(B, H, W, 3).contiguous().to(device)


def pairwise_reference(im, pl, pr):
    """float64 similarities [B, n_pairs, 2] of oracle/dcnf.py on the given pair list, and their bound.

    With the sums of squares s exact, a = sqrtf(s) = sqrt(s)(1 + d), |d| <= u, and expf(-a) within 2 ulp of exp(-a), so
    |got - exp(-sqrt s)| <= exp(-sqrt s) sqrt(s) u (1 + small) + 2 ulp (gamma = 1: -gamma a is exact)."""
    sp = OD.superpixels(im.double().cpu())                                  # [B, n, 1600, 3]
    hist = torch.stack([torch.stack([OD.color_histogram(t) for t in bt]) for bt in sp])
    feats = (sp.mean(-1), hist)
    sims, bounds = [], []
    for f in feats:
        dist = torch.linalg.vector_norm(f[:, pl] - f[:, pr], dim=2)
        ref = torch.exp(-dist)
        sims.append(ref)
        first = ref * dist * U * (1 + 1e-6)
        bounds.append(first + 2 * ulp32(ref + first))
    return torch.stack(sims, -1), torch.stack(bounds, -1)


def assert_similarities_span(ref):
    """both features reach below 0.05 and above 0.95: a kernel that drops or saturates either cannot pass"""
    for j, what in enumerate(("colour", "histogram")):
        lo, hi = float(ref[..., j].min()), float(ref[..., j].max())
        assert lo < 0.05 and hi > 0.95, f"{what} similarities span only [{lo:.3g}, {hi:.3g}]"


def pair_graph(n_pairs):
    """the DCNF pair list with n_pairs pairs (48: the reference checkerboard graph, 82: grid4)"""
    pl, pr = OD.pair_indices()
    if n_pairs != len(pl):
        pl, pr = dcnf_mod.grid4_pairs()
    assert len(pl) == n_pairs, n_pairs
    return list(pl), list(pr)


def _put_pairs(c, pl_t, pr_t):
    pl, pr = pair_graph(pl_t.numel())
    c.put(pl_t, torch.tensor(pl, dtype=torch.float64, device=DEV))
    c.put(pr_t, torch.tensor(pr, dtype=torch.float64, device=DEV))
    return pl, pr


def r_pairwise_features(c):
    v = c.v
    im = v["images"]
    B, H, W, _ = im.shape
    assert v["gamma"] == 1.0
    pl, pr = _put_pairs(c, v["pl"], v["pr"])
    x = pairwise_image(B, H, W, torch.Generator().manual_seed(int(torch.randint(0, 2 ** 31, (1,), generator=c.g,
                                                                                device=DEV))))
    im.copy_(x)
    ref, bound = pairwise_reference(x, pl, pr)
    assert_similarities_span(ref)
    out = v["out"]
    c.expect_within("similarities", out, ref.to(DEV).view(out.shape), bound.to(DEV).view(out.shape))


# -- the CRF (crf.cu crf_kernel)
EPS32 = float(torch.tensor(1e-7, dtype=torch.float32))      # the kernel's eps (the oracle's is the float64 1e-7)
PI32 = float(torch.tensor(math.pi, dtype=torch.float32))     # CUDART_PI_F


def build_A(r, pl, pr, n):
    """A = I + diag(R 1) - R of each image, R scattered pair by pair with the kernel's last-write-wins (float64 [B, n, n],
    differentiable in r [B, n_pairs])"""
    last = {}
    for k, (a, b) in enumerate(zip(pl, pr)):
        last[(a, b)] = k
        last[(b, a)] = k
    rows, cols = zip(*last)
    idx = torch.tensor(list(last.values()))
    B = r.shape[0]
    bi = torch.arange(B)[:, None].expand(B, len(idx))
    R = torch.zeros(B, n, n, dtype=torch.float64).index_put((bi, torch.tensor(rows).expand(B, -1),
                                                              torch.tensor(cols).expand(B, -1)), r[:, idx])
    return torch.eye(n, dtype=torch.float64) + torch.diag_embed(R.sum(2)) - R


def crf_reference(z, y, r, pl, pr, grad_scale, naive):
    """float64 reference of a3d_crf_fwd_bwd on float32 z, y [B, n] and r [B, n_pairs] (CPU) and the first-order bound
    of each float32 output: dict name -> (value, bound).  nll and its gradients are float64 autograd of
    oracle/dcnf.nll_stable or nll_naive on A built from r.

    Error terms, first order in u, with L the Cholesky factor of A and y* = A^-1 z (Higham, ch. 8 and 10):
    - forming A: each diagonal entry is 1 plus a sum of the deg_i non-zero r of its row, |dA_form| <= gamma(deg_i + 1)
      A_ii on the diagonal;
    - the right-looking Cholesky (Thm 10.3) and the two substitutions (Thm 8.5, every dot product a sum of < n terms in
      any order): (A + E) y^ = z with |E| <= E3 = dA_form + gamma(3n + 1) |L||L^T|, so |y^ - y*| <= |A^-1| E3 |y^|;
      the quadratic form ||L^-1 z||^2 = z^T (A + E)^-1 z is within |y*|^T E3 |y*| (+ the rounding of its sum);
    - log det: 2 sum logf(L^_ii) with L^ L^T = A + E', |E'| <= dA_form + gamma(n + 1)|L||L^T|: within
      sum |A^-1| o E' + (4u + 2 gamma(13)) sum |log L_ii| (logf <= 1 ulp, a sum through 13 additions);
    - block sums (one term per thread, 5 shuffle levels, 8 warps): gamma(14) of the sum of |terms|; the energy's row
      dot products add gamma(n) per row;
    - the naive loss (src/models.py:163-171 in float32): relative errors through expf (2 ulp), powf (4 ulp, and
      CUDART_PI_F != pi), sqrtf(expf(logdet)), the products and quotients (one rounding each) and logf (1 ulp); the
      kernel's eps = fl(1e-7) differs from the oracle's 1e-7 by |EPS32 - 1e-7|.
    The naive gradient is g = u/(u + eps) times the stable one (g computed in float32): it drops the factor (Z - eps)/Z
    of d log Z, the eps (sum z) term of d(z^T (A^-1 + eps) z)/dz and sqrt(det)/(sqrt(det) + eps) of d log fac/dr.  The
    difference to the naive loss's exact gradient is computed here in float64 and added to the bound: the kernel is
    checked against the documented approximation within its rounding."""
    B, n = z.shape
    gs = float(torch.tensor(grad_scale, dtype=torch.float32))
    z, y = z.double().clone().requires_grad_(True), y.double()
    r = r.double().clone().requires_grad_(True)
    A = build_A(r, pl, pr, n)
    zc, yc = z[:, :, None], y[:, :, None]
    nll_fn = OD.nll_naive if naive else OD.nll_stable
    nll = torch.stack([nll_fn(A[b:b + 1], yc[b:b + 1], zc[b:b + 1]) for b in range(B)])
    dz, dr = torch.autograd.grad(nll.sum(), (z, r))
    z, r, A, nll = z.detach(), r.detach(), A.detach(), nll.detach()
    dz, dr = gs * dz, gs * dr
    L = torch.linalg.cholesky(A)
    Ai = torch.linalg.inv(A)
    ys = torch.linalg.solve(A, z[:, :, None])[..., 0]
    logdet = 2 * torch.log(torch.diagonal(L, dim1=1, dim2=2)).sum(1)
    LL = L.abs() @ L.abs().transpose(1, 2)
    diagA = torch.diagonal(A, dim1=1, dim2=2)
    deg = ((A != 0).sum(2) - 1).double()
    Eform = torch.diag_embed(gamma(deg + 1) * diagA)
    E3 = Eform + gamma(3 * n + 1) * LL
    ya = ys.abs()
    dys = (Ai.abs() @ (E3 @ ya[:, :, None]))[..., 0]                                    # |y^ - y*|
    eld = (Ai.abs() * (Eform + gamma(n + 1) * LL)).sum((1, 2)) + \
        (4 * U + 2 * gamma(13)) * torch.log(torch.diagonal(L, dim1=1, dim2=2)).abs().sum(1)
    quad = (z * ys).sum(1)
    equad = (ya[:, None, :] @ E3 @ ya[:, :, None])[:, 0, 0] + gamma(14) * quad.abs()
    zz = (z * z).sum(1)
    ezz = gamma(14) * zz
    Ay = (A.abs() @ y.abs()[:, :, None])[..., 0]
    TE = (y.abs() * Ay + 2 * (z * y).abs() + z * z).sum(1)
    energy = (y * (A @ y[:, :, None])[..., 0]).sum(1) - 2 * (z * y).sum(1) + zz
    eE = gamma(n + 17) * TE + (y.abs() * (Eform @ y.abs()[:, :, None])[..., 0]).sum(1)
    c0 = 0.5 * n * math.log(math.pi)
    ec0 = 0.5 * n * (abs(math.log(PI32) - math.log(math.pi)) + 2 * U * math.log(math.pi)) + U * c0
    if not naive:
        p1 = energy + c0
        p2 = p1 - 0.5 * logdet
        p3 = p2 + quad
        enll = eE + ec0 + 0.5 * eld + equad + ezz + U * (p1.abs() + p2.abs() + p3.abs() + nll.abs())
        g = torch.ones(B, dtype=torch.float64)
        rg = torch.zeros(B, dtype=torch.float64)
    else:
        ex_E = torch.exp(-energy)
        rE = eE + 2 * ulp32(ex_E) / ex_E
        sq = torch.exp(0.5 * logdet)
        rfac = 4 * 2 * U + 0.5 * n * abs(PI32 - math.pi) / math.pi + (eld + 4 * U) / 2 + U + \
            abs(EPS32 - 1e-7) / sq + 2 * U
        zsum = z.sum(1)
        Q = quad + 1e-7 * zsum * zsum - zz
        eQ = equad + ezz + 1e-7 * zsum * zsum * (2 * U + 2 * gamma(14)) + abs(EPS32 - 1e-7) * zsum * zsum + \
            U * ((quad + 1e-7 * zsum * zsum).abs() + Q.abs())
        ex_Q = torch.exp(Q)
        rQ = eQ + 2 * ulp32(ex_Q) / ex_Q
        fac = math.pi ** (n / 2) / (sq + 1e-7)
        Z = fac * ex_Q + 1e-7
        rZ = (rfac + rQ + U) * (fac * ex_Q) / Z + U + abs(EPS32 - 1e-7) / Z
        uu = ex_E / Z
        ru = rE + rZ + U
        g = uu / (uu + 1e-7)
        enll = g * ru + abs(EPS32 - 1e-7) / (uu + 1e-7) + U + 2 * U * nll.abs()
        rg = (1 - g) * ru + 2 * U + abs(EPS32 - 1e-7) / (uu + 1e-7)
    # dz = (gs g) 2 (y^ - y): the kernel's formula, its rounding, and what separates it from the exact gradient
    dzk = 2 * gs * g[:, None] * (ys - y)
    edz = dzk.abs() * (rg[:, None] + 3 * U) + 2 * gs * g[:, None] * dys + (dz - dzk).abs()
    out = dict(ystar=(ys, dys), logdet=(logdet, eld), nll=(nll, enll), dz=(dz, edz), A=A, z=z, E3=E3)
    # dr_k = (gs g)((y_l - y_r)^2 - (y^_l - y^_r)^2 - 0.5 ||L^-1 (e_l - e_r)||^2)
    plt, prt = torch.tensor(pl), torch.tensor(pr)
    V = torch.zeros(len(pl), n, dtype=torch.float64)
    V[torch.arange(len(pl)), plt] += 1
    V[torch.arange(len(pl)), prt] -= 1
    P = Ai @ V.t()                                                                     # [B, n, n_pairs] = A^-1 v_k
    nrm = (V.t()[None] * P).sum(1)
    enrm = (P.abs() * (E3 @ P.abs())).sum(1) + gamma(n + 2) * nrm.abs()
    dyv, dsv = y[:, plt] - y[:, prt], ys[:, plt] - ys[:, prt]
    eds = dys[:, plt] + dys[:, prt] + U * dsv.abs()
    drk = gs * g[:, None] * (dyv ** 2 - dsv ** 2 - 0.5 * nrm)
    inner = 2 * U * dyv ** 2 + 2 * dsv.abs() * eds + U * dsv ** 2 + 0.5 * enrm + \
        3 * U * (dyv ** 2 + dsv ** 2 + 0.5 * nrm.abs())
    edr = gs * g[:, None] * inner + drk.abs() * (rg[:, None] + 2 * U) + (dr - drk).abs()
    out["dr"] = (dr, edr)
    out["approx"] = (float((dz - dzk).abs().max()), float((dr - drk).abs().max()))
    out["g"] = g
    return out


def crf_inputs(B, n, n_pairs, gen, device="cpu"):
    """z, y in [0, 1), r >= 0 in [0, 2]: A = I + a weighted graph Laplacian, SPD with kappa_inf(A) <= 1 + 2 max_i
    sum_j r_ij <= 17 (degree <= 4)"""
    z = torch.rand(B, n, generator=gen)
    y = torch.rand(B, n, generator=gen)
    r = torch.rand(B, n_pairs, generator=gen) * 2
    return z.to(device), y.to(device), r.to(device)


def expect_crf(c, outs, ref, B, n, n_pairs):
    """declares the CRF outputs of a call (dict of output tensors, entries may be None) against crf_reference"""
    c.expect("status", outs["status"], torch.zeros(B, dtype=torch.int32, device=DEV))
    for key in ("ystar", "logdet", "nll", "dz", "dr"):
        t = outs.get(key)
        if t is not None:
            val, bound = ref[key]
            c.expect_within(key, t, val.to(DEV).view(t.shape), bound.to(DEV).view(t.shape))
    c.post.append(lambda: crf_solution_checks(c.stats, outs["ystar"], ref))


def crf_solution_checks(stats, ystar, ref):
    """ystar through its normwise backward error ||z - A y^||_inf / (||A||_inf ||y^||_inf + ||z||_inf), bounded by the
    same norm of E3 |y^| (crf_reference; about (3n + 1) u ||L||L^T|||_inf / ||A||_inf, printed as c in c n u), and the
    forward error below 1e-5"""
    A, z, E3 = ref["A"], ref["z"], ref["E3"]
    n = z.shape[1]
    yh = ystar.double().cpu().view(z.shape)
    denom = A.abs().sum(2).amax(1) * yh.abs().amax(1) + z.abs().amax(1)
    eta = (z - (A @ yh[:, :, None])[..., 0]).abs().amax(1) / denom
    bound = (E3 @ yh.abs()[:, :, None])[..., 0].amax(1) / denom
    stats["ystar backward error"] = float((eta / bound).max())
    stats["c of c n u"] = float((bound / (n * U)).max())
    fwd = float((yh - ref["ystar"][0]).abs().max())
    if not bool((eta <= bound).all()):
        return f"ystar: backward error {float(eta.max()):.3g} above its bound {float(bound.max()):.3g}"
    if not fwd < 1e-5:
        return f"ystar: forward error {fwd:.3g} >= 1e-5"
    return None


def r_crf(c):
    v = c.v
    z_t, y_t, r_t = v["z"], v["y"], v["r"]
    B, n = z_t.shape
    n_pairs = r_t.shape[1]
    pl, pr = _put_pairs(c, v["pl"], v["pr"])
    gen = torch.Generator().manual_seed(int(torch.randint(0, 2 ** 31, (1,), generator=c.g, device=DEV)))
    z, y, r = crf_inputs(B, n, n_pairs, gen)
    for t, x in ((z_t, z), (y_t, y), (r_t, r)):
        c.put(t, x.double().to(DEV))
    ref = crf_reference(z, y, r, pl, pr, v["grad_scale"], v["naive"])
    if v["naive"]:
        assert float(ref["logdet"][0].max()) < 80            # float32 det(A) = expf(logdet) does not overflow
    outs = v["out"]
    assert outs is not None, "the models pass their output buffers"
    expect_crf(c, outs, ref, B, n, n_pairs)




REPLAY = {name[2:]: fn for name, fn in list(globals().items()) if name.startswith("r_") and callable(fn)}


def replay(ctx, rec, seed):
    """(mismatch descriptions of one rebuilt call, empty when every output is right; {output: worst error as a share of
    its bound, or the share of elements where a bf16 / E4M3 rounding may go either way})"""
    c = Call(ctx, rec, seed)
    return c.run(REPLAY[rec["m"]](c)), c.stats


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
        if isinstance(x, dict) and "O" in x:
            return "{" + ", ".join(f"{k}: {short(y)}" for k, y in x["O"].items()) + "}"
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
        # the batch-dependent dense paths (tc_gemm.cu, conv.cu): forward tiles bn = 64 / 128 / 256 and a partial 44-row
        # chunk past 256 rows; the SIMT dgrad + separate epilogue above 128 rows; the rows dgrad at row counts that are
        # not multiples of 128; the TF32 tiles of bn = 64
        **{f"bf16 dense_fwd at M = {m}": (lambda m: lambda r: r["m"] == "dense_fwd" and bf16(r, 0, "x") and
                                          rows(r, 0, "x") == m)(m) for m in (33, 100, 130, 300)},
        "dense_dgrad_act at M = 130": lambda r: r["m"] == "dense_dgrad_act" and rows(r, 0, "dy") == 130,
        **{f"DCNF dense_dgrad at M = {m}": (lambda m: lambda r: r["m"] == "dense_dgrad" and bf16(r, 0, "dy") and
                                            rows(r, 0, "dy") == m)(m) for m in (144, 288)},
        "tf32 dense wgrad at M = 33": lambda r: r["m"] == "dense_wgrad" and f32(r, 0, "x") and rows(r, 1, "dy") == 33,
        "tf32 dense dgrad at M = 33": lambda r: r["m"] == "dense_dgrad_act" and f32(r, 0, "dy") and
        rows(r, 0, "dy") == 33,
        # the CRF as DCNF trains: the naive loss (its default), the 82-pair grid4 graph, one image
        "crf naive": lambda r: r["m"] == "crf" and r["k"].get("naive") is True,
        "crf on 82 pairs": lambda r: r["m"] == "crf" and _tensor_arg(r, 2, "r")["T"][1] == 82,
        "crf at B = 1": lambda r: r["m"] == "crf" and _tensor_arg(r, 0, "z")["T"][0] == 1,
        "crf with dr": lambda r: r["m"] == "crf" and isinstance(r["k"]["out"]["O"].get("dr"), dict),
        "coarse silog_loss gradient at ld 4096": lambda r: r["m"] == "silog_loss" and r["k"].get("dout_ld") == 4096 and
        (isinstance(r["k"].get("dout"), dict) or isinstance(r["k"].get("dout_bf16"), dict)),
        "bf16 silog_loss gradient": lambda r: r["m"] == "silog_loss" and isinstance(r["k"].get("dout_bf16"), dict),
        "resize_bilinear_tf1_s2d pipelined (float32 source)": lambda r: r["m"] == "resize_bilinear_tf1_s2d" and
        f32(r, 0, "src") and bf16(r, 4, "out") and resize_s2d_kernel(
            _tensor_arg(r, 0, "src")["al"], _tensor_arg(r, 0, "src")["T"][2], 3, r["a"][3], 64) == "pipelined",
        "resize_bilinear_tf1_s2d float32 output (TF32 modes)": lambda r: r["m"] == "resize_bilinear_tf1_s2d" and
        f32(r, 4, "out"),
        **{f"{m} in FP8 inference": (lambda m: lambda r: r["m"] == m)(m) for m in (
            "quantize_rows_e4m3", "quantize_e4m3", "maxpool2x2_quantize_e4m3", "resize_bilinear_tf1_s2d_e4m3")},
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


def test_fused_dense_update_stays_within_its_batch_limit(inventory):
    """a3d_dense_wgrad_adam takes at most L.DENSE_WGRAD_ADAM_MAX_M rows: above it the MSDN step must record the separate
    weight gradients of both coarse dense kernels instead (which TF-Adam then updates as a group)."""
    calls = inventory[0]
    over = [describe(cfg, rec) for cfg, rec in calls
            if rec["m"] == "dense_wgrad_adam" and _tensor_arg(rec, 1, "dy")["T"][0] > L.DENSE_WGRAD_ADAM_MAX_M]
    assert not over, over
    widths = {_tensor_arg(rec, 0, "x")["T"][1] for cfg, rec in calls
              if "msdn bf16 B=33 phase 1" in cfg and rec["m"] == "dense_wgrad" and _tensor_arg(rec, 1, "dy")["T"][0] == 33}
    assert widths == {4096, 12288}, widths          # dense_1 reads d0 [B, 4096], dense_0 reads c4 [B, 12288]


@pytest.mark.parametrize("method", sorted(REPLAY))
def test_replay_is_exact(ctx, inventory, method, capsys):
    calls = [(cfg, rec) for cfg, rec in inventory[0] if rec["m"] == method]
    assert calls, f"no recorded configuration calls {method}"
    failures, worst = [], {}
    for i, (cfg, rec) in enumerate(calls):
        try:
            bad, stats = replay(ctx, rec, i)
        except AssertionError as e:
            bad, stats = [f"replay: {e}"], {}
        failures += [f"{describe(cfg, rec)}: {b}" for b in bad]
        for k, x in stats.items():
            worst[k] = max(worst.get(k, 0.0), x)
        torch.cuda.empty_cache()
    print(f"{method}: {len(calls)} signatures replayed")
    if worst:
        with capsys.disabled():
            print(f"\n  {method}: worst error / bound (bf16 and E4M3: share of elements within the bound of a rounding "
                  f"midpoint): " + ", ".join(f"{k} {x:.3g}" for k, x in sorted(worst.items())))
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


# ----------------------------------------------------------------------------- cases the models do not record
def _check(msgs):
    bad = [m for m, _ in msgs if m]
    assert not bad, "\n".join(bad)


@pytest.mark.parametrize("case", ["pipelined", "pipelined uint8", "s2d4c3", "generic s=2", "generic C=1", "tf32"])
def test_resize_s2d_kernels(ctx, case):
    """Each kernel behind a3d_resize_bilinear_tf1_s2d against the float64 lerp on oracle coordinates: the row-pipelined
    one (float32 and uint8 sources), the s = 4 / C = 3 fallback for a source that is not 16-byte aligned, the generic
    one (s = 2, or C = 1) and the float32 output of the TF32 modes.  The recorded models reach only the first and the
    last (required_signatures)."""
    g = torch.Generator(device=DEV).manual_seed(11)
    B, H, W, C, OH, OW, s = {"generic s=2": (2, 50, 66, 3, 24, 32, 2), "generic C=1": (2, 55, 73, 1, 56, 76, 4)}.get(
        case, (3, 240, 320, 3, 116, 152, 4))
    dstC = (s * s * C + 7) // 8 * 8 + 8
    n = B * H * W * C
    if case == "pipelined uint8":
        src = torch.randint(0, 256, (B, H, W, C), generator=g, device=DEV, dtype=torch.uint8)
    else:
        buf = torch.rand(n + 4, generator=g, device=DEV)
        src = buf[1:n + 1].view(B, H, W, C) if case == "s2d4c3" else buf[:n].view(B, H, W, C)
    if case != "pipelined uint8":
        assert resize_s2d_kernel(src.data_ptr(), W, C, s, dstC) == case.split()[0] or case == "tf32"
    out = torch.full((B, OH // s, OW // s, dstC), SENTINEL, device=DEV,
                     dtype=torch.float32 if case == "tf32" else torch.bfloat16)
    ctx.resize_bilinear_tf1_s2d(src, OH, OW, s, out=out)
    ref, mag = resize_ref(src.double(), OH, OW)
    ref, mag = s2d(ref, s), s2d(mag, s)
    real = s * s * C
    sc = float(torch.tensor(1 / 255, dtype=torch.float32)) if src.dtype == torch.uint8 else 1.0
    bound = (LERP_U + (sc != 1.0)) * U * mag * sc
    check = within if case == "tf32" else rounded
    _check([check(out[..., :real], ref * sc, bound, case)])
    assert bool((out[..., real:] == 0).all()), "padding channels are not zero"


def test_silog_loss_row_pitch(ctx):
    """the gradient rows at a pitch of 4096 (the coarse prediction's [B, 4096] gradient): within the bounds of
    silog_reference, the 26 columns past n untouched, float32 and bf16"""
    g = torch.Generator(device=DEV).manual_seed(12)
    B, n, ld = 3, 4070, 4096
    o = torch.rand(B, n, generator=g, device=DEV) * 1.6 - 0.4
    o = torch.where(o.abs() < 1e-3, 0.5, o)
    t = torch.randint(0, 256, (B, n), generator=g, device=DEV).float() / 255
    lon = float(torch.tensor(0.5 / 4070, dtype=torch.float32))
    ref = silog_reference(o, t, lon)
    d32 = torch.full((B, ld), SENTINEL, device=DEV)
    d16 = torch.full((B, ld), SENTINEL, device=DEV, dtype=torch.bfloat16)
    lps, loss = torch.empty(B, device=DEV), torch.empty(1, device=DEV)
    ctx.silog_loss(o, t, 0.5 / 4070, want_grad=False, loss_ps=lps, loss=loss, dout=d32, dout_ld=ld)
    ctx.silog_loss(o, t, 0.5 / 4070, want_grad=False, loss_ps=lps, loss=loss, dout_bf16=d16, dout_ld=ld)
    _check([within(lps, *ref["loss_ps"], "loss_ps"), within(loss, *ref["loss"], "loss"),
            within(d32[:, :n], *ref["grad"], "dout"), rounded(d16[:, :n], *ref["grad"], "dout_bf16")])
    assert bool((d32[:, n:] == SENTINEL).all() and (d16[:, n:] == torch.tensor(SENTINEL).bfloat16()).all())
    assert bool((d32[:, :n][o < 0] == 0).all()), "the NaN branch's gradient is not exactly 0"


def _crf_call(ctx, z, y, r, pl, pr, naive):
    B = z.shape[0]
    dev = lambda x, dt=torch.float32: torch.tensor(x, dtype=dt, device=DEV) if not torch.is_tensor(x) else x.to(DEV)
    return ctx.crf(dev(z), dev(y), dev(r), dev(pl, torch.int32), dev(pr, torch.int32), grad_scale=1.0 / B,
                   want_dr=True, naive=naive)


@pytest.mark.parametrize("n_pairs", [48, 82])
def test_crf_naive_unsaturated(ctx, n_pairs, capsys):
    """The naive loss (the DCNF default) where it is not saturated: u/(u + eps) between 0.01 and 0.99 for some images,
    logdet < 80 (float32 expf(logdet) overflows above 88.7, as TF 1.3's float32 determinant does: reference behaviour).
    Every output against crf_reference; the size of the documented gradient approximation is printed."""
    pl, pr = pair_graph(n_pairs)
    g = torch.Generator().manual_seed(13)
    B, n = 8, 48
    rho = torch.linspace(0.05, 0.6, B) * 48 / n_pairs            # the same spread of log det on the denser graph
    z = (0.5 + 0.05 * torch.randn(B, n, generator=g)).float()
    y = (z.double() + 0.02 * torch.randn(B, n, generator=g, dtype=torch.float64)).float()
    r = (rho[:, None] * (1 + 0.1 * torch.rand(B, n_pairs, generator=g))).float()
    ref = crf_reference(z, y, r, pl, pr, 1.0 / B, True)
    gg = ref["g"]
    assert bool(((gg > 0.01) & (gg < 0.99)).sum() >= 3) and float(ref["logdet"][0].max()) < 80, (gg, ref["logdet"][0])
    res = _crf_call(ctx, z, y, r, pl, pr, True)
    assert int(res["status"].abs().max()) == 0
    msgs = [within(res[k], ref[k][0].to(DEV), ref[k][1].to(DEV), k) for k in ("ystar", "logdet", "nll", "dz", "dr")]
    msgs.append((crf_solution_checks({}, res["ystar"], ref), None))
    with capsys.disabled():
        dz = ref["dz"][0]
        print(f"\n  naive CRF, {n_pairs} pairs: worst error / bound " +
              ", ".join(f"{k} {f:.3g}" for k, (_, f) in zip(("ystar", "logdet", "nll", "dz", "dr"), msgs)) +
              f"; dropped terms of the naive gradient: dz {ref['approx'][0]:.3g} ({ref['approx'][0] / float(dz.abs().max()):.2g}"
              f" of max |dz|), dr {ref['approx'][1]:.3g}")
    _check(msgs)


@pytest.mark.parametrize("naive", [False, True])
@pytest.mark.parametrize("n_pairs", [48, 82])
@pytest.mark.parametrize("B", [1, 3, 6, 16])
def test_crf_not_spd(ctx, B, n_pairs, naive):
    """r < 0 can leave the SPD cone (the reference's pairwise layer is unconstrained): the image reports the Cholesky
    step that failed in `status` and every output of it is 0, not NaN; the other images of the batch are unaffected."""
    pl, pr = pair_graph(n_pairs)
    g = torch.Generator().manual_seed(14 + B)
    z, y, r = crf_inputs(B, 48, n_pairs, g)
    bad = torch.arange(B) % 2 == 0
    r[bad] = -1.0
    res = _crf_call(ctx, z, y, r, pl, pr, naive)
    st = res["status"].cpu()
    assert bool((st[bad] > 0).all()) and bool((st[~bad] == 0).all()), st
    for k in ("ystar", "nll", "logdet", "dz", "dr"):
        got = res[k].cpu()
        assert bool((got[bad] == 0).all()), f"{k} of a non-SPD image is not 0"
        assert bool(torch.isfinite(got).all()), k
    if bool((~bad).any()):
        ref = crf_reference(z[~bad], y[~bad], r[~bad], pl, pr, 1.0 / B, naive)
        _check([within(res[k].cpu()[~bad], *ref[k], k) for k in ("ystar", "logdet", "nll", "dz", "dr")])
