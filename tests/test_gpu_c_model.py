"""The model-level C entry points (`a3d_msdn_create / _step / _infer`, include/a3d.h): one MSDN step driven through
ctypes ALONE -- no ann3depth_b200 host logic on the path, torch only owns the device buffers -- must reproduce the step
of the Python host (`models.msdn`, same kernels, same sequential schedule) and the float64 oracle.  This is the boundary a
non-Python host binds (INTEGRATION.md): `session.run(model_op)` of src/ann3depth.py:126-127 for src/models.py:203-367."""
import ctypes as C
import math

import pytest
import torch

pytestmark = pytest.mark.gpu

from oracle import msdn as OM

if torch.cuda.is_available():
    from ann3depth_b200 import _lib as L
    from ann3depth_b200 import models
    from ann3depth_b200.params import Arena, msdn_specs, pack

DEV = "cuda:0"


def cos(a, b):
    a, b = a.double().cpu().reshape(-1), b.double().cpu().reshape(-1)
    return float((a @ b) / (a.norm() * b.norm() + 1e-300))


class CNet:
    """ctypes-only driver of the C model API."""

    def __init__(self, B, in_hw=(480, 640), depth_hw=(55, 73), train=True, beta2=1.0, seed=2):
        self.lib = L.load()
        ctx = models.get_context(0)                       # only for the a3d_ctx handle
        self.h = ctx.h
        self.B = B
        nbytes = self.lib.a3d_msdn_workspace_bytes(self.h, B, in_hw[0], in_hw[1], depth_hw[0], depth_hw[1], int(train))
        assert nbytes > 0
        self.ws = torch.empty(nbytes, dtype=torch.uint8, device=DEV)       # the ONE caller-owned buffer
        self.net = C.c_void_p()
        L.check(self.lib.a3d_msdn_create(self.h, B, in_hw[0], in_hw[1], depth_hw[0], depth_hw[1], int(train),
                                         C.c_void_p(self.ws.data_ptr()), nbytes, None, C.byref(self.net)), "msdn_create")
        L.check(self.lib.a3d_msdn_configure(self.net, beta2, seed), "msdn_configure")
        ptrs = [C.c_void_p() for _ in range(5)]
        total = C.c_size_t()
        L.check(self.lib.a3d_msdn_arena(self.net, *[C.byref(p) for p in ptrs], C.byref(total)), "msdn_arena")
        self.total = total.value
        self.w_ptr, self.m_ptr, self.v_ptr, self.g_ptr, self.wb_ptr = [p.value for p in ptrs]

    def segments(self):
        out = {}
        n = self.lib.a3d_msdn_segment(self.net, -1, None, None, None, None)
        for i in range(n):
            name, off, numel, shape = C.c_char_p(), C.c_size_t(), C.c_size_t(), (C.c_int * 4)()
            self.lib.a3d_msdn_segment(self.net, i, C.byref(name), C.byref(off), C.byref(numel), C.byref(shape))
            out[name.value.decode()] = (off.value, numel.value, tuple(s for s in shape if s))
        return out

    def view(self, ptr, dtype=torch.float32):
        """torch view of an arena buffer inside the workspace (for loading / reading back)"""
        off = ptr - self.ws.data_ptr()
        nb = self.total * (4 if dtype == torch.float32 else 2)
        return self.ws[off:off + nb].view(dtype)

    def load_packed(self, packed_w):
        self.view(self.w_ptr).copy_(packed_w)
        L.check(self.lib.a3d_msdn_sync_weights(self.net, None), "sync_weights")

    def step(self, images, depths, mask=None):
        losses = torch.zeros(2, device=DEV)
        rc = self.lib.a3d_msdn_step(self.net, C.c_void_p(images.data_ptr()), C.c_void_p(depths.data_ptr()),
                                    C.c_void_p(mask.data_ptr()) if mask is not None else None,
                                    C.c_void_p(losses.data_ptr()), None)
        assert rc >= 1, (rc, self.lib.a3d_last_error())
        return rc, losses

    def infer(self, images):
        fine = torch.empty(self.B, 55, 74, device=DEV)
        coarse = torch.empty(self.B, 55, 74, device=DEV)
        L.check(self.lib.a3d_msdn_infer(self.net, C.c_void_p(images.data_ptr()), C.c_void_p(fine.data_ptr()),
                                        C.c_void_p(coarse.data_ptr()), None), "msdn_infer")
        return fine, coarse

    def close(self):
        self.lib.a3d_msdn_destroy(self.net)


def make(B):
    g = torch.Generator().manual_seed(0)
    images = torch.rand(B, 480, 640, 3, generator=g)
    depths = torch.rand(B, 55, 73, 1, generator=g) * 0.95 + 0.05
    mask = (torch.rand(B, 4096, generator=torch.Generator().manual_seed(2)) < 0.5).to(torch.uint8)
    p = OM.init_params(1, torch.float32, bias_range=0.05)
    p["coarse/dense/dense_1/bias"] += 1.0
    p["fine/third/bias"] += 1.0
    return images, depths, mask, p


def packed_arena(p):
    a = Arena(msdn_specs(), "cpu", with_adam=False)
    a.load_tf(p)
    return a


def test_segment_table_matches_the_python_arena():
    net = CNet(2)
    a = Arena(msdn_specs(), "cpu", with_adam=False)
    segs = net.segments()
    assert list(segs) == list(a.specs) and net.total == a.total
    for name, s in a.specs.items():
        assert segs[name] == (s.offset, s.numel, tuple(s.packed_shape)), name
    net.close()


def c_step_and_python_step(B):
    """One phase-1 step of a fresh C net and of the Python host (same kernels, sequential schedule, no graph) from the same
    weights, inputs and dropout mask, checked against each other.  Returns what the oracle comparison needs."""
    images, depths, mask, p = make(B)
    a = packed_arena(p)
    im, dp, mk = images.to(DEV), depths.to(DEV), mask.to(DEV)
    net = CNet(B, beta2=0.999)
    net.load_packed(a.w.to(DEV))
    phase, losses = net.step(im, dp, mk)
    torch.cuda.synchronize()
    assert phase == 1 and net.lib.a3d_msdn_global_step(net.net) == 1
    op = models.msdn(im.clone(), dp.clone(), train=True, beta2=0.999, overlap=False)
    op.net.load_params(p)
    op.net.set_dropout_mask(mk)
    op.run(use_graph=False)
    torch.cuda.synchronize()
    lc, lf = float(losses[0]), float(losses[1])
    assert math.isfinite(lc) and math.isfinite(lf)
    assert abs(lc - float(op.net.loss_coarse)) <= 1e-4 * abs(lc) and abs(lf - float(op.net.loss_fine)) <= 1e-4 * abs(lf)
    cm, cw = net.view(net.m_ptr), net.view(net.w_ptr)
    lo, hi = a.group_range("CoarseDense")[0], a.group_range("CoarseConv")[1]
    assert cos(cm[lo:hi], op.net.arena.m[lo:hi]) > 0.9999               # split-K atomics: last-bit differences only
    assert cos(cw[lo:hi] - a.w[lo:hi].to(DEV), op.net.arena.w[lo:hi] - a.w[lo:hi].to(DEV)) > 0.99
    lo, hi = a.group_range("FineA")[0], a.group_range("FineB")[1]
    assert float(cm[lo:hi].abs().max()) == 0.0 and torch.equal(cw[lo:hi], a.w[lo:hi].to(DEV))    # phase 1: fine untouched
    return net, a, images, depths, mask, p, lc, lf, cm


def test_c_step_equals_python_step_and_oracle():
    c_step_equals_python_step_and_oracle(2)


def test_c_step_equals_python_step_and_oracle_above_fused_batch_limit():
    """batch 33, past the fused dense wgrad + TF-Adam kernel's batch limit: the C model runs the separate kernels."""
    c_step_equals_python_step_and_oracle(33)


def c_step_equals_python_step_and_oracle(B):
    net, a, images, depths, mask, p, lc, lf, cm = c_step_and_python_step(B)
    # ... and the float64 oracle at the BF16 storage points
    st = OM.TrainState({k: v.double() for k, v in p.items()}, beta2=0.999)
    out, _ = OM.train_step(st, images.double(), depths.double(), mask.double(), q=OM.bf16_round)
    assert abs(lc - float(out["loss_coarse"])) < 1e-2 * abs(lc) and abs(lf - float(out["loss_fine"])) < 1e-2 * abs(lf)
    got_m = a.export_tf(cm.cpu())
    for name in ("coarse/dense/dense_0/kernel", "coarse/conv/conv2d_1/kernel", "coarse/conv/conv2d_0/kernel",
                 "coarse/dense/dense_1/bias"):
        assert cos(got_m[name], st.m[name]) > 0.999, name
    net.close()


def test_c_step_at_the_largest_batch():
    """batch 256, the upper bound a3d_msdn_create accepts: phase 1 runs with finite losses and equals the Python step."""
    c_step_and_python_step(256)[0].close()


def test_c_phase2_and_inference():
    B = 2
    images, depths, mask, p = make(B)
    a = packed_arena(p)
    im, dp = images.to(DEV), depths.to(DEV)
    net = CNet(B, beta2=0.999)
    net.load_packed(a.w.to(DEV))
    t = (C.c_int * 4)(0, 0, 0, 0)
    L.check(net.lib.a3d_msdn_set_step(net.net, 2000000 // B, C.byref(t), None), "set_step")
    phase, losses = net.step(im, dp, mask.to(DEV))
    torch.cuda.synchronize()
    assert phase == 2
    cm = net.view(net.m_ptr)
    lo, hi = a.group_range("CoarseDense")[0], a.group_range("CoarseConv")[1]
    assert float(cm[lo:hi].abs().max()) == 0.0                          # coarse stack untouched in phase 2
    st = OM.TrainState({k: v.double() for k, v in p.items()}, beta2=0.999)
    st.global_step = 2000000 // B
    OM.train_step(st, images.double(), depths.double(), mask.double(), q=OM.bf16_round)
    got_m = a.export_tf(cm.cpu())
    for name in ("fine/first/conv2d/kernel", "fine/second/conv2d/kernel", "fine/third/kernel", "fine/first/conv2d/bias"):
        assert cos(got_m[name], st.m[name]) > 0.999, name
    # inference on a fresh net (train = 0): dropout off
    inet = CNet(B, train=False)
    inet.load_packed(a.w.to(DEV))
    fine, coarse = inet.infer(im)
    torch.cuda.synchronize()
    ref = OM.forward({k: v.double() for k, v in p.items()}, images.double(), depths.double(), None, False)
    rel = lambda x, y: float((x.double().cpu() - y.reshape(x.shape)).abs().max() / y.abs().max())
    assert rel(fine, ref["fine"]) < 1e-2 and rel(coarse, ref["coarse"]) < 1e-2
    net.close()
    inet.close()


def test_c_step_is_graph_capturable():
    """begin (host) + enqueue (captured): replays of the phase-1 graph advance global_step and keep the losses stable."""
    B = 2
    images, depths, mask, p = make(B)
    a = packed_arena(p)
    im, dp, mk = images.to(DEV), depths.to(DEV), mask.to(DEV)
    net = CNet(B)                                                      # reference Adam (beta2 = 1): weights frozen
    net.load_packed(a.w.to(DEV))
    _, l0 = net.step(im, dp, mk)                                       # first call: autotuning happens outside capture
    torch.cuda.synchronize()
    s = torch.cuda.Stream()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.stream(s):
        ph = net.lib.a3d_msdn_step_begin(net.net, C.c_void_p(s.cuda_stream))
        assert ph == 1
        with torch.cuda.graph(g, stream=s):
            L.check(net.lib.a3d_msdn_step_enqueue(net.net, 1, C.c_void_p(im.data_ptr()), C.c_void_p(dp.data_ptr()),
                                                  C.c_void_p(mk.data_ptr()), C.c_void_p(s.cuda_stream)), "enqueue")
        g.replay()
        assert net.lib.a3d_msdn_step_begin(net.net, C.c_void_p(s.cuda_stream)) == 1
        g.replay()
    torch.cuda.synchronize()
    assert net.lib.a3d_msdn_global_step(net.net) == 3
    lp = net.lib.a3d_msdn_losses(net.net)
    off = lp - net.ws.data_ptr()
    l2 = net.ws[off:off + 8].view(torch.float32)
    assert abs(float(l2[0]) - float(l0[0])) <= 1e-4 * abs(float(l0[0]))
    assert torch.equal(net.view(net.w_ptr), a.w.to(DEV))
    net.close()


def test_pure_c_host_runs_a_step():
    """examples/msdn_host.c: a host without Python (gcc + libcudart + liba3d.so) runs a train step and an inference."""
    import os
    import subprocess
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    exe = os.path.join(root, "examples", "msdn_host")
    if not os.path.exists(exe):
        subprocess.run(["make", "-C", os.path.join(root, "examples")], check=True)
    r = subprocess.run([exe, "2"], capture_output=True, text=True, timeout=300)
    print(r.stdout, r.stderr)
    assert r.returncode == 0, (r.returncode, r.stdout, r.stderr)
    assert "a3d_msdn_step: phase 1 global_step 1" in r.stdout


def test_c_dcnf_step_equals_python_step():
    """a3d_dcnf_create / _step / _infer over ctypes alone == the Python host's DCNF step (same kernels) and the oracle's
    loss on the same z (src/models.py:129-200)."""
    from ann3depth_b200.params import dcnf_specs
    from oracle import dcnf as OD
    lib = L.load()
    h = models.get_context(0).h
    B = 2
    g = torch.Generator().manual_seed(3)
    images = torch.rand(B, 480, 640, 3, generator=g).to(DEV)
    depths = (torch.rand(B, 480, 640, 1, generator=g) * 0.95 + 0.05).to(DEV)
    p = OD.init_params(5, torch.float32, bias_range=0.05, pairwise_nonneg=True)
    a = Arena(dcnf_specs(), "cpu", with_adam=False)
    a.load_tf(p)
    nbytes = lib.a3d_dcnf_workspace_bytes(h, B, 480, 640, 480, 640, 1)
    ws = torch.empty(nbytes, dtype=torch.uint8, device=DEV)
    net = C.c_void_p()
    L.check(lib.a3d_dcnf_create(h, B, 480, 640, 480, 640, 1, C.c_void_p(ws.data_ptr()), nbytes, None, C.byref(net)), "dcnf_create")
    L.check(lib.a3d_dcnf_configure(net, 0), "dcnf_configure")                  # stable loss form
    # segment table == the Python arena
    nseg = lib.a3d_dcnf_segment(net, -1, None, None, None, None)
    names = []
    for i in range(nseg):
        name, off, numel, shape = C.c_char_p(), C.c_size_t(), C.c_size_t(), (C.c_int * 4)()
        lib.a3d_dcnf_segment(net, i, C.byref(name), C.byref(off), C.byref(numel), C.byref(shape))
        s = a.specs[name.value.decode()]
        assert (off.value, numel.value, tuple(x for x in shape if x)) == (s.offset, s.numel, tuple(s.packed_shape))
        names.append(name.value.decode())
    assert names == list(a.specs)
    w_ptr, g_ptr, wb_ptr, total = C.c_void_p(), C.c_void_p(), C.c_void_p(), C.c_size_t()
    L.check(lib.a3d_dcnf_arena(net, C.byref(w_ptr), C.byref(g_ptr), C.byref(wb_ptr), C.byref(total)), "dcnf_arena")
    assert total.value == a.total

    def view(ptr):
        off = ptr.value - ws.data_ptr()
        return ws[off:off + total.value * 4].view(torch.float32)
    view(w_ptr).copy_(a.w)
    L.check(lib.a3d_dcnf_sync_weights(net, None), "sync")
    loss = torch.zeros(1, device=DEV)
    L.check(lib.a3d_dcnf_step(net, C.c_void_p(images.data_ptr()), C.c_void_p(depths.data_ptr()), C.c_void_p(loss.data_ptr()),
                              None), "dcnf_step")
    torch.cuda.synchronize()
    assert lib.a3d_dcnf_global_step(net) == 1
    # Python host, same kernels
    op = models.dcnf(images.clone(), depths.clone(), train=True, naive_loss=False)
    op.net.load_params(p)
    op.run()
    torch.cuda.synchronize()
    assert abs(float(loss) - float(op.net.loss)) <= 1e-4 * max(1.0, abs(float(op.net.loss)))
    lo, hi = a.group_range("SGD")
    assert cos(view(g_ptr)[lo:hi], op.net.arena.g[lo:hi]) > 0.9999
    assert cos(view(w_ptr)[lo:hi] - a.w[lo:hi].to(DEV), op.net.arena.w[lo:hi] - a.w[lo:hi].to(DEV)) > 0.9999
    lo, hi = a.group_range("Pairwise")
    assert torch.equal(view(w_ptr)[lo:hi], a.w[lo:hi].to(DEV))                  # no gradient reaches the pairwise layer
    # inference outputs
    out = torch.empty(B, 240, 320, device=DEV)
    z = torch.empty(B, 48, device=DEV)
    r = torch.empty(B, 48, device=DEV)
    L.check(lib.a3d_dcnf_infer(net, C.c_void_p(images.data_ptr()), C.c_void_p(out.data_ptr()), C.c_void_p(z.data_ptr()),
                               C.c_void_p(r.data_ptr()), None), "dcnf_infer")
    torch.cuda.synchronize()
    assert bool(torch.isfinite(out).all()) and float((r - op.net.r).abs().max()) < 1e-5
    ref_out = OD.T.resize_bilinear_tf1(z.cpu().double().reshape(B, 6, 8, 1), 240, 320)
    assert float((out.cpu().double() - ref_out.reshape(B, 240, 320)).abs().max()) < 1e-5
    lib.a3d_dcnf_destroy(net)
