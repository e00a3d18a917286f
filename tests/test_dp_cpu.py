"""CPU tests (gloo, world_size 2) of the data-parallel protocol and host-side layout logic.

The GPU path sum-allreduces flat gradient buckets with NCCL and folds 1/n into the optimizer
(ann3depth_b200/dp.py).  Here the same protocol runs over gloo with the CPU oracle as the per-rank
model: n ranks x batch B must equal one rank x batch n*B (SURVEY.md 8e)."""
import os
import subprocess
import sys

import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from ann3depth_b200.dp import DataParallel
from ann3depth_b200.params import Arena, msdn_specs, pack, unpack
from oracle import msdn as OM

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _batch(n, seed=0):
    g = torch.Generator().manual_seed(seed)
    images = torch.rand(n, 480, 640, 3, generator=g)
    depths = torch.rand(n, 55, 73, 1, generator=g) * 0.95 + 0.05
    mask = (torch.rand(n, 4096, generator=g) < 0.5).float()
    return images, depths, mask


def _params():
    p = OM.init_params(1, torch.float32, bias_range=0.05)
    p["coarse/dense/dense_1/bias"] += 1.0
    return p


def _worker(rank, world, port, out):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    torch.set_num_threads(2)
    images, depths, mask = _batch(world)
    p = _params()
    sl = slice(rank, rank + 1)                                    # shard: one sample per rank
    g, _ = OM.grads(p, images[sl], depths[sl], mask[sl], "coarse")
    # flat bucket in arena order, sum-allreduce, then the optimizer's grad_scale = 1/n
    names = [n for n in g]
    flat = torch.cat([g[n].reshape(-1) for n in names])
    dist.all_reduce(flat, op=dist.ReduceOp.SUM)
    flat *= 1.0 / world
    if rank == 0:
        torch.save({"names": names, "flat": flat}, out)
    dist.barrier()
    dist.destroy_process_group()


def test_dp_mean_of_rank_gradients_equals_big_batch(tmp_path):
    world, port = 2, 29531
    out = str(tmp_path / "dp.pt")
    mp.spawn(_worker, args=(world, port, out), nprocs=world, join=True)
    got = torch.load(out)
    images, depths, mask = _batch(world)
    ref, _ = OM.grads(_params(), images, depths, mask, "coarse")
    flat_ref = torch.cat([ref[n].reshape(-1) for n in got["names"]])
    cos = float(got["flat"] @ flat_ref / (got["flat"].norm() * flat_ref.norm()))
    assert cos > 0.99999
    assert float((got["flat"] - flat_ref).abs().max() / flat_ref.abs().max()) < 1e-3


class _Net:
    def __init__(self):
        self.arena = Arena(msdn_specs(), "cpu", with_adam=False)


def test_arena_layout_and_buckets():
    net = _Net()
    a = net.arena
    assert a.num_real_params() == 70877171                      # KA2
    # every segment 16-byte aligned in both the f32 and the bf16 view
    for s in a.specs.values():
        assert s.offset % 64 == 0 and s.size % 64 == 0
    # optimizer groups are contiguous, disjoint, and cover the arena in backward order
    order = ["CoarseDense", "CoarseConv", "FineA", "FineB"]
    pos = 0
    for g in order:
        lo, hi = a.group_range(g)
        assert lo == pos
        pos = hi
    assert pos == a.total
    br = DataParallel.bucket_range
    d1, d0, cc = br(net, "dense_1"), br(net, "dense_0"), br(net, "coarse_conv")
    assert d1[0] == 0 and d1[1] == d0[0] and d0[1] == cc[0]      # buckets become ready front to back
    assert br(net, "CoarseDense") == (d1[0], d0[1])
    fa, fb = a.group_range("FineA"), a.group_range("FineB")
    assert br(net, "fine") == (fa[0], fb[1])


def test_pack_unpack_roundtrip_and_masks():
    a = _Net().arena
    g = torch.Generator().manual_seed(0)
    for name in ("coarse/conv/conv2d_0/kernel", "fine/first/conv2d/kernel", "fine/first/conv2d/bias",
                 "coarse/dense/dense_1/kernel", "coarse/conv/conv2d_3/kernel"):
        s = a.specs[name]
        t = torch.rand(s.tf_shape, generator=g)
        assert torch.equal(unpack(s, pack(s, t)), t)
    m = a.masks["coarse/conv/conv2d_0/kernel"].view(96, 3, 3, 64)        # space-to-depth(4) packing of 11x11x3
    assert int(m.sum()) == 96 * 11 * 11 * 3 and not bool(m[..., 48:].any())
    assert not bool(m[:, 2, :, 36:48].any())                              # filter row 11 (= 4*2+3) does not exist
    m = a.masks["fine/first/conv2d/kernel"].view(64, 5, 5, 16)
    assert int(m.sum()) == 63 * 9 * 9 * 3 and not bool(m[63].any())
    assert "coarse/conv/conv2d_2/kernel" not in a.masks
    m = a.masks["coarse/conv/conv2d_1/kernel"].view(256, 5, 5, 128)      # input channels stored 96 -> 128
    assert int(m.sum()) == 256 * 5 * 5 * 96 and not bool(m[..., 96:].any())


def _gather_worker(rank, world, port, out):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    B, K, N = 4, 64, 48
    g = torch.Generator().manual_seed(10 + rank)
    x, dy = torch.randn(B, K, generator=g), torch.randn(B, N, generator=g)
    # activation-gather protocol of dp.dense_gather_adam_merged: gather the small matrices, update own rows only
    xs, dys = [torch.empty_like(x) for _ in range(world)], [torch.empty_like(dy) for _ in range(world)]
    dist.all_gather(xs, x)
    dist.all_gather(dys, dy)
    x_all, dy_all = torch.cat(xs), torch.cat(dys)
    r = N // world
    mine = (dy_all.t() @ x_all)[rank * r:(rank + 1) * r] / world
    # reference protocol: per-rank gradient, sum-allreduce, 1/n
    full = dy.t() @ x
    dist.all_reduce(full, op=dist.ReduceOp.SUM)
    full /= world
    rows = [torch.empty_like(mine) for _ in range(world)]
    dist.all_gather(rows, mine)                                   # = the all-gather of the updated weight rows
    if rank == 0:
        torch.save({"gathered": torch.cat(rows), "allreduced": full}, out)
    dist.barrier()
    dist.destroy_process_group()


def test_dense_activation_gather_equals_gradient_allreduce(tmp_path):
    """dW = dy^T x has rank B: all-gathering x and dy and updating one's own rows is the same update as the
    gradient sum-allreduce it replaces (dp.dense_gather_adam_merged)."""
    world, port = 2, 29532
    out = str(tmp_path / "gather.pt")
    mp.spawn(_gather_worker, args=(world, port, out), nprocs=world, join=True)
    got = torch.load(out)
    assert torch.allclose(got["gathered"], got["allreduced"], atol=1e-5)


def test_dense_gather_eligibility():
    net = _Net()
    dp = DataParallel.__new__(DataParallel)
    for world, ok in ((2, True), (4, True), (8, True), (3, False)):
        dp.world = world
        for k in ("coarse/dense/dense_1/kernel", "coarse/dense/dense_0/kernel"):
            assert dp.can_gather_dense(net, k, 32) is ok, (world, k)
    dp.world = 8
    assert not dp.can_gather_dense(net, "coarse/dense/dense_0/kernel", 64)       # gathered batch 512 > 256
    s = net.arena.specs["coarse/dense/dense_1/kernel"]
    assert s.packed_shape == (4096, 4096) and s.tf_shape == (4096, 4070)          # rows padded for equal slices
    t = torch.rand(4096, 4070)
    assert torch.equal(unpack(s, pack(s, t)), t) and float(pack(s, t)[4070:].abs().max()) == 0.0


def test_bench_reference_arm_other_ranks_are_silent():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2",
                        "--steps", "1", "--warmup", "0"], env=env, capture_output=True, text=True, timeout=120)
    assert r.returncode == 0 and r.stdout.strip() == ""


# ----------------------------------------------------------------------------- sharded optimizer state (gloo, world 2)
class _GlooCtx:
    """liba3d's in-place collectives (ops.Context.allreduce_sum / allgather / reduce_scatter_sum) over gloo."""

    def allreduce_sum(self, t, count=None):
        dist.all_reduce(t, op=dist.ReduceOp.SUM)

    def allgather(self, t, chunk):
        r = dist.get_rank()
        parts = [torch.empty(chunk, dtype=t.dtype) for _ in range(dist.get_world_size())]
        dist.all_gather(parts, t[r * chunk:(r + 1) * chunk].clone())
        t.copy_(torch.cat(parts))


def _fake_dp(rank, world):
    dp = DataParallel.__new__(DataParallel)
    dp.ctx, dp.rank, dp.world, dp.stream, dp._done, dp.bytes_per_step = _GlooCtx(), rank, world, None, [], 0
    return dp


def _shard_worker(rank, world, port, outdir):
    from ann3depth_b200 import ann3depth as drv
    from ann3depth_b200.params import dcnf_specs
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)

    class Net:
        pass
    net = Net()
    net.arena = a = Arena(dcnf_specs(), "cpu", with_adam=True)
    net.global_step, net.adam_t = 17, {"SGD": 17}
    op = type("Op", (), {"net": net})()
    dp = _fake_dp(rank, world)
    lo, hi = a.group_range("SGD")
    chunk = (hi - lo) // world
    truth = {k: torch.arange(a.total, dtype=torch.float32) * s for k, s in (("w", 1e-3), ("m", 2e-3), ("v", 3e-3))}
    own = slice(lo + rank * chunk, lo + (rank + 1) * chunk)
    for k in ("w", "m", "v"):                       # a sharded optimizer: only this rank's slice is current
        buf = getattr(a, k)
        buf.fill_(-1.0)
        buf[own] = truth[k][own]
        buf[:lo], buf[hi:] = truth[k][:lo], truth[k][hi:]     # outside the sharded bucket everything is replicated
    # 1. the f32 biases the kernels read become current on every rank (ADVICE r1: stale biases outside the own slice)
    dp._sync_sharded_biases(net, lo, hi, chunk)
    for s in a.specs.values():
        if s.kind == "bias" and lo <= s.offset < hi:
            got, exp = a.w[s.offset:s.offset + s.numel], truth["w"][s.offset:s.offset + s.numel]
            assert torch.equal(got, exp), (rank, s.name)
    # 2. a checkpoint taken under DP holds the owners' values of EVERY slice (gather_master before the chief writes)
    dp._sharded = {"SGD"}
    drv.save_checkpoint(op, outdir, comm=dp, write=rank == 0)
    dist.barrier()
    net2 = Net()
    net2.arena = Arena(dcnf_specs(), "cpu", with_adam=True)
    net2.global_step, net2.adam_t = 0, {"SGD": 0}
    assert drv.restore_checkpoint(type("Op", (), {"net": net2})(), outdir)
    for k in ("w", "m", "v"):
        # (padding entries of a packed segment are not variables and are not part of the checkpoint)
        exp_full = truth[k]
        got_tf = net2.arena.export_tf(getattr(net2.arena, k))
        exp_tf = {n: unpack(sp, a.view(exp_full, n)) for n, sp in a.specs.items()}
        for n in exp_tf:
            assert torch.equal(got_tf[n], exp_tf[n]), (rank, k, n)
    assert net2.global_step == 17 and net2.adam_t == {"SGD": 17}
    assert torch.equal(net2.arena.wb, net2.arena.w.to(torch.bfloat16))
    dist.barrier()
    dist.destroy_process_group()


def test_sharded_bias_sync_and_dp_checkpoint(tmp_path):
    world, port = 2, 29533
    mp.spawn(_shard_worker, args=(world, port, str(tmp_path)), nprocs=world, join=True)


def test_stop_consensus_single_process_passthrough():
    from ann3depth_b200.ann3depth import StopConsensus
    c = StopConsensus(1)
    assert c.decide(3, 10, True) == (10, True) and c.decide(4, 0, False) == (0, False)


def _stop_worker(rank, world, port, out):
    from ann3depth_b200.ann3depth import StopConsensus
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    c = StopConsensus(world, every=4)
    log = []
    for step in range(12):
        # rank 1 receives SIGUSR1 (10) "during" step 5; the chief's checkpoint timer fires at step 2
        sig = 10 if (rank == 1 and step >= 5) else 0
        due = rank == 0 and step >= 2
        s, ck = c.decide(step, sig, due)
        log.append((step, s, ck))
        if s:
            break
    torch.save(log, out + f".{rank}")
    dist.barrier()
    dist.destroy_process_group()


def test_stop_consensus_all_ranks_stop_at_the_same_step(tmp_path):
    world, port = 2, 29534
    out = str(tmp_path / "stop")
    mp.spawn(_stop_worker, args=(world, port, out), nprocs=world, join=True)
    a, b = torch.load(out + ".0"), torch.load(out + ".1")
    assert a == b                                             # identical decisions on both ranks
    assert a[-1] == (8, 10, True)                             # first consensus point after the signal: step 8
    assert (4, 0, True) in a and (0, 0, False) in a           # the chief's checkpoint request reaches rank 1 too
