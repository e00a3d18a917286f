"""CPU tests of the evaluation layer: the float64 metric oracle on known answers, the single-pass test-split reader
(order, partial last batch, shards, errors), the cross-rank reduction of `evaluate.DepthMetrics` over gloo, and the
driver's --evalfreq default."""
import os
import struct

import numpy as np
import pytest
import torch

from ann3depth_b200 import data
from ann3depth_b200.evaluate import DepthMetrics
from oracle import metrics as OM

from test_data_cpu import _example, _write


def _gt(seed=0, shape=(30, 40)):
    rng = np.random.default_rng(seed)
    return rng.integers(1, 256, size=shape).astype(np.float32) / np.float32(255.0)


def _metrics(pairs, median=False):
    return OM.dataset_metrics(np.stack([OM.image_sums(p, g, median=median)[0] for p, g in pairs]))


def test_oracle_perfect_prediction():
    g = _gt()
    r = _metrics([(g, g)])
    for k in ("abs_rel", "sq_rel", "rmse", "rmse_log", "log10", "silog"):
        assert r[k] == 0.0, k
    assert r["delta1"] == r["delta2"] == r["delta3"] == 1.0
    assert r["pixels"] == g.size and r["images"] == 1 and r["nonfinite"] == 0


@pytest.mark.parametrize("c", [0.5, 0.9, 1.2, 1.3])
def test_oracle_constant_factor(c):
    g = _gt(1) * np.float32(0.5) + np.float32(0.1)                 # c * g stays inside (1e-3, 1]
    p = (g.astype(np.float64) * c).astype(np.float32)
    r = _metrics([(p, g)])
    assert r["abs_rel"] == pytest.approx(abs(c - 1), rel=1e-5)
    assert r["rmse_log"] == pytest.approx(abs(np.log(c)), rel=1e-5)
    assert r["silog"] == pytest.approx(0.0, abs=1e-6)
    assert r["delta1"] == (1.0 if max(c, 1 / c) < 1.25 else 0.0)


def test_oracle_median_scaling_removes_a_constant_factor():
    g = _gt(2) * np.float32(0.5) + np.float32(0.1)
    p = g * np.float32(0.6)
    r = _metrics([(p, g)], median=True)
    for k in ("abs_rel", "sq_rel", "rmse", "rmse_log", "log10", "silog"):
        assert r[k] == pytest.approx(0.0, abs=1e-6), k
    assert r["delta1"] == 1.0
    _, s = OM.image_sums(p, g, median=True)
    assert s == np.float32(np.sort(g.ravel())[(g.size - 1) // 2]) / np.float32(np.sort(p.ravel())[(p.size - 1) // 2])


def test_oracle_all_invalid_image_contributes_nothing():
    g = _gt(3)
    bad = np.zeros_like(g)                                          # exact zeros: excluded by min_depth
    sums, s = OM.image_sums(np.full_like(g, np.nan), bad, median=True)
    assert not sums.any() and s == 1.0
    both = _metrics([(g * np.float32(1.1), g), (g, bad)])
    one = _metrics([(g * np.float32(1.1), g)])
    assert both["images"] == 2 and both["pixels"] == one["pixels"]
    for k in OM.METRICS:
        assert both[k] == one[k] and np.isfinite(both[k]), k


def test_oracle_nonfinite_prediction_maps_to_min_depth():
    g = _gt(4)
    p = g.copy()
    p[0, :5] = np.nan
    p[1, :2] = np.inf
    sums, _ = OM.image_sums(p, g)
    assert sums[10] == 7
    ref, _ = OM.image_sums(np.where(np.isnan(p), np.float32(1e-3), np.minimum(p, 1.0)).astype(np.float32), g)
    assert np.allclose(sums[:10], ref[:10])


def _split(tmp_path, n, dhw=(2, 3), corrupt=None):
    recs = []
    for i in range(n):
        img = np.full((4, 6, 3), (i + 1) / 255. - .5, dtype=np.float32)
        dep = np.full((*dhw, 1), (i + 1) / 510. - .5, dtype=np.float32)
        if i == corrupt:
            dep = dep[:, :-1]                                       # payload of the wrong size: the parse must fail
        recs.append(_example({"image_height": 4, "image_width": 6, "image_channels": 3, "depth_height": dhw[0],
                              "depth_width": dhw[1], "depth_channels": 1, "image": img.tobytes(),
                              "depth": np.ascontiguousarray(dep).tobytes()}, True))
    os.makedirs(tmp_path / "nyu", exist_ok=True)
    _write(tmp_path / "nyu" / "test.tfrecords", recs)
    return str(tmp_path)


def _drain(inp):
    out = []
    while True:
        n = inp.next_batch()
        ids = torch.round(inp.images[:, 0, 0, 0] * 255).long()[:n].tolist()
        out.append((n, [i - 1 for i in ids]))
        if n == 0:
            return out


def test_test_split_reader_order_and_partial_batch(tmp_path):
    inp = data.inputs(_split(tmp_path, 5), "nyu", 2, "test", epochs=1, device="cpu")
    got = _drain(inp)
    assert [n for n, _ in got] == [2, 2, 1, 0]
    assert [i for _, ids in got for i in ids] == [0, 1, 2, 3, 4]
    assert inp.next_batch() == 0                                    # stays at the end
    inp.close()


def test_test_split_reader_shards(tmp_path):
    root = _split(tmp_path, 5)
    seen = []
    for r in range(2):
        inp = data.inputs(root, "nyu", 2, "test", epochs=1, shard=(r, 2), device="cpu")
        seen.append([i for _, ids in _drain(inp) for i in ids])
        inp.close()
    assert seen == [[0, 2, 4], [1, 3]]


def test_test_split_reader_errors_raise(tmp_path):
    with pytest.raises(FileNotFoundError):
        data.inputs(str(tmp_path), "none", 2, "test", epochs=1, device="cpu")
    inp = data.inputs(_split(tmp_path, 5, corrupt=3), "nyu", 2, "test", epochs=1, device="cpu")
    with pytest.raises(Exception):
        for _ in range(4):
            inp.next_batch()
    with pytest.raises(Exception):                                  # the reader is gone: raise again, do not hang
        inp.next_batch()
    inp.close()


def _image_sums(k, seed=5):
    rng = np.random.default_rng(seed)
    out = []
    for i in range(k):
        g = _gt(10 + i)
        if i == 2:
            g[:] = 0.0                                              # no valid pixel
        p = (g * rng.uniform(0.7, 1.4, size=g.shape)).astype(np.float32)
        out.append(OM.image_sums(p, g)[0])
    return np.stack(out)


def _gloo_worker(rank, world, port, sums, q):
    import torch.distributed as dist
    dist.init_process_group("gloo", init_method=f"tcp://127.0.0.1:{port}", rank=rank, world_size=world)
    m = DepthMetrics(None)
    m.add_sums(torch.from_numpy(sums[rank::world]))
    m.reduce()
    q.put((rank, m.result()))
    dist.destroy_process_group()


def test_depth_metrics_two_rank_reduce_matches_single_process():
    import socket
    import torch.multiprocessing as mp
    sums = _image_sums(5)
    single = DepthMetrics(None)
    single.add_sums(torch.from_numpy(sums))
    ref = single.result()
    oracle = OM.dataset_metrics(sums)
    for k in OM.METRICS:
        assert ref[k] == pytest.approx(oracle[k], rel=1e-12), k
    assert ref["images"] == 5 and ref["pixels"] == oracle["pixels"]
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        port = s.getsockname()[1]
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    procs = [ctx.Process(target=_gloo_worker, args=(r, 2, port, sums, q)) for r in range(2)]
    for p in procs:
        p.start()
    res = dict(q.get(timeout=120) for _ in procs)
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    for r in range(2):
        for k, v in ref.items():
            assert res[r][k] == pytest.approx(v, rel=1e-12), (r, k)


def test_evalfreq_defaults_to_off():
    from ann3depth_b200.ann3depth import parse_args
    assert parse_args(["nyu"]).evalfreq == 0
    assert parse_args(["nyu", "--evalfreq", "50"]).evalfreq == 50
