"""bench.py contract checks that need no GPU: the reference arm (`--impl reference`) prints ONE JSON line with the keys
the driver reads, and the GPU arm refuses to run without a device instead of falling back to anything."""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_json_line():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0"],
                         capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.strip().splitlines() if l.startswith("{")]
    assert len(lines) == 1
    line = json.loads(lines[0])
    assert line["impl"] == "reference" and line["unit"] == "images/s" and line["higher_is_better"] is True
    assert line["value"] > 0 and line["n_gpus"] == 1 and line["steps"] == 1
    assert line["cpu_baseline"]["kind"] == "port" and line["cpu_baseline"]["cores"] >= 1
    assert line["cpu_baseline"]["value"] == line["value"] == line["e2e"]["value"]
    assert line["e2e"]["h2d_bytes_per_step"] == 0 and line["e2e"]["d2h_bytes_per_step"] == 0
    assert "workload" in line["config"] and "model" not in line["config"]


def test_dump_outputs_writes_float32_npy(tmp_path):
    """`--dump-outputs` format: one float32 .npy file per array the step gives its caller, values unchanged."""
    import types
    import numpy as np
    import torch
    sys.path.insert(0, ROOT)
    import bench
    g = torch.Generator().manual_seed(6)
    op = types.SimpleNamespace(losses={"loss/coarse_loss": torch.tensor([1.5]), "loss/fine_loss": torch.tensor([2.5])},
                               coarse=torch.rand(32, 55, 74, 1, generator=g), outputs=torch.rand(32, 55, 74, 1, generator=g))
    bench.dump_outputs(op, str(tmp_path), torch)
    assert sorted(os.listdir(tmp_path)) == ["coarse.npy", "fine.npy", "loss_coarse.npy", "loss_fine.npy"]
    for name, t in (("coarse", op.coarse), ("fine", op.outputs), ("loss_coarse", op.losses["loss/coarse_loss"]),
                    ("loss_fine", op.losses["loss/fine_loss"])):
        a = np.load(tmp_path / (name + ".npy"))
        assert a.dtype == np.float32
        np.testing.assert_array_equal(a, t.numpy())


def test_gpu_arm_needs_a_gpu():
    import torch
    if torch.cuda.is_available():
        import pytest
        pytest.skip("a GPU is present")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "1", "--warmup", "0", "--no-cpu-baseline"],
                         capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode != 0                       # no CPU / PyTorch fallback of the product path
    assert not [l for l in out.stdout.splitlines() if l.startswith("{")]
