"""bench.py on the GPU: `--steps` sets the timed steps, and `--dump-outputs` writes what the timed step computed, the same
(up to rounding) in every run with the same arguments."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def run_bench(out_dir):
    env = dict(os.environ, A3D_BENCH_U8="0")           # the uint8 e2e pass runs after the dump: not needed here
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--steps", "2", "--warmup", "0",
                          "--no-extra", "--no-cpu-baseline", "--dump-outputs", str(out_dir)],
                         capture_output=True, text=True, timeout=900, cwd=ROOT, env=env)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1 and json.loads(lines[0])["steps"] == 2
    return {n[:-4]: np.load(os.path.join(out_dir, n)) for n in os.listdir(out_dir)}


@pytest.mark.gpu
def test_bench_dump_outputs_reproducible(tmp_path):
    a, b = run_bench(tmp_path / "a"), run_bench(tmp_path / "b")
    assert sorted(a) == sorted(b) == ["coarse", "fine", "loss_coarse", "loss_fine"]
    assert a["loss_coarse"].shape == a["loss_fine"].shape == (1,)
    assert a["coarse"].shape == a["fine"].shape == (32, 55, 74, 1)
    for n in a:
        assert a[n].dtype == np.float32 and np.isfinite(a[n]).all() and np.abs(a[n]).max() > 0, n
        # bf16 activations and autotuned split-K sums: two runs agree to within one bf16 rounding unit of the scale
        assert np.abs(a[n].astype(np.float64) - b[n]).max() <= 2.0 ** -8 * np.abs(a[n]).max(), n
