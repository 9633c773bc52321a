"""bench.py --dump-outputs at a tiny size: the timed path's last generation is written as float arrays, the seeded inputs
make it reproducible, and --steps sets how many generations are timed."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")
if not torch.cuda.is_available():
    pytest.skip("needs a CUDA device", allow_module_level=True)

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
NAMES = ("theta", "gradient", "returns", "centered_ranks", "logits", "actions")


def _bench(out_dir, steps, warmup):
    cmd = [sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--steps", str(steps), "--warmup", str(warmup),
           "--pop", "8", "--episode-len", "3", "--noise-count", "6000000", "--no-cpu-baseline", "--dump-outputs", str(out_dir)]
    env = {k: v for k, v in os.environ.items() if k not in ("RANK", "WORLD_SIZE", "LOCAL_RANK")}
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=600, env=env)
    assert r.returncode == 0, r.stderr[-3000:]
    line = json.loads(r.stdout.strip().splitlines()[-1])
    return line, {n: np.load(os.path.join(out_dir, n + ".npy")) for n in NAMES}


def test_dump_outputs_reproducible_and_steps_timed(tmp_path):
    # the second generation is the last timed one in both runs: once after a warm-up generation, once with none
    one, a = _bench(tmp_path / "a", steps=1, warmup=1)
    two, b = _bench(tmp_path / "b", steps=2, warmup=0)
    assert one["steps"] == 1 and two["steps"] == 2 and two["e2e"]["value"] > 0
    # the library's launch counter covers the timed generations only
    assert abs(two["gpu_launches"] - 2 * one["gpu_launches"]) <= one["gpu_launches"] // 10
    assert sum(x.nbytes for x in a.values()) <= 64 << 20
    n_pairs, P = 4, 4_052_658
    assert a["theta"].shape == a["gradient"].shape == (P,)
    assert a["returns"].shape == a["centered_ranks"].shape == (n_pairs, 2)
    assert a["logits"].shape == (2 * n_pairs, 18) and a["actions"].shape == (2 * n_pairs,)
    for n in NAMES:
        assert a[n].dtype in (np.float32, np.float64) and np.isfinite(a[n]).all(), n
        np.testing.assert_array_equal(a[n], b[n], err_msg=n)          # fixed summation orders: bit-identical
