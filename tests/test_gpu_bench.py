"""bench.py --dump-outputs on the GPU: seeded inputs and weights, so two runs with the same arguments hand back the same
loss and parameters after exactly --steps timed steps."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ARGS = ["--gpus", "1", "--steps", "3", "--warmup", "1", "--no-cpu-baseline", "--no-large-batch", "--no-configs"]


def _bench(out_dir):
	res = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *ARGS, "--dump-outputs", str(out_dir)],
		capture_output=True, text=True, timeout=600)
	assert res.returncode == 0, res.stdout[-2000:] + res.stderr[-3000:]
	lines = res.stdout.strip().splitlines()
	assert len(lines) == 1, lines
	return json.loads(lines[0])


def test_bench_dump_outputs_repeat_bit_identically(tmp_path):
	a, b = _bench(tmp_path / "a"), _bench(tmp_path / "b")
	assert a["steps"] == b["steps"] == 3
	names = sorted(os.listdir(tmp_path / "a"))
	assert names == sorted(os.listdir(tmp_path / "b"))
	assert "loss.npy" in names and "param.layers.input.forward_weights.npy" in names
	for n in names:
		x, y = np.load(tmp_path / "a" / n), np.load(tmp_path / "b" / n)
		assert x.dtype == np.float32 and np.isfinite(x).all(), n
		assert np.array_equal(x, y), n
	assert float(np.load(tmp_path / "a" / "loss.npy")[0]) > 0.0
