"""Graphed training step with a user-defined surrogate against the built-in one.

Two configurations of bench.py's network (ALIF 784-128-10, recurrent, learn_beta, periodic encoder, T = 100): B = 256
(the headline step: lean BPTT sweep) and B = 4096 (tensor-core recurrence).  In each, one network trains with
HeavisideSigmoidApprox (the derivative evaluated inside the BPTT kernels) and one with a PyTorch restatement of the
same formula (evaluated once per step over the saved membrane trace by its own ``backward``, then streamed by the
sweep).  Both run as captured CUDA graphs on HBM-resident rasters; their timed windows alternate in one process.

	python tools/bench_custom_surrogate.py [--rounds 5 --steps 50]

Prints the device name and power limit, then per configuration the median step time of each variant (CUDA events).
"""
import argparse
import os
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

from snnimageclassification_b200 import SNN, FusedAdam, LayerType, ToSpikes, _cabi  # noqa: E402
from snnimageclassification_b200.modules.spike_funcs import HeavisideSigmoidApprox, SpikeFunction  # noqa: E402


class RestatedFastSigmoid(SpikeFunction):
	@staticmethod
	def backward(ctx, grad):
		v, thr, gamma = ctx.saved_tensors
		return grad / (gamma * (v - thr).abs() + 1.0) ** 2, None, None


def power_limit() -> str:
	try:
		out = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
			capture_output=True, text=True, timeout=30)
		return out.stdout.strip() or "unknown"
	except (OSError, subprocess.SubprocessError):
		return "unknown"


def build(func, B, T, dev, pool=2):
	torch.manual_seed(0)
	enc = ToSpikes(T, use_periods=True)
	net = SNN(784, 10, 128, use_recurrent_connection=True, int_time_steps=T, spike_func=func,
		hidden_layer_type=LayerType.ALIF, device=dev, learn_beta=True, input_encoder=enc)
	net.train()
	opt = FusedAdam(net.parameters(), lr=1e-3, weight_decay=1e-5)
	crit = torch.nn.NLLLoss()
	g = torch.Generator().manual_seed(1)
	steps = []
	for _ in range(pool):
		img = (torch.randint(1, 256, (B, 784), generator=g).float() / 255.0) * (torch.rand(B, 784, generator=g) < 0.19)
		x = enc.encode_batch(img.to(dev))
		y = torch.randint(0, 10, (B,), generator=g).to(dev)
		steps.append(net.graphed_train_step(x, y, crit, opt, static_inputs=True))
	return steps


def timed(steps, n):
	e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
	torch.cuda.synchronize()
	e0.record()
	for i in range(n):
		steps[i % len(steps)]()
	e1.record()
	torch.cuda.synchronize()
	return e0.elapsed_time(e1) / n


def main():
	ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
	ap.add_argument("--rounds", type=int, default=5)
	ap.add_argument("--steps", type=int, default=50)
	ap.add_argument("--T", type=int, default=100)
	ap.add_argument("--batches", type=int, nargs="+", default=[256, 4096])
	a = ap.parse_args()
	dev = torch.device("cuda:0")
	_cabi.require_b200(dev)
	print(f"device: {torch.cuda.get_device_name(dev)}, power limit {power_limit()}")
	for B in a.batches:
		variants = {"built-in FastSigmoid": build(HeavisideSigmoidApprox, B, a.T, dev),
			"restated FastSigmoid (sigma' trace)": build(RestatedFastSigmoid, B, a.T, dev)}
		for steps in variants.values():
			timed(steps, 10)          # warm-up
		times = {k: [] for k in variants}
		for _ in range(a.rounds):     # alternate the variants' timed windows
			for k, steps in variants.items():
				times[k].append(timed(steps, a.steps))
		print(f"B = {B}, T = {a.T} ({a.rounds} rounds x {a.steps} graphed steps):")
		for k, ts in times.items():
			ts = sorted(ts)
			print(f"  {k:38s} median {ts[len(ts) // 2]:.4f} ms/step  (min {ts[0]:.4f}, max {ts[-1]:.4f})")


if __name__ == "__main__":
	main()
