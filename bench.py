#!/usr/bin/env python
"""bench.py -- train samples/sec (fwd + BPTT), ALIF 784-128-10 recurrent, batch 256 per GPU, T = 100.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl native|reference] [--dump-outputs DIR]

One step = one pass of the hot path over one batch: input projection, fused recurrence + readout, fused
max-over-time/log-softmax/NLL head, reverse-time BPTT, weight-gradient contraction, [gradient all-reduce],
Adam step (reference snn.py:384-415).  Reported on the ONE JSON line:

  value       whole-job samples/s with the spike rasters already resident in HBM (device-timed, max over ranks)
  e2e         the same metric through the public API (SNN._exec_batch) from PINNED HOST images: H2D copy, GPU
              spike encoder, train step, loss read-back -- every step, inside the timed region
  roofline    the dominant kernel's algorithmic bytes / its CUDA-event duration against the measured HBM peak
  cpu_baseline the CPU restatement of the reference (oracle/torch_port.py) timed on this box's host cores

--impl reference times that CPU restatement alone (the reference itself is pure Python and cannot travel to the
GPU box; oracle/torch_port.py is pinned against it by tests/test_oracle_golden.py).

--dump-outputs DIR writes what the timed resident step handed its caller after the last of the K timed steps -- the
batch loss and every updated parameter -- as DIR/<name>.npy (float32).  Inputs and initial weights are seeded, so two
builds run with the same arguments can be compared output for output.
"""
import argparse
import json
import os
import sys
import threading
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

B_PER_GPU, T, N, H, O = 256, 100, 784, 128, 10
WORKLOAD = "ALIF 784-128-10 recurrent, learn_beta, periodic to_spikes (tau=0.02), batch 256/GPU, T=100, FastSigmoid"
METRIC = "train samples/sec (fwd+BPTT) ALIF H=128"
N_POOL = 4   # rotating input batches: 4 x 80 MB of rasters > 126 MB L2, so no step finds its input in L2


def synthetic_images(n, seed):
	"""MNIST-shaped images: k/255 levels with ink probability 0.19 (SURVEY.md 8d), uniform labels."""
	g = torch.Generator().manual_seed(seed)
	img = (torch.randint(1, 256, (n, N), generator=g).float() / 255.0) * (torch.rand(n, N, generator=g) < 0.19)
	return img, torch.randint(0, O, (n,), generator=g)


# ---------------------------------------------------------------------------------------------------------------------
class ClockSampler(threading.Thread):
	"""Samples SM clocks and throttle reasons through NVML while the timed region runs."""
	REASONS = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown", 0x4: "sw_power_cap",
		0x80: "hw_power_brake_slowdown"}

	def __init__(self, index):
		super().__init__(daemon=True)
		self.index, self.samples, self.reasons, self.max_mhz, self._stop_evt = index, [], set(), None, threading.Event()
		try:
			import pynvml
			pynvml.nvmlInit()
			self.nv = pynvml
			self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
			self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
		except Exception:
			self.nv = None

	def run(self):
		while self.nv is not None and not self._stop_evt.is_set():
			try:
				self.samples.append(self.nv.nvmlDeviceGetClockInfo(self.h, self.nv.NVML_CLOCK_SM))
				mask = self.nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
				for bit, name in self.REASONS.items():
					if mask & bit:
						self.reasons.add(name)
			except Exception:
				pass
			time.sleep(0.0005)     # the timed region is a few tens of milliseconds long

	def stop(self):
		self._stop_evt.set()
		self.join(timeout=2)
		return {"sm_mhz": float(np.median(self.samples)) if self.samples else None, "sm_max_mhz": self.max_mhz,
			"reasons": sorted(self.reasons), "samples": len(self.samples)}


# ---------------------------------------------------------------------------------------------------------------------
def cpu_reference_run(steps, warmup, budget_s=150.0):
	"""Times oracle/torch_port.py (the reference's algorithm as PyTorch-CPU ops + autograd) on the host cores."""
	from oracle.torch_port import TorchPortSNN
	import oracle
	cores = os.cpu_count() or 1
	torch.set_num_threads(cores)
	net = TorchPortSNN(N, H, O, T, layer_type=1, surrogate=0, recurrent=True, learn_beta=True, seed=0)
	opt = torch.optim.Adam(net.parameters(), lr=1e-3, weight_decay=1e-5)
	img, labels = synthetic_images(B_PER_GPU, seed=0)
	x = torch.from_numpy(oracle.encode(img.numpy(), T, None, tau=0.02, thr=0.2, periodic=True, eps=1e-7)).float()
	t0 = time.perf_counter()
	net.exec_batch(x, labels, opt)
	first = time.perf_counter() - t0
	b = B_PER_GPU
	if first * (steps + warmup) > budget_s:      # keep the whole run within a few minutes: bound the sample
		b = max(8, int(B_PER_GPU * budget_s / (first * (steps + warmup))))
		x, labels = x[:b], labels[:b]
	for _ in range(max(warmup - 1, 0)):
		net.exec_batch(x, labels, opt)
	t0 = time.perf_counter()
	for _ in range(steps):
		net.exec_batch(x, labels, opt)
	dt = time.perf_counter() - t0
	return {"value": b * steps / dt, "ms_per_step": 1e3 * dt / steps, "cores": cores, "batch": b, "steps": steps}


def base_config(world):
	"""The keys both arms print (the driver compares them): what the workload IS, nothing about how an arm runs it."""
	return {"workload": WORKLOAD, "global_batch": world * B_PER_GPU, "parallelism": f"dp{world}",
		"l2": f"{N_POOL} rotating input batches ({N_POOL * B_PER_GPU * T * N * 4 >> 20} MiB) > 126 MB L2",
		"optimizer": "Adam(lr=1e-3, weight_decay=1e-5)"}


def reference_arm(args, rank):
	if rank != 0:
		return
	world = int(os.environ.get("WORLD_SIZE", "1"))
	r = cpu_reference_run(args.steps, max(args.warmup, 1))
	sample = f"{r['steps']} train steps of batch {r['batch']} (of {B_PER_GPU}), T={T}, rasters resident in host memory"
	print(json.dumps({
		"impl": "reference", "metric": METRIC, "value": r["value"], "unit": "samples/s", "n_gpus": args.gpus,
		"steps": args.steps, "warmup": args.warmup, "ms_per_step": r["ms_per_step"], "higher_is_better": True,
		"scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
		"config": base_config(world), "details": {"batch_per_step": r["batch"]},
		"cpu_baseline": {"value": r["value"], "unit": "samples/s", "cores": r["cores"], "kind": "port", "sample": sample},
		"e2e": {"value": r["value"], "unit": "samples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
	}))


# ---------------------------------------------------------------------------------------------------------------------
def main():
	ap = argparse.ArgumentParser()
	ap.add_argument("--gpus", type=int, default=1)
	ap.add_argument("--steps", type=int, default=400)
	ap.add_argument("--warmup", type=int, default=20)
	ap.add_argument("--impl", default="native", choices=["native", "reference"])
	ap.add_argument("--no-cpu-baseline", action="store_true")
	ap.add_argument("--no-large-batch", action="store_true")
	ap.add_argument("--no-configs", action="store_true", help="skip the c1/c3/c4/c5 sub-lines")
	ap.add_argument("--quick-sweep", action="store_true", help="c5: ALIF and T in {10, 100} only")
	ap.add_argument("--dump-outputs", metavar="DIR",
		help="write the loss and the parameters after the last timed step as DIR/<name>.npy")
	args = ap.parse_args()
	if args.steps < 1:
		ap.error("--steps must be at least 1")
	args.warmup = max(args.warmup, 3)

	rank = int(os.environ.get("RANK", "0"))
	world = int(os.environ.get("WORLD_SIZE", "1"))
	local_rank = int(os.environ.get("LOCAL_RANK", "0"))
	if args.impl == "reference":
		reference_arm(args, rank)
		return

	import torch.distributed as dist
	from snnimageclassification_b200 import SNN, FusedAdam, LayerType, SpikeFuncType, ToSpikes, _cabi
	dev = torch.device("cuda", local_rank)
	torch.cuda.set_device(dev)
	_cabi.require_b200(dev)          # fails loudly: no fallback
	if world > 1:
		dist.init_process_group("nccl", device_id=dev)

	torch.manual_seed(0)             # same initial weights on every rank
	enc = ToSpikes(T, use_periods=True)      # production encoder settings (tau = 0.02, datasets.py:21)
	net = SNN(N, O, H, use_recurrent_connection=True, int_time_steps=T, spike_func=SpikeFuncType.FastSigmoid,
		hidden_layer_type=LayerType.ALIF, device=dev, learn_beta=True, input_encoder=enc)
	opt = FusedAdam(net.parameters(), lr=1e-3, weight_decay=1e-5)    # torch.optim.Adam semantics, one libsnnk launch
	dp_fused = world > 1 and os.environ.get("SNNK_DP_FUSED", "1") != "0" and opt.enable_data_parallel()
	crit = torch.nn.NLLLoss()
	net.train()

	pool_img, pool_lab = [], []
	for i in range(N_POOL):
		img, lab = synthetic_images(B_PER_GPU, seed=1000 * rank + i)
		pool_img.append(img.pin_memory()); pool_lab.append(lab.pin_memory())
	rasters = [enc.encode_batch(img.to(dev)) for img in pool_img]       # (B,T,N) fp32 resident in HBM
	labels_dev = [lab.to(dev) for lab in pool_lab]

	# one captured CUDA graph per resident batch (forward, fused head, BPTT, weight gradients, [all-reduce], Adam)
	graphs = [net.graphed_train_step(rasters[i], labels_dev[i], crit, opt, static_inputs=True) for i in range(N_POOL)]

	def step_resident(i):
		return graphs[i % N_POOL]()

	def step_eager(i):
		loss = net.batch_loss(rasters[i % N_POOL], labels_dev[i % N_POOL], crit)
		opt.zero_grad()
		loss.backward()
		net._allreduce_gradients(opt)
		opt.step()
		return loss

	def barrier():
		if world > 1:
			dist.barrier()
		torch.cuda.synchronize()

	def timed(fn, steps):
		barrier()
		e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
		e0.record()
		for i in range(steps):
			fn(i)
		e1.record()
		barrier()
		ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
		if world > 1:
			dist.all_reduce(ms, op=dist.ReduceOp.MAX)
		return float(ms.item())

	for i in range(args.warmup):
		step_resident(i)
	sampler = ClockSampler(local_rank)
	sampler.start()
	for i in range(50):         # the same steps, untimed, while the sampler thread comes up: the GPU is under this load when
		step_resident(i)        # the first NVML query returns (a 30 ms timed region alone sometimes caught a single sample)
	ms = timed(step_resident, args.steps)
	clocks = sampler.stop()
	if args.dump_outputs and rank == 0:      # before the measurements below train the same network further
		dump_outputs(args.dump_outputs, graphs[(args.steps - 1) % N_POOL].loss, net)
	timeline = None
	if dp_fused:     # last resident step on every rank, rank-local device clocks, us since kernel start
		timeline = [None] * world
		dist.all_gather_object(timeline, [round(v, 2) for v in opt.exchange_timeline()[0]])
	value = world * B_PER_GPU * args.steps / (ms * 1e-3)

	# The production encoder repeats frames, which the library exploits (frame-dedup variant, SURVEY.md 8f.1).  For
	# inputs that do NOT repeat, the same rasters without their run tables go through the dense kernels: reported
	# beside the headline so that nobody mistakes the shortcut for kernel speed.
	from snnimageclassification_b200.modules.functional import get_runs, mark_binary
	tab = get_runs(rasters[0])
	dedup = {"active": bool(tab is not None and int(tab[1]) == 1),
		"runs_per_sample": (float(tab[0]) / B_PER_GPU) if tab is not None else None}
	dense_rasters = [mark_binary(r.clone()) for r in rasters]
	dense_graphs = [net.graphed_train_step(dense_rasters[i], labels_dev[i], crit, opt, static_inputs=True)
		for i in range(N_POOL)]
	def step_dense(i):
		return dense_graphs[i % N_POOL]()
	for i in range(args.warmup):
		step_dense(i)
	ms_dense = timed(step_dense, args.steps)
	dedup["value_dense_kernels"] = world * B_PER_GPU * args.steps / (ms_dense * 1e-3)
	dedup["ms_per_step_dense_kernels"] = ms_dense / args.steps
	del dense_graphs, dense_rasters
	# ... and the same batches as BIT-PACKED rasters resident in HBM (2.5 MB instead of 80 MB per batch): the projection
	# and weight-gradient GEMMs expand the words in shared memory (SNNK_F_INPUT_BITS; no run table: dense kernels)
	from snnimageclassification_b200.modules.functional import mark_bits
	packed_rasters = [mark_bits(enc.encode_batch_bits(img.to(dev)), N) for img in pool_img]
	packed_graphs = [net.graphed_train_step(packed_rasters[i], labels_dev[i], crit, opt, static_inputs=True) for i in range(N_POOL)]
	def step_packed(i):
		return packed_graphs[i % N_POOL]()
	for i in range(args.warmup):
		step_packed(i)
	ms_packed = timed(step_packed, args.steps)
	packed = {"value": world * B_PER_GPU * args.steps / (ms_packed * 1e-3), "ms_per_step": ms_packed / args.steps,
		"input": "bit-packed rasters (B,T,25) int32 resident in HBM, dense kernels k_proj_bits / k_wgrad_bits"}
	del packed_graphs

	# end to end through the public API: pinned host images -> H2D -> GPU encoder -> train step -> loss read-back
	def step_e2e(i):
		return net._exec_batch(pool_img[i % N_POOL], pool_lab[i % N_POOL], crit, opt)
	for i in range(3):
		step_e2e(i)
	ms_e2e = timed(step_e2e, args.steps)
	e2e = world * B_PER_GPU * args.steps / (ms_e2e * 1e-3)
	h2d = B_PER_GPU * N * 4 + B_PER_GPU * 8

	# the same from pinned host RASTERS (what a reference DataLoader would hand over): H2D of 80 MB per step
	host_rasters = [r.cpu().pin_memory() for r in rasters[:2]]
	net.input_encoder = None
	def step_e2e_raster(i):
		return net._exec_batch(host_rasters[i % 2], pool_lab[i % 2], crit, opt)
	for i in range(2):
		step_e2e_raster(i)
	ms_r = timed(step_e2e_raster, max(args.steps // 5, 3))
	e2e_raster = world * B_PER_GPU * max(args.steps // 5, 3) / (ms_r * 1e-3)
	# ... and from pinned host rasters in the bit-packed format (SNNK_BITS, 1/32 of the bytes; unpacked on the device)
	host_bits = [enc.encode_batch_bits(pool_img[i].to(dev)).cpu().pin_memory() for i in range(2)]
	def step_e2e_bits(i):
		return net._exec_batch(host_bits[i % 2], pool_lab[i % 2], crit, opt)
	for i in range(3):
		step_e2e_bits(i)
	ms_b = timed(step_e2e_bits, args.steps)
	e2e_bits = world * B_PER_GPU * args.steps / (ms_b * 1e-3)
	net.input_encoder = enc

	# per-kernel CUDA-event timing (separate short loop, same process) -> roofline of the dominant kernel
	kern = profile_kernels(step_eager)     # event brackets need real launches, not a graph replay

	big = None
	if world == 1 and not args.no_large_batch:
		big = large_batch_rooflines(net, enc, dev)
	# the other BASELINE configurations (c1, c3 and the inference sweep c5 on one GPU; c4 = 512 rows per GPU at every N)
	configs = {}
	if not args.no_configs:
		sub_steps = max(10, min(args.steps, 100))
		for spec in TRAIN_CONFIGS:
			if world > 1 and not spec["multi_gpu"]:
				continue
			st = sub_steps if spec["H"] <= 128 else max(5, sub_steps // 5)
			configs[spec["key"]] = run_train_config(spec, dev, world, rank, st, max(3, args.warmup // 4), timed, dp=True)
		if world == 1:
			configs["c5"] = run_inference_sweep(dev, quick=args.quick_sweep)
	if rank != 0:
		finish(world)
		return
	peaks = {}
	try:
		peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
	except Exception:
		pass
	peak_hbm = float(peaks.get("hbm_gbs", 6650.0))
	# dominant kernel = largest per-step time among the kernels that move the step's data; the optimizer launch is
	# left out: in a data-parallel run its duration is mostly the wait for the slowest peer, not work
	cand = {k: v for k, v in kern.items() if v["bytes"] > 0 and not k.startswith("k_adam")}
	top = max(cand, key=lambda k: cand[k]["ms_per_step"]) if cand else None
	roofline = None
	if top:
		ach = kern[top]["bytes"] / (kern[top]["ms"] * 1e-3) / 1e9
		ev = ncu_evidence(top.split()[0])
		smem_peak = 148 * 128 * float(peaks.get("sm_max_mhz", 1965.0)) * 1e6 / 1e9      # GB/s: 128 B/cycle/SM
		smem_gbs = (ev["smem_wavefronts"] * 128 / (kern[top]["ms"] * 1e-3) / 1e9) if (ev and ev.get("smem_wavefronts")) else None
		roofline = {"bound": "hbm", "achieved": ach, "peak": peak_hbm, "unit": "GB/s", "frac": ach / peak_hbm,
			"traffic": ev["traffic"] if ev else None, "kernel": top, "peak_source": "measured" if peaks else "fallback",
			"kernel_ms": kern[top]["ms"], "algorithmic_bytes": kern[top]["bytes"],
			"traffic_source": (f"{ev['source']} ({ev['kernel'][:60]})" if ev else None),
			"smem_achieved": smem_gbs, "smem_peak": smem_peak,
			"smem_frac": (smem_gbs / smem_peak) if smem_gbs else None,
			"smem_note": "shared-memory wavefronts x 128 B (ncu, per launch) / this run's kernel time, against 128 B/cycle/SM",
			"all_kernels": {k: {"ms_per_step": round(v["ms_per_step"], 4), "launches_per_step": v["launches_per_step"],
				"GBps": round(v["bytes"] / (v["ms_per_step"] * 1e-3) / 1e9, 1)} for k, v in kern.items()}}
	launches_per_step = sum(v["launches_per_step"] for v in kern.values()) if kern else 0
	# the profiler brackets the kernels that matter for time; three small helpers of a step carry no bracket:
	# k_split_w, k_prep_rec (forward) and, with the dedup variant, the backward gather on the helper stream
	launches_per_step += 2 + (1 if dedup["active"] else 0)
	cpu = None
	if world == 1 and not args.no_cpu_baseline:
		r = cpu_reference_run(steps=40, warmup=2, budget_s=25.0)
		cpu = {"value": r["value"], "unit": "samples/s", "cores": r["cores"], "kind": "port",
			"sample": f"{r['steps']} train steps of batch {r['batch']} (of {B_PER_GPU}), T={T}, oracle/torch_port.py"}
	print(json.dumps({
		"metric": METRIC, "value": value, "unit": "samples/s", "n_gpus": world, "steps": args.steps,
		"warmup": args.warmup, "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak",
		"vs_baseline": None, "dtype": "f32", "data": "synthetic",
		"config": base_config(world),
		"details": {"optimizer_kernel": "snnk_adam_step (one launch for all tensors)", "launch": "one CUDA graph per step",
			"frame_dedup": dedup, "packed_input": packed,
			"grad_exchange": ("none (1 rank)" if world == 1 else
				"fused into snnk_adam_step_dp over NVLink peer memory" if dp_fused else "NCCL all-reduce (mean)"),
			"exchange_timeline_us": ({"columns": ["stores_issued", "peers_seen", "done"], "per_rank": timeline}
				if dp_fused else None)},
		"clocks": clocks,
		"e2e": {"value": e2e, "unit": "samples/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": 8,
			"readback": "the step's loss, posted by the head kernel as one 8-byte word into pinned host memory and polled by the host",
			"ms_per_step": ms_e2e / args.steps, "input": "pinned host images (B,784) fp32 + labels; GPU to_spikes",
			"from_host_rasters": {"value": e2e_raster, "h2d_bytes_per_step": B_PER_GPU * T * N * 4 + B_PER_GPU * 8},
			"from_host_bitpacked_rasters": {"value": e2e_bits,
				"h2d_bytes_per_step": B_PER_GPU * T * ((N + 31) // 32) * 4 + B_PER_GPU * 8}},
		"gpu_launches": int(round(launches_per_step * args.steps)),
		"roofline": roofline, "cpu_baseline": cpu, "large_batch_kernels": big, "configs": configs,
	}))
	finish(world)



# ---------------------------------------------------------------------------------------------------------------------
# The other BASELINE.json configurations (the headline above is configs[1]); one sub-object each under "configs".
TRAIN_CONFIGS = [
	dict(key="c1", name="LIF 784-128-10 non-recurrent, FastSigmoid, batch 256, MNIST-shaped periodic to_spikes",
		H=128, layer="LIF", rec=False, ink=0.19, B=256, multi_gpu=False),
	dict(key="c3", name="ALIF 784-64-10 non-recurrent, learn_beta, Fashion-MNIST-shaped (ink 0.5) periodic to_spikes, batch 256",
		H=64, layer="ALIF", rec=False, ink=0.50, B=256, multi_gpu=False),
	dict(key="c4", name="ALIF recurrent H=1024, learn_beta, batch 512 per GPU (4096 over 8 GPUs), data parallel",
		H=1024, layer="ALIF", rec=True, ink=0.19, B=512, multi_gpu=True),
]


def load_peaks():
	try:
		pk = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
		return float(pk["hbm_gbs"]), float(pk.get("bf16_tflops_sustained", pk.get("bf16_tflops", 1400.0))), "measured"
	except Exception:
		return 6650.0, 1400.0, "fallback"


def per_sample_work(Hh, rec, alif, train, traces=True, Tt=T):
	"""Algorithmic FLOPs and HBM bytes per sample (SURVEY.md 8d): fwd 2T(NH + [rec]H^2 + HO), bwd 2T(NH + 2[rec]H^2 + 2HO);
	bytes fwd = X + traces (s = 2 LIF, 3 ALIF) + y, the backward reads the same again."""
	r = 1 if rec else 0
	flops = 2 * Tt * (N * Hh + r * Hh * Hh + Hh * O)
	byts = Tt * N * 4 + ((3 if alif else 2) * Tt * Hh * 4 if traces else 0) + Tt * O * 4
	if train:
		flops += 2 * Tt * (N * Hh + 2 * r * Hh * Hh + 2 * Hh * O)
		byts *= 2
	return flops, byts


def step_roofline(value_per_gpu, Hh, rec, alif, train, traces=True, Tt=T):
	"""Whole-step roofline of one configuration on one GPU: which of HBM or the (3 x BF16 split) tensor pipe bounds
	the algorithmic work, and the fraction of that ceiling the measured throughput reaches."""
	hbm, tf, src = load_peaks()
	flops, byts = per_sample_work(Hh, rec, alif, train, traces, Tt)
	ceil_hbm = hbm * 1e9 / byts
	ceil_tc3 = tf * 1e12 / 3.0 / flops         # fp32-grade products on bf16 tensor cores cost three passes
	if ceil_tc3 < ceil_hbm:
		ach = value_per_gpu * flops * 3.0 / 1e12
		return {"scope": "whole step", "bound": "tensor", "achieved": ach, "peak": tf, "unit": "TFLOP/s", "frac": ach / tf,
			"traffic": None, "peak_source": src, "note": "3xBF16-split FLOPs (fp32-grade products) against the sustained bf16 peak",
			"ceiling_samples_per_s": ceil_tc3, "hbm_ceiling_samples_per_s": ceil_hbm}
	ach = value_per_gpu * byts / 1e9
	return {"scope": "whole step", "bound": "hbm", "achieved": ach, "peak": hbm, "unit": "GB/s", "frac": ach / hbm,
		"traffic": None, "peak_source": src, "ceiling_samples_per_s": ceil_hbm, "tensor3x_ceiling_samples_per_s": ceil_tc3}


def kernel_table(step_fn, iters=3):
	from snnimageclassification_b200 import _cabi
	for i in range(2):
		step_fn(i)
	torch.cuda.synchronize()
	with _cabi.kernel_profile() as prof:
		for i in range(iters):
			step_fn(i)
	return {name: round(ms / iters, 4) for name, (ms, n) in prof.result.items()}


def run_train_config(spec, dev, world, rank, steps, warmup, timed, dp):
	"""value / ms_per_step / roofline of one training configuration, measured exactly like the headline: rasters (with
	their run tables) resident in HBM, rotating batches, one CUDA graph per step, CUDA events, max over ranks."""
	from snnimageclassification_b200 import SNN, FusedAdam, LayerType, SpikeFuncType, ToSpikes
	alif = spec["layer"] == "ALIF"
	torch.manual_seed(0)
	enc = ToSpikes(T, use_periods=True)
	net = SNN(N, O, spec["H"], use_recurrent_connection=spec["rec"], int_time_steps=T, spike_func=SpikeFuncType.FastSigmoid,
		hidden_layer_type=LayerType.ALIF if alif else LayerType.LIF, device=dev, **({"learn_beta": True} if alif else {}))
	opt = FusedAdam(net.parameters(), lr=1e-3, weight_decay=1e-5)
	if dp and world > 1:
		opt.enable_data_parallel()
	crit = torch.nn.NLLLoss()
	net.train()
	B = spec["B"]
	pool = max(2, -(-(140 << 20) // (B * T * N * 4)))       # rotating batches > 126 MB of L2
	xs, ys, xbs = [], [], []
	g = torch.Generator().manual_seed(4242 + rank)
	for i in range(pool):
		img = (torch.randint(1, 256, (B, N), generator=g).float() / 255.0) * (torch.rand(B, N, generator=g) < spec["ink"])
		xs.append(enc.encode_batch(img.to(dev)))
		xbs.append(enc.encode_batch_bits(img.to(dev)))      # the same raster bit-packed (SNNK_F_INPUT_BITS kernels)
		ys.append(torch.randint(0, O, (B,), generator=g).to(dev))
	graphs = [net.graphed_train_step(xs[i], ys[i], crit, opt, static_inputs=True) for i in range(pool)]
	def step(i):
		return graphs[i % pool]()
	for i in range(warmup):
		step(i)
	ms = timed(step, steps)
	value = world * B * steps / (ms * 1e-3)
	def eager(i):
		loss = net.batch_loss(xs[i % pool], ys[i % pool], crit)
		opt.zero_grad()
		loss.backward()
	kern = kernel_table(eager) if world == 1 else None
	del graphs
	graphs_b = [net.graphed_train_step(xbs[i], ys[i], crit, opt, static_inputs=True) for i in range(pool)]
	def step_b(i):
		return graphs_b[i % pool]()
	for i in range(warmup):
		step_b(i)
	ms_b = timed(step_b, steps)
	out = {"workload": spec["name"], "value": value, "unit": "samples/s", "ms_per_step": ms / steps, "steps": steps,
		"global_batch": world * B, "n_gpus": world, "roofline": step_roofline(value / world, spec["H"], spec["rec"], alif, True),
		"kernel_ms_per_step_eager": kern,
		"packed_input": {"value": world * B * steps / (ms_b * 1e-3), "ms_per_step": ms_b / steps,
			"input": "the same rasters bit-packed, resident in HBM (bit-fed GEMMs, no run table)"}}
	del graphs_b, xs, xbs, ys, net, opt
	torch.cuda.empty_cache()
	return out


def run_inference_sweep(dev, quick=False):
	"""BASELINE configs[4]: inference only (no traces), batch 8192, H in {128, 512, 2048}, LIF / ALIF recurrent,
	T in {2, 10, 32, 100} on encoder output, plus the spike-sparsity sweep on Bernoulli(p) rasters (H = 128, T = 100)."""
	from snnimageclassification_b200 import SNN, LayerType, SpikeFuncType, ToSpikes
	from snnimageclassification_b200.modules.functional import mark_binary
	B = 8192
	g = torch.Generator().manual_seed(99)
	img = (torch.randint(1, 256, (B, N), generator=g).float() / 255.0) * (torch.rand(B, N, generator=g) < 0.19)
	img = img.to(dev)
	rows = []

	def measure(net, x, iters):
		net.eval()
		with torch.no_grad():
			for _ in range(2):
				net.get_prediction_logits(x, re_outputs_trace=False, re_hidden_states=False)
			e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
			torch.cuda.synchronize()
			e0.record()
			for _ in range(iters):
				net.get_prediction_logits(x, re_outputs_trace=False, re_hidden_states=False)
			e1.record()
			torch.cuda.synchronize()
		return e0.elapsed_time(e1) / iters

	cases = [(Hh, layer, Tt) for Hh in (128, 512, 2048) for layer in ("LIF", "ALIF") for Tt in (2, 10, 32, 100)]
	if quick:
		cases = [c for c in cases if c[2] in (10, 100) and c[1] == "ALIF"]
	for Hh, layer, Tt in cases:
		alif = layer == "ALIF"
		torch.manual_seed(0)
		net = SNN(N, O, Hh, use_recurrent_connection=True, int_time_steps=Tt, spike_func=SpikeFuncType.FastSigmoid,
			hidden_layer_type=LayerType.ALIF if alif else LayerType.LIF, device=dev, **({"learn_beta": True} if alif else {}))
		x = ToSpikes(Tt, use_periods=True).encode_batch(img, frame_runs=False)      # (B,T,N) fp32 resident, > L2 from T = 10 on
		ms = measure(net, x, 3 if Hh >= 512 and Tt >= 32 else 10)
		v = B / (ms * 1e-3)
		del x
		xb = ToSpikes(Tt, use_periods=True).encode_batch_bits(img)                  # the same raster as (B,T,25) int32 words
		ms_b = measure(net, xb, 3 if Hh >= 512 and Tt >= 32 else 10)
		rows.append({"H": Hh, "layer": layer, "T": Tt, "input": "periodic to_spikes, ink 0.19", "ms": round(ms, 4), "value": v,
			"roofline": step_roofline(v, Hh, True, alif, False, traces=False, Tt=Tt),
			"packed_input": {"ms": round(ms_b, 4), "value": B / (ms_b * 1e-3)}})
		del net, xb
		torch.cuda.empty_cache()
	for p in (0.004, 0.01, 0.1, 0.4):
		torch.manual_seed(0)
		net = SNN(N, O, 128, use_recurrent_connection=True, int_time_steps=T, spike_func=SpikeFuncType.FastSigmoid,
			hidden_layer_type=LayerType.ALIF, device=dev, learn_beta=True)
		x = mark_binary((torch.rand(B, T, N, device=dev) < p).float())
		ms = measure(net, x, 10)
		v = B / (ms * 1e-3)
		rows.append({"H": 128, "layer": "ALIF", "T": T, "input": f"Bernoulli({p})", "ms": round(ms, 4), "value": v,
			"roofline": step_roofline(v, 128, True, True, False, traces=False)})
		del net, x
		torch.cuda.empty_cache()
	best = max(rows, key=lambda r: r["value"])
	return {"workload": "inference only (no traces), recurrent LIF/ALIF, batch 8192, 1 GPU; eager launches, rasters resident in HBM",
		"unit": "samples/s", "value": next(r["value"] for r in rows if (r["H"], r["layer"], r["T"], r["input"][:3]) == (128, "ALIF", 100, "per")),
		"value_of": "ALIF H=128, T=100 from the fp32 raster (SURVEY 8d); packed_input = the same rasters bit-packed",
		"value_packed_input": next(r["packed_input"]["value"] for r in rows if (r["H"], r["layer"], r["T"], r["input"][:3]) == (128, "ALIF", 100, "per")),
		"sweep": rows, "best": {k: best[k] for k in ("H", "layer", "T", "input", "value")}}


# ---- ncu evidence parsed from the committed summaries (never hand-copied numbers) --------------------------------------
_UNIT = {"byte": 1.0, "Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9, "": 1.0, "ns": 1e-3, "nsecond": 1e-3, "us": 1.0, "usecond": 1.0,
	"ms": 1e3, "msecond": 1e3}      # durations end up in microseconds


def ncu_summary_rows(path):
	"""Rows of an `ncu --page raw --csv` export (first row metric names, second row units) as dicts; values converted
	to base units with the unit row (a Kbyte column read as bytes was a 1000x error in round 1)."""
	import csv
	try:
		with open(path, newline="") as fh:
			rows = list(csv.reader(fh))
	except OSError:
		return []
	if len(rows) < 3:
		return []
	names, units = rows[0], rows[1]
	out = []
	for r in rows[2:]:
		d = {}
		for n, u, v in zip(names, units, r):
			if n in ("Kernel Name", "Function Name"):
				d["kernel"] = v
				continue
			try:
				d[n] = float(v.replace(",", "")) * _UNIT.get(u, 1.0)
			except ValueError:
				d[n] = v
		out.append(d)
	return out


NCU_SUMMARIES = ["profiles/r02_ncu_full_summary.csv", "profiles/r01_ncu_full_summary_final.csv"]
# the kernels the HEADLINE configuration launches (B = 256: the one-row-per-CTA SIMT recurrences)
KERNEL_REGEX = {"K1": ("k_proj_tc",), "K2": ("k_recur_fwd_lean", "k_recur_fwd<"), "K3": ("k_recur_bwd_lean", "k_recur_bwd<"),
	"K4": ("k_wgrad_tc",), "K5": ("k_encode",), "K6": ("k_head_nll",)}      # first pattern with a capture wins


def ncu_evidence(kernel_key):
	"""(dram traffic bytes per launch, shared-memory wavefronts per launch, source file) of the LONGEST launch of the
	kernel family in the newest committed ncu summary that has it."""
	pats = KERNEL_REGEX.get(kernel_key)
	if not pats:
		return None
	for pat, rel in ((p_, r_) for p_ in pats for r_ in NCU_SUMMARIES):
		rows = [r for r in ncu_summary_rows(os.path.join(ROOT, rel)) if pat in str(r.get("kernel", ""))]
		if rows:
			r = max(rows, key=lambda q: q.get("gpu__time_duration.sum", 0.0))
			return {"traffic": r.get("dram__bytes_read.sum", 0.0) + r.get("dram__bytes_write.sum", 0.0),
				"smem_wavefronts": r.get("l1tex__data_pipe_lsu_wavefronts_mem_shared.sum"), "kernel": r["kernel"],
				"ncu_duration_us": r.get("gpu__time_duration.sum", 0.0),
				"source": rel}
	return None



def large_batch_rooflines(net, enc, dev, B=4096, iters=5):
	"""Per-kernel achieved bandwidth of the same kernels at batch 4096 (BASELINE configs[4] regime), where the
	recurrence is no longer bound by the latency of its 2T sequential steps.  Extra information, not the headline."""
	from snnimageclassification_b200 import _cabi
	img, lab = synthetic_images(B, seed=77)
	x = enc.encode_batch(img.to(dev), frame_runs=False)    # dense kernels: every row of X is projected and contracted
	lab = lab.to(dev)
	crit = torch.nn.NLLLoss()

	def step():
		loss = net.batch_loss(x, lab, crit)
		net.zero_grad()
		loss.backward()
	for _ in range(2):
		step()
	torch.cuda.synchronize()
	with _cabi.kernel_profile() as prof:
		for _ in range(iters):
			step()
	BT = B * T
	algo = {"K1": BT * N * 4 + BT * H * 4, "K2": BT * H * 4 + 3 * BT * H * 4 + BT * O * 4 + BT * H // 8,
		"K3": 2 * BT * H * 4 + BT * H // 8 + 2 * BT * H * 4, "K4": BT * N * 4 + 2 * BT * H * 4 + BT * H * 4}
	peak = 6560.0
	try:
		peak = float(json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))["hbm_gbs"])
	except Exception:
		pass
	out = {"batch": B}
	for name, (ms, n) in prof.result.items():
		key = name.split()[0]
		if key in algo:
			gbs = algo[key] / (ms / iters * 1e-3) / 1e9
			out[name] = {"ms": round(ms / iters, 4), "GBps": round(gbs, 1), "frac_of_hbm_peak": round(gbs / peak, 3)}
	del x
	# the bit-fed GEMMs on the same batch (tensor-pipe bound: achieved 2-plane FLOP/s against the sustained bf16 peak;
	# kind::f16 runs at the bf16 rate, kind::tf32 at half of it)
	xb = enc.encode_batch_bits(img.to(dev))
	def step_b():
		loss = net.batch_loss(xb, lab, crit)
		net.zero_grad()
		loss.backward()
	for _ in range(2):
		step_b()
	torch.cuda.synchronize()
	with _cabi.kernel_profile() as prof:
		for _ in range(iters):
			step_b()
	_, tf, _src = load_peaks()
	flops = {"K1": 2.0 * BT * 832 * 2 * H, "K4": 2.0 * BT * 1024 * 2 * H}      # k / feature extents padded to the tiles
	rate = {"K1": 1.0, "K4": 0.5}
	bits = {}
	for name, (ms, n) in prof.result.items():
		key = name.split()[0]
		if key in flops:
			ach = flops[key] / (ms / iters * 1e-3) / 1e12
			bits[name] = {"ms": round(ms / iters, 4), "TFLOPs": round(ach, 1), "frac_of_tensor_peak": round(ach / (tf * rate[key]), 3),
				"kind": "f16, two fp16 planes" if key == "K1" else "tf32, two tf32 planes"}
	out["bit_packed_input"] = bits
	del xb
	return out


def dump_outputs(out_dir, loss, net):
	"""The last timed step's batch loss and the parameters its Adam update left, one float32 .npy file each."""
	os.makedirs(out_dir, exist_ok=True)
	arrays = {"loss": loss.detach().reshape(1)}
	arrays.update({f"param.{name}": p.detach() for name, p in net.named_parameters()})
	for name, t in arrays.items():
		np.save(os.path.join(out_dir, f"{name}.npy"), t.float().cpu().numpy())


def finish(world):
	"""Leave without tearing NCCL down: destroy_process_group() can block behind the captured graphs' communicator
	references, and there is nothing left to flush but stdout."""
	sys.stdout.flush()
	sys.stderr.flush()
	if world > 1:
		os._exit(0)


def profile_kernels(step_fn, iters=10):
	"""Average CUDA-event duration and launch count of every kernel of the library over ``iters`` train steps
	(snnk_profile_begin/end: events recorded on the launching stream around each launch)."""
	from snnimageclassification_b200 import _cabi
	for i in range(2):
		step_fn(i)
	torch.cuda.synchronize()
	with _cabi.kernel_profile() as prof:
		for i in range(iters):
			step_fn(i)
	# algorithmic bytes per launch (DESIGN.md "Kernels"): what the kernel must read and write at least once
	BT = B_PER_GPU * T
	algo = {
		"K1": BT * N * 4 + BT * H * 4,                                   # read X, write I_in
		"K2": BT * H * 4 + 3 * BT * H * 4 + BT * O * 4 + BT * H // 8,      # read I_in; write V,a,Z,y,zbits
		"K3": 2 * BT * H * 4 + BT * H // 8 + BT * H * 4,                   # read V,a,zbits; write gI
		"K4": BT * N * 4 + BT * H * 4 + BT * H // 8,                       # read X, gI, zbits
		"K5": B_PER_GPU * N * 4 + BT * N * 4,                              # read images, write rasters
		"K6": B_PER_GPU * O * 4 * 3,
	}
	res = {}
	for name, (ms, n) in prof.result.items():
		res[name] = {"ms": ms / n, "launches_per_step": n / iters, "ms_per_step": ms / iters,
			"bytes": algo.get(name.split()[0], 0)}
	return res


if __name__ == "__main__":
	main()
