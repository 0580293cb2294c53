"""Image -> spike-train encoder -- mirror of the reference's src/datasets/datasets.py (``ToSpikes``).

Same constructor and methods as the reference; the arithmetic runs in the ``snnk_encode`` CUDA kernel
(csrc/encode_head.cuh).  Two ways to use it:

* drop-in, per sample, like the reference transform: ``ToSpikes(n_steps)(x)`` with ``x`` a numpy array or a
  tensor of shape (n_pix,) returns a float64 tensor ``(n_steps, n_pix)`` on the device ``x`` lives on (CPU inputs
  are staged through the GPU and copied back, which keeps reference pipelines working unchanged);
* B200-native, per batch: ``encode_batch(images (B, n_pix))`` -> ``(B, n_steps, n_pix)`` float32 on the GPU, so
  the raster never exists on the host (``SNN(..., input_encoder=ToSpikes(...))`` uses this).

Bit-exactness: integer latencies are identical to the reference's for every k/255 pixel level and the
reference's golden vectors (tests/); see DESIGN.md for the one-ulp ``log`` caveat on arbitrary float32 inputs.
"""
from __future__ import annotations

import enum
from typing import Optional, Union

import os

import numpy as np
import torch

from .. import _cabi

_DT = {torch.float32: _cabi.SNNK_F32, torch.float64: _cabi.SNNK_F64, torch.uint8: _cabi.SNNK_U8,
	torch.int64: _cabi.SNNK_I64}


class DatasetId(enum.Enum):
	# reference datasets.py:11-13
	MNIST = enum.auto()
	FASHION_MNIST = enum.auto()


class ToSpikes:
	def __init__(self, n_steps: int, t_max: float = None, tau=20.0 * 1e-3, thr=0.2, use_periods=False,
			epsilon=1e-7, device: Optional[Union[str, torch.device]] = None):
		"""Same parameters as the reference (datasets.py:17-40) plus the CUDA ``device`` used for CPU inputs."""
		self.n_steps = n_steps
		self.t_max = n_steps if t_max is None else t_max
		self.tau = tau
		self.thr = thr
		self.epsilon = epsilon
		self.spikes_indices = None  # kept for attribute compatibility; the kernel needs no index cache
		self.use_periods = use_periods
		self.spikes_gen_func = self.firing_periods_to_spikes if use_periods else self.firing_times_to_spikes
		self.device = torch.device(device) if device is not None else None

	# ---- plumbing ---------------------------------------------------------------------------------------------------
	def _device(self) -> torch.device:
		if self.device is not None:
			return self.device
		if not torch.cuda.is_available():
			raise RuntimeError("ToSpikes runs on a CUDA sm_100 device only; there is no CPU fallback")
		return torch.device("cuda", torch.cuda.current_device())

	def _stage(self, x, dtype=None):
		"""-> (2-D contiguous CUDA tensor, original leading shape, came_from_cpu, was_numpy)."""
		was_numpy = isinstance(x, np.ndarray)
		t = torch.from_numpy(np.ascontiguousarray(x)) if was_numpy else x
		if dtype is not None:
			t = t.to(dtype)
		elif t.dtype not in (torch.float32, torch.float64):
			t = t.to(torch.float64 if was_numpy else torch.float32)
		on_cpu = not t.is_cuda
		if on_cpu:
			t = t.to(self._device())
		shape = tuple(t.shape)
		t2 = t.reshape(1, t.numel()) if t.ndim <= 1 else t.reshape(shape[0], int(np.prod(shape[1:])))
		return t2.contiguous(), shape, on_cpu, was_numpy

	def _run(self, x2: torch.Tensor, periodic: bool, out_dtype: torch.dtype, want_periods: bool, want_raster: bool = True):
		_cabi.require_b200(x2.device)
		n_items, n_pix = x2.shape
		out = torch.empty((n_items, self.n_steps if want_raster else 1, n_pix), dtype=out_dtype, device=x2.device)
		per = torch.empty((n_items, n_pix), dtype=torch.int64, device=x2.device) if want_periods else None
		with torch.cuda.device(x2.device):
			rc = _cabi.lib().snnk_encode(
				_cabi.ptr(x2), _DT[x2.dtype], n_items, n_pix, self.n_steps if want_raster else 1, float(self.t_max),
				float(self.tau), float(self.thr), float(self.epsilon), int(periodic), _cabi.ptr(out), _DT[out_dtype],
				_cabi.ptr(per), _cabi.stream_ptr())
		_cabi.check(rc, "snnk_encode")
		return out, per

	@staticmethod
	def _back(t: torch.Tensor, on_cpu: bool, was_numpy: bool):
		if on_cpu or was_numpy:
			t = t.cpu()
		return t.numpy() if was_numpy else t

	# ---- the reference's methods --------------------------------------------------------------------------------------
	def pixels_to_firing_periods(self, x):
		"""First-spike latency / period of every pixel: int(tau * ln(x / (x - thr))), t_max below thr (datasets.py:42-54)."""
		x2, shape, on_cpu, was_numpy = self._stage(x)
		_, per = self._run(x2, False, torch.uint8, want_periods=True, want_raster=False)
		return self._back(per.reshape(shape), on_cpu, was_numpy)

	def firing_periods_to_spikes(self, firing_periods):
		"""Periodic raster: p = clamp(period, 1, n_steps-1), spikes at p, 2p, ... (datasets.py:72-79)."""
		p2, shape, on_cpu, was_numpy = self._stage(firing_periods, dtype=torch.int64)
		out, _ = self._run(p2, True, torch.float64, want_periods=False)
		out = out.reshape((self.n_steps,) + shape) if len(shape) <= 1 else out.transpose(0, 1).reshape((self.n_steps,) + shape)
		return self._back(out, on_cpu, was_numpy)

	def firing_times_to_spikes(self, firing_times):
		"""Latency raster: one spike at t = firing time if it is < n_steps (datasets.py:81-86)."""
		p2, shape, on_cpu, was_numpy = self._stage(firing_times, dtype=torch.int64)
		out, _ = self._run(p2, False, torch.float64, want_periods=False)
		out = out.reshape((self.n_steps,) + shape) if len(shape) <= 1 else out.transpose(0, 1).reshape((self.n_steps,) + shape)
		return self._back(out, on_cpu, was_numpy)

	def __call__(self, x) -> torch.Tensor:
		"""x (n_pix,) [or (d0, ...)] -> float64 tensor (n_steps, *x.shape), as the reference (datasets.py:93-97)."""
		x2, shape, on_cpu, _ = self._stage(x)
		if len(shape) <= 1:
			out, _ = self._run(x2, self.use_periods, torch.float64, want_periods=False)
			out = out.reshape((self.n_steps,) + shape)
		else:
			out, _ = self._run(x2.reshape(1, -1), self.use_periods, torch.float64, want_periods=False)
			out = out.reshape((self.n_steps,) + shape)
		return out.cpu() if on_cpu else out

	# ---- the batched GPU entry point ----------------------------------------------------------------------------------
	def encode_batch_bits(self, images: torch.Tensor) -> torch.Tensor:
		"""images (B, n_pix) -> the spike trains bit-packed: (B, n_steps, ceil(n_pix/32)) int32 on the GPU, bit l of
		word w = pixel 32 w + l (``SNNK_BITS``).  1/32 of the fp32 raster: the format to store rasters in or to move them
		between host and device; ``SNN`` accepts it directly (``unpack_raster`` is applied on the device)."""
		if images.ndim != 2:
			images = images.reshape(images.shape[0], int(np.prod(images.shape[1:])))
		x2, _, _, _ = self._stage(images)
		_cabi.require_b200(x2.device)
		n_items, n_pix = x2.shape
		out = torch.empty((n_items, self.n_steps, (n_pix + 31) // 32), dtype=torch.int32, device=x2.device)
		with torch.cuda.device(x2.device):
			rc = _cabi.lib().snnk_encode(
				_cabi.ptr(x2), _DT[x2.dtype], n_items, n_pix, self.n_steps, float(self.t_max), float(self.tau),
				float(self.thr), float(self.epsilon), int(self.use_periods), _cabi.ptr(out), _cabi.SNNK_BITS, None,
				_cabi.stream_ptr())
		_cabi.check(rc, "snnk_encode")
		return out

	def encode_batch(self, images: torch.Tensor, out_dtype: torch.dtype = torch.float32, frame_runs: bool = True,
			lazy: bool = False) -> torch.Tensor:
		"""images (B, n_pix) float32|float64 (any device) -> spike trains (B, n_steps, n_pix) on the GPU.

		The result is tagged as exactly {0,1} (the tensor-core kernels then skip their input check) and, with
		``frame_runs``, carries the batch's frame-run table (``snnk_encode_runs``): the production encoder repeats
		the same frame over long stretches of time steps, which ``SNN`` exploits (SURVEY.md 8f.1).  ``lazy`` (used by
		``SNN`` for its own intermediate raster, never for a tensor handed to the user): rows that the kernels consuming
		the table will not read are left unwritten."""
		if images.ndim != 2:
			images = images.reshape(images.shape[0], int(np.prod(images.shape[1:])))
		x2, _, _, _ = self._stage(images)
		n_items, n_pix = x2.shape
		nbytes = _cabi.lib().snnk_run_table_bytes(n_items, self.n_steps) if (frame_runs and n_items > 0 and n_pix > 0) else 0
		if nbytes == 0:
			out, _ = self._run(x2, self.use_periods, out_dtype, want_periods=False)
			out._snnk_binary = True
			return out
		_cabi.require_b200(x2.device)
		out = torch.empty((n_items, self.n_steps, n_pix), dtype=out_dtype, device=x2.device)
		changed = torch.empty((n_items, self.n_steps), dtype=torch.uint8, device=x2.device)
		# fp32 rasters: the first row of every run also goes behind the table, tiled for the compact projection, so that
		# the training step does not gather those rows at its head (include/snnk.h, SNNK_F_RUNS_TILED)
		tiled = 0
		if out_dtype == torch.float32 and os.environ.get("SNNK_RUNS_TILED", "1") != "0":
			tiled = _cabi.lib().snnk_run_table_tiled_bytes(n_items, self.n_steps, n_pix)
			if tiled > (256 << 20):      # sized for the table's capacity (a quarter of the rows): not worth it for huge batches
				tiled = 0
		table = torch.empty(((tiled or nbytes) // 4,), dtype=torch.int32, device=x2.device)
		with torch.cuda.device(x2.device):
			rc = _cabi.lib().snnk_encode_runs(
				_cabi.ptr(x2), _DT[x2.dtype], n_items, n_pix, self.n_steps, float(self.t_max), float(self.tau),
				float(self.thr), float(self.epsilon), int(self.use_periods), _cabi.ptr(out), _DT[out_dtype], None,
				_cabi.ptr(changed), _cabi.ptr(table), int(bool(lazy)) | (2 if tiled else 0), _cabi.stream_ptr())
		_cabi.check(rc, "snnk_encode_runs")
		out._snnk_binary = True
		out._snnk_runs = table
		return out


class SyntheticSpikeImages(torch.utils.data.Dataset):
	"""MNIST-shaped synthetic images (k/255 levels, given ink probability) with uniform labels.

	The reference downloads MNIST / Fashion-MNIST through torchvision (datasets.py:128-139); there is no network
	in the build or benchmark environment, so tests and bench.py use this generator (SURVEY.md 8d).
	"""

	def __init__(self, n_items: int, n_pix: int = 784, n_classes: int = 10, ink: float = 0.19, seed: int = 0):
		g = torch.Generator().manual_seed(seed)
		levels = torch.randint(1, 256, (n_items, n_pix), generator=g).float() / 255.0
		mask = torch.rand((n_items, n_pix), generator=g) < ink
		self.images = levels * mask
		self.labels = torch.randint(0, n_classes, (n_items,), generator=g)

	def __len__(self):
		return self.images.shape[0]

	def __getitem__(self, i):
		return self.images[i], self.labels[i]


def unpack_raster(bits: torch.Tensor, n_pix: int) -> torch.Tensor:
	"""(..., ceil(n_pix/32)) int32 bit-packed raster on the GPU -> (..., n_pix) float32 {0,1}, tagged as exactly binary."""
	if bits.dtype != torch.int32 or bits.shape[-1] != (n_pix + 31) // 32:
		raise ValueError("expected an int32 tensor whose last dimension is ceil(n_pix / 32)")
	_cabi.require_b200(bits.device)
	b = bits.contiguous()
	out = torch.empty(b.shape[:-1] + (n_pix,), dtype=torch.float32, device=b.device)
	n_rows = int(np.prod(b.shape[:-1])) if b.ndim > 1 else 1
	with torch.cuda.device(b.device):
		rc = _cabi.lib().snnk_unpack_raster(_cabi.ptr(b), n_rows, n_pix, _cabi.ptr(out), _cabi.stream_ptr())
	_cabi.check(rc, "snnk_unpack_raster")
	out._snnk_binary = True
	return out
