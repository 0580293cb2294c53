"""Shared helpers for the test-suite: fixture loading, parity metrics, kernel selection and guard bands."""
import os
import re

import numpy as np

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def load(name):
	return np.load(os.path.join(GOLDEN, name), allow_pickle=False)


def unpack_bits(bits, shape):
	n = int(np.prod(shape))
	return np.unpackbits(bits)[:n].reshape(shape)


def dynamics_case(z, name):
	"""Returns the dict stored for one dynamics case."""
	pre = name + "/"
	return {k[len(pre):]: z[k] for k in z.files if k.startswith(pre)}


def rel_err(a, b):
	"""max |a-b| / max(|b|, tiny): the relative measure used for gradients and losses."""
	a = np.asarray(a, dtype=np.float64)
	b = np.asarray(b, dtype=np.float64)
	den = max(np.abs(b).max(), 1e-30)
	return float(np.abs(a - b).max() / den)


def first_divergence(Za, Zb):
	"""Per sample, the first time step at which two rasters (B,T,H) differ (T if never)."""
	diff = (np.asarray(Za) != np.asarray(Zb)).any(axis=2)
	T = diff.shape[1]
	return np.where(diff.any(axis=1), diff.argmax(axis=1), T)


def elementwise_err(a, b, floor_frac=1e-3):
	"""max over elements of |a-b| / max(|b|, floor), floor = floor_frac * max|b|: an ELEMENTWISE relative error with an
	absolute floor, so that small-magnitude entries are checked too (``rel_err`` above is a max-norm bar: it only sees
	the entries near the largest magnitude)."""
	a = np.asarray(a, dtype=np.float64)
	b = np.asarray(b, dtype=np.float64)
	floor = max(np.abs(b).max() * floor_frac, 1e-30)
	return float((np.abs(a - b) / np.maximum(np.abs(b), floor)).max())


def unexplained_forks(Z_test, Z_ref, V_ref, thr_ref, tol=2e-5):
	"""Rasters of a chaotic recurrent net can only be compared up to the first spike that sits ON the threshold: a
	membrane potential within rounding distance of its threshold flips under ANY change of summation order (also
	between the reference on CPU and on GPU), after which that sample follows another trajectory.

	For every sample whose raster differs from the reference's, look at the FIRST differing step: every neuron that
	differs there must be such a near-tie in the reference's own trace, |V - thr| <= tol * max(|thr|, |V|).  Returns
	(number of forked samples, number of forked samples whose first difference is NOT a near-tie).  The second number
	must be 0; the first is reported and bounded separately."""
	Z_test, Z_ref = np.asarray(Z_test), np.asarray(Z_ref)
	B, T, H = Z_ref.shape
	thr_ref = np.broadcast_to(np.asarray(thr_ref, dtype=np.float32), Z_ref.shape)
	first = first_divergence(Z_test, Z_ref)
	forked = unexplained = 0
	for b in np.nonzero(first < T)[0]:
		t = first[b]
		forked += 1
		diff = Z_test[b, t] != Z_ref[b, t]
		v, th = V_ref[b, t][diff].astype(np.float64), thr_ref[b, t][diff].astype(np.float64)
		if np.any(np.abs(v - th) > tol * np.maximum(np.abs(th), np.abs(v))):
			unexplained += 1
	return forked, unexplained


# ---- which kernels ran -----------------------------------------------------------------------------------------------
def launched(fn):
	"""Runs ``fn()`` under torch.profiler with CUDA activity and returns (its result, the names of the device kernels it
	launched).  A profile without any kernel of the library fails: a selection test must not pass on an empty list."""
	import torch
	from torch.autograd import DeviceType
	torch.cuda.synchronize()
	with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
		# Late in a long session the profiler can lose the first few device records of a window (a list without the
		# first kernels of fn, or an empty one); a few throw-away kernels take that place.
		pad = torch.zeros(1, device="cuda")
		for _ in range(16):
			pad.add_(1.0)
		torch.cuda.synchronize()
		res = fn()
		torch.cuda.synchronize()
	names = [e.name for e in prof.events() if e.device_type == DeviceType.CUDA]
	assert any("snnk::" in n for n in names), f"the profiler reports no kernel of the library: {names[:8]}"
	return res, names


def ran(names, pattern):
	return any(re.search(pattern, n) for n in names)


# ---- guard bands -------------------------------------------------------------------------------------------------------
GUARD = 4096          # bytes on each side
SENT = 0xA5


class Guarded:
	"""A tensor of `shape` on cuda:0 carved out of a byte buffer with GUARD sentinel bytes in front of and behind it."""

	def __init__(self, shape, dtype=None, fill_inside=True):
		import torch
		dtype = torch.float32 if dtype is None else dtype
		n = int(np.prod(shape)) * torch.empty((), dtype=dtype).element_size()
		pad = (-n) % 256
		self.raw = torch.full((GUARD + n + pad + GUARD,), SENT, dtype=torch.uint8, device="cuda:0")
		self.n, self.pad = n, pad
		self.t = self.raw[GUARD:GUARD + n].view(dtype).view(shape)

	def check(self, name, written=True):
		import torch
		front, back = self.raw[:GUARD], self.raw[GUARD + self.n:]
		assert bool((front == SENT).all()), f"{name}: write in front of the buffer"
		assert bool((back == SENT).all()), f"{name}: write behind the buffer"
		if written and self.t.dtype == torch.float32:
			# 0xA5A5A5A5 as a float is -2.87e-16: exact sentinel words inside mean unwritten elements
			words = self.raw[GUARD:GUARD + self.n].view(torch.int32)
			assert int((words == int(np.array([0xA5A5A5A5], dtype=np.uint32).view(np.int32)[0])).sum()) == 0, f"{name}: unwritten elements"
			assert bool(torch.isfinite(self.t).all()), f"{name}: non-finite values"
