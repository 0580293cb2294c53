"""Surrogate spike functions -- mirror of the reference's src/modules/spike_funcs.py.

Same names and calling convention (``Func.apply(V, threshold, gamma)``); the arithmetic runs in libsnnk.so
(``snnk_spike_forward`` / ``snnk_spike_backward``).  Inside ``SNN.forward`` these classes are only *tags*: the
fused kernels apply the Heaviside step and its surrogate derivative in-register, and the class selects which
derivative (``SURROGATE_ID``).  A user-defined subclass (``SURROGATE_ID = None``, own ``backward``, the base
``forward``) trains too: its ``backward`` is evaluated once over the saved membrane trace and the BPTT kernels stream
the result (see ``SpikeFunction`` and ``fused_surrogate``).
"""
from __future__ import annotations

import enum
from typing import Any

import torch

from .. import _cabi


class SpikeFuncType(enum.Enum):
	# reference spike_funcs.py:7-9
	FastSigmoid = enum.auto()
	Phi = enum.auto()


def _as_f32_cuda(t: torch.Tensor, like: torch.Tensor) -> torch.Tensor:
	t = torch.as_tensor(t, dtype=torch.float32, device=like.device)
	return t.contiguous()


class SpikeFunction(torch.autograd.Function):
	"""Heaviside forward ``out = (inputs >= threshold)`` (reference spike_funcs.py:12-29).

	A user-defined surrogate is a subclass that keeps this ``forward`` and overrides ``backward(ctx, grad)``:
	it reads ``inputs, threshold, gamma = ctx.saved_tensors`` (what this ``forward`` saves) and returns
	``(grad * f(inputs, threshold, gamma), None, None)``, with ``f`` elementwise.  Inside ``SNN`` that ``backward``
	is called once per backward pass with ``grad`` = ones over the whole saved (B, T, H) membrane trace and the
	per-step threshold (theta for LIF, theta + beta a_t for ALIF, v_peak for Izhikevich); it must not synchronise
	with the host if the training step is to be captured in a CUDA graph.  The base class itself has no surrogate:
	inference runs, training raises ``NotImplementedError`` as in the reference.
	"""
	SURROGATE_ID = None

	@staticmethod
	def forward(ctx: Any, inputs: torch.Tensor, threshold: torch.Tensor = torch.tensor(1.0),
			gamma: torch.Tensor = torch.tensor(0.3)):
		_cabi.require_b200(inputs.device)
		v = inputs.detach().float().contiguous()
		thr = _as_f32_cuda(threshold, v)
		if thr.numel() != 1 and thr.shape != v.shape:
			thr = thr.expand_as(v).contiguous()
		gam = _as_f32_cuda(gamma, v).reshape(-1)[:1].contiguous()
		ctx.save_for_backward(v, thr, gam)
		out = torch.empty_like(v)
		with torch.cuda.device(v.device):
			rc = _cabi.lib().snnk_spike_forward(
				_cabi.ptr(v), _cabi.ptr(thr), v.numel(), thr.numel(), _cabi.ptr(out), _cabi.stream_ptr())
		_cabi.check(rc, "snnk_spike_forward")
		return out

	@staticmethod
	def backward(ctx: Any, grad_outputs):
		raise NotImplementedError  # reference spike_funcs.py:31-39: the base class has no surrogate

	@classmethod
	def _surrogate_backward(cls, ctx: Any, grad_outputs: torch.Tensor):
		v, thr, gam = ctx.saved_tensors
		g = grad_outputs.detach().float().contiguous()
		out = torch.empty_like(v)
		with torch.cuda.device(v.device):
			rc = _cabi.lib().snnk_spike_backward(
				cls.SURROGATE_ID, _cabi.ptr(v), _cabi.ptr(thr), _cabi.ptr(gam), _cabi.ptr(g), v.numel(),
				thr.numel(), _cabi.ptr(out), _cabi.stream_ptr())
		_cabi.check(rc, "snnk_spike_backward")
		return out, None, None  # threshold and gamma get no gradient (spike_funcs.py:62/79)


class HeavisideSigmoidApprox(SpikeFunction):
	"""Backward: ``g / (gamma |V - thr| + 1)^2`` (reference spike_funcs.py:46-62, Zenke & Ganguli 2018)."""
	SURROGATE_ID = _cabi.SNNK_FAST_SIGMOID

	@staticmethod
	def backward(ctx: Any, grad_outputs):
		return HeavisideSigmoidApprox._surrogate_backward(ctx, grad_outputs)


class HeavisidePhiApprox(SpikeFunction):
	"""Backward: ``g (gamma/(thr+eps)) max(0, 1 - |(V - thr)/(thr+eps)|)`` (reference spike_funcs.py:65-79)."""
	epsilon = 1e-5
	SURROGATE_ID = _cabi.SNNK_PHI

	@staticmethod
	def backward(ctx: Any, grad_outputs):
		return HeavisidePhiApprox._surrogate_backward(ctx, grad_outputs)


def fused_surrogate(func) -> int:
	"""The surrogate kind the fused kernels run for the spike function class ``func`` (SnnkDesc.surrogate): the
	built-ins' ``SURROGATE_ID``, otherwise ``SNNK_SURROGATE_TRACE`` -- the derivative is ``func.backward``'s, handed
	to the BPTT sweep as a trace.  The fused forward is the Heaviside step ``V >= threshold``, so a class with its
	own ``forward`` is refused."""
	if not (isinstance(func, type) and issubclass(func, SpikeFunction)):
		raise TypeError(f"spike function {func!r} is not a SpikeFunction subclass")
	if func.forward is not SpikeFunction.forward:
		raise NotImplementedError(
			f"spike function {func.__name__} overrides forward: the fused B200 kernels fire on the Heaviside step "
			"V >= threshold of SpikeFunction.forward; only backward (the surrogate) may be user-defined")
	return _cabi.SNNK_SURROGATE_TRACE if func.SURROGATE_ID is None else func.SURROGATE_ID


SpikeFuncType2Func = {
	SpikeFuncType.FastSigmoid: HeavisideSigmoidApprox,
	SpikeFuncType.Phi: HeavisidePhiApprox,
}
