"""Spiking layers -- mirror of the reference's src/modules/spiking_layers.py.

The classes keep the reference's constructor signature, parameter names/shapes, initialisation order (so a seed
gives the same weights) and per-layer ``forward(inputs (B,F), state) -> (out, state)`` contract.  They hold the
parameters; ``SNN.forward`` does not call them once per time step -- it hands the whole sequence to the fused
CUDA kernels (see modules/functional.py).  The single-step ``forward`` below goes through the same kernels with
T = 1.
"""
from __future__ import annotations

import enum
from typing import Optional, Tuple, Type

import numpy as np
import torch
from torch import nn

from .. import _cabi
from . import functional as F_
from .spike_funcs import HeavisideSigmoidApprox, SpikeFunction, fused_surrogate


class LayerType(enum.Enum):
	# reference spiking_layers.py:11-14
	LIF = enum.auto()
	ALIF = enum.auto()
	Izhikevich = enum.auto()


class RNNLayer(torch.nn.Module):
	"""Parameter container (reference spiking_layers.py:17-93)."""

	def __init__(self, input_size: int, output_size: int, use_recurrent_connection=True, use_rec_eye_mask=True,
			dt=1e-3, device=None, **kwargs):
		super().__init__()
		self.input_size = input_size
		self.output_size = output_size
		self.use_recurrent_connection = use_recurrent_connection
		self.device = device
		if self.device is None:
			self._set_default_device_()
		self.dt = dt
		self.kwargs = kwargs
		self._set_default_kwargs()

		f32 = dict(device=self.device, dtype=torch.float32)
		self.forward_weights = nn.Parameter(torch.empty((input_size, output_size), **f32), requires_grad=True)
		self.use_rec_eye_mask = use_rec_eye_mask
		if use_recurrent_connection:
			self.recurrent_weights = nn.Parameter(torch.empty((output_size, output_size), **f32), requires_grad=True)
			# a plain attribute, not a buffer: it must stay out of state_dict (reference :50-57)
			self.rec_mask = (1 - torch.eye(output_size, **f32)) if use_rec_eye_mask else torch.ones(
				(output_size, output_size), **f32)
		else:
			self.recurrent_weights = None
			self.rec_mask = None

	def _set_default_kwargs(self):
		raise NotImplementedError()

	def _set_default_device_(self):
		self.device = torch.device("cuda") if torch.cuda.is_available() else torch.device("cpu")

	def create_empty_state(self, batch_size: int = 1) -> Tuple[torch.Tensor, ...]:
		raise NotImplementedError

	def _zeros_state(self, batch_size: int, n: int) -> Tuple[torch.Tensor, ...]:
		return tuple(
			torch.zeros((batch_size, self.output_size), device=self.device, dtype=torch.float32, requires_grad=True)
			for _ in range(n))

	def _init_forward_state(self, state=None, batch_size: int = 1) -> Tuple[torch.Tensor, ...]:
		# reference :69-83: None, or a tuple with None entries, means zeros
		if state is None:
			return self.create_empty_state(batch_size)
		if any(e is None for e in state):
			empty = self.create_empty_state(batch_size)
			return tuple(empty[i] if e is None else e for i, e in enumerate(state))
		return state

	def forward(self, inputs: torch.Tensor, state=None):
		raise NotImplementedError

	def initialize_weights_(self):
		for param in self.parameters():
			if param.ndim > 2:
				torch.nn.init.xavier_normal_(param)
			else:
				torch.nn.init.normal_(param)

	def _apply(self, fn, *args, **kwargs):
		# keep the non-buffer tensors (rec_mask and the scalar constants) on the module's device after .to()/.cuda()
		super()._apply(fn, *args, **kwargs)
		for name in ("rec_mask", "alpha", "threshold", "gamma", "rho", "kappa"):
			t = getattr(self, name, None)
			if isinstance(t, torch.Tensor) and not isinstance(t, nn.Parameter):
				setattr(self, name, fn(t))
		beta = getattr(self, "beta", None)
		if isinstance(beta, torch.Tensor) and not isinstance(beta, nn.Parameter):
			self.beta = fn(beta)
		if self.forward_weights is not None:
			self.device = self.forward_weights.device
		return self


class LIFLayer(RNNLayer):
	"""Leaky integrate-and-fire layer (reference spiking_layers.py:96-171).

	V_t = (alpha V_{t-1} + x_t W_in + Z_{t-1} (W_rec . M)) (1 - Z_{t-1}.detach());  Z_t = H(V_t - theta).
	"""
	SNNK_LAYER_TYPE = _cabi.SNNK_LIF

	def __init__(self, input_size: int, output_size: int, use_recurrent_connection=True, use_rec_eye_mask=True,
			spike_func: Type[SpikeFunction] = HeavisideSigmoidApprox, dt=1e-3, device=None, **kwargs):
		self.spike_func = spike_func
		super().__init__(
			input_size=input_size, output_size=output_size, use_recurrent_connection=use_recurrent_connection,
			use_rec_eye_mask=use_rec_eye_mask, dt=dt, device=device, **kwargs)
		f32 = dict(dtype=torch.float32, device=self.device)
		self.alpha = torch.tensor(np.exp(-dt / self.kwargs["tau_m"]), **f32)
		self.threshold = torch.tensor(self.kwargs["threshold"], **f32)
		self.gamma = torch.tensor(self.kwargs["gamma"], **f32)
		self.initialize_weights_()

	def _set_default_kwargs(self):
		self.kwargs.setdefault("tau_m", 10.0 * self.dt)
		self.kwargs.setdefault("threshold", 1.0)
		# The reference tests isinstance(<class>, HeavisideSigmoidApprox), which is never true, so its gamma
		# default is 1.0 whatever the surrogate (spiking_layers.py:127-130).  Kept for parity.
		self.kwargs.setdefault("gamma", 1.0)

	def initialize_weights_(self):
		gain = self.threshold.data
		for param in self.parameters():
			if param.ndim > 2:
				torch.nn.init.xavier_normal_(param, gain=gain)
			else:
				torch.nn.init.normal_(param, std=gain)

	def create_empty_state(self, batch_size: int = 1) -> Tuple[torch.Tensor, ...]:
		"""(V, Z), each (batch_size, output_size) zeros (reference :140-154)."""
		return self._zeros_state(batch_size, 2)

	# -- constants handed to the C ABI ----------------------------------------------------------------------------
	def snnk_consts(self, kappa: float = 0.0, tensor_core: bool = False) -> F_.LayerConsts:
		return F_.LayerConsts(
			layer_type=self.SNNK_LAYER_TYPE, surrogate=fused_surrogate(self.spike_func),
			recurrent=bool(self.use_recurrent_connection), alpha=float(self.alpha), rho=float(getattr(self, "rho", 0.0)),
			theta=float(self.threshold), gamma=float(self.gamma), kappa=kappa, tensor_core=tensor_core,
			spike_func=self.spike_func)

	def _beta_tensor(self) -> Optional[torch.Tensor]:
		return None

	def _step(self, inputs: torch.Tensor, state):
		"""One time step through the fused kernel (T = 1, dummy zero readout).  Not differentiable."""
		assert inputs.ndim == 2
		B = inputs.shape[0]
		state = self._init_forward_state(state, B)
		H = self.output_size
		if not hasattr(self, "_snnk_const_cache"):
			self._snnk_const_cache = self.snnk_consts()
		zero_out = torch.zeros((H, 1), dtype=torch.float32, device=inputs.device)
		zero_b = torch.zeros((1,), dtype=torch.float32, device=inputs.device)
		x = inputs.detach().float().reshape(B, 1, -1).contiguous()
		Hp = F_.padded_width(H)
		Wi, Wr, M, Wo = F_._pad_hidden(H, Hp, F_._c(self.forward_weights), F_._c(self.recurrent_weights),
			F_._c(self.rec_mask), zero_out)
		if Hp != H:
			state = tuple(torch.nn.functional.pad(F_._c(s_), (0, Hp - H)) for s_ in state)
		out = F_.run_forward(self._snnk_const_cache, x, Wi, Wr, M, F_._c(self._beta_tensor()), Wo, zero_b, traces=True,
			state=state)
		for k in ("V", "a", "Z"):
			if out[k] is not None:
				out[k] = out[k][..., :H]
		return out

	def forward(self, inputs: torch.Tensor, state: Tuple[torch.Tensor, ...] = None):
		out = self._step(inputs, state)
		next_V, next_Z = out["V"][:, 0], out["Z"][:, 0]
		return next_Z, (next_V, next_Z)


class ALIFLayer(LIFLayer):
	"""Adaptive LIF (reference spiking_layers.py:174-243): a_t = rho a_{t-1} + Z_{t-1}; A_t = theta + beta a_t."""
	SNNK_LAYER_TYPE = _cabi.SNNK_ALIF

	def __init__(self, input_size: int, output_size: int, use_recurrent_connection=True, use_rec_eye_mask=True,
			spike_func: Type[SpikeFunction] = HeavisideSigmoidApprox, dt=1e-3, device=None, **kwargs):
		super().__init__(
			input_size=input_size, output_size=output_size, use_recurrent_connection=use_recurrent_connection,
			use_rec_eye_mask=use_rec_eye_mask, spike_func=spike_func, dt=dt, device=device, **kwargs)
		f32 = dict(dtype=torch.float32, device=self.device)
		self.beta = torch.tensor(self.kwargs["beta"], **f32)
		# The reference indexes the caller's kwargs directly and raises KeyError when learn_beta is not passed
		# (spiking_layers.py:197); here the documented default (False) applies instead.
		if self.kwargs["learn_beta"]:
			self.beta = torch.nn.Parameter(self.beta, requires_grad=True)
		self.rho = torch.tensor(np.exp(-dt / self.kwargs["tau_a"]), **f32)

	def _set_default_kwargs(self):
		self.kwargs.setdefault("tau_m", 20.0 * self.dt)
		self.kwargs.setdefault("tau_a", 200.0 * self.dt)
		self.kwargs.setdefault("beta", 1.6)
		self.kwargs.setdefault("threshold", 0.03)
		self.kwargs.setdefault("gamma", 0.3)  # same never-true isinstance test as LIF (spiking_layers.py:206-209)
		self.kwargs.setdefault("learn_beta", False)

	def create_empty_state(self, batch_size: int = 1) -> Tuple[torch.Tensor, ...]:
		"""(V, a, Z) zeros (reference :212-227)."""
		return self._zeros_state(batch_size, 3)

	def _beta_tensor(self) -> Optional[torch.Tensor]:
		return self.beta.reshape(1)

	def forward(self, inputs: torch.Tensor, state: Tuple[torch.Tensor, ...] = None):
		out = self._step(inputs, state)
		next_V, next_a, next_Z = out["V"][:, 0], out["a"][:, 0], out["Z"][:, 0]
		return next_Z, (next_V, next_a, next_Z)


class IzhikevichLayer(RNNLayer):
	"""Third LayerType member of the reference (spiking_layers.py:246-353), SURVEY.md 8f.3.

	V' = (V + dt (k (V - v_rest)(V - v_th) - u + I) / C)(1 - Z) + c Z;  u' = u + dt a (b (V - v_rest) - u) + d Z;
	Z' = H(V' - v_peak).  Same kernels as LIF/ALIF with a different elementwise body (widths up to 128 on the register-resident kernels,
	wider layers on the fp32 kernels of recur_gen.cuh).
	"""
	SNNK_LAYER_TYPE = _cabi.SNNK_IZHIKEVICH

	def __init__(self, input_size: int, output_size: int, use_recurrent_connection=True, use_rec_eye_mask=True,
			spike_func: Type[SpikeFunction] = HeavisideSigmoidApprox, dt=1e-3, device=None, **kwargs):
		self.spike_func = spike_func
		super().__init__(
			input_size=input_size, output_size=output_size, use_recurrent_connection=use_recurrent_connection,
			use_rec_eye_mask=use_rec_eye_mask, dt=dt, device=device, **kwargs)
		for name in ("C", "v_rest", "v_th", "k", "a", "b", "c", "d", "v_peak", "gamma"):
			setattr(self, name, torch.tensor(self.kwargs[name], dtype=torch.float32, device=self.device))
		self.initialize_weights_()

	def _set_default_kwargs(self):
		# gamma: the reference's isinstance(<class>, HeavisideSigmoidApprox) test is never true, so 1.0 (:297-300)
		for k, v in dict(C=100.0, v_rest=-60.0, v_th=-40.0, k=0.7, a=0.03, b=-2.0, c=-50.0, d=100.0,
				v_peak=35.0, gamma=1.0).items():
			self.kwargs.setdefault(k, v)

	def create_empty_state(self, batch_size: int = 1) -> Tuple[torch.Tensor, ...]:
		"""(V = v_rest, u = 0, Z = 0), each (batch_size, output_size) (reference :308-328)."""
		V, u, Z = self._zeros_state(batch_size, 3)
		with torch.no_grad():
			V += self.v_rest
		return V, u, Z

	def snnk_consts(self, kappa: float = 0.0, tensor_core: bool = False) -> F_.LayerConsts:
		izh = tuple(float(v) for v in (self.dt, self.C, self.v_rest, self.v_th, self.k, self.a, self.b, self.c, self.d,
			self.v_peak))
		return F_.LayerConsts(
			layer_type=self.SNNK_LAYER_TYPE, surrogate=fused_surrogate(self.spike_func),
			recurrent=bool(self.use_recurrent_connection), alpha=0.0, rho=0.0, theta=float(self.v_peak),
			gamma=float(self.gamma), kappa=kappa, tensor_core=tensor_core, izh=izh, spike_func=self.spike_func)

	def _beta_tensor(self) -> Optional[torch.Tensor]:
		return None

	_step = LIFLayer._step

	def forward(self, inputs: torch.Tensor, state: Tuple[torch.Tensor, ...] = None):
		out = self._step(inputs, state)
		next_V, next_u, next_Z = out["V"][:, 0], out["a"][:, 0], out["Z"][:, 0]
		return next_Z, (next_V, next_u, next_Z)


class ReadoutLayer(RNNLayer):
	"""Leaky non-spiking readout y_t = kappa y_{t-1} + Z_t W_out + b (reference spiking_layers.py:356-408)."""

	def __init__(self, input_size: int, output_size: int, dt=1e-3, device=None, **kwargs):
		super().__init__(
			input_size=input_size, output_size=output_size, use_recurrent_connection=False, dt=dt, device=device,
			**kwargs)
		self.bias_weights = nn.Parameter(torch.empty((self.output_size,), device=self.device), requires_grad=True)
		self.kappa = torch.tensor(np.exp(-self.dt / self.kwargs["tau_out"]), dtype=torch.float32, device=self.device)
		self.initialize_weights_()

	def _set_default_kwargs(self):
		self.kwargs.setdefault("tau_out", 10.0 * self.dt)

	def initialize_weights_(self):
		super().initialize_weights_()
		torch.nn.init.constant_(self.bias_weights, 0.0)

	def create_empty_state(self, batch_size: int = 1) -> Tuple[torch.Tensor, ...]:
		return self._zeros_state(batch_size, 1)

	def forward(self, inputs: torch.Tensor, state: Tuple[torch.Tensor, ...] = None):
		# Stand-alone single step: one small library GEMM.  Inside SNN.forward the readout is fused into the
		# recurrence kernel (csrc/recur_fwd.cuh) and this method is not used.
		assert inputs.ndim == 2
		V, = self._init_forward_state(state, inputs.shape[0])
		next_V = self.kappa * V + torch.matmul(inputs, self.forward_weights) + self.bias_weights
		return next_V, (next_V,)


LayerType2Layer = {
	LayerType.LIF: LIFLayer,
	LayerType.ALIF: ALIFLayer,
	LayerType.Izhikevich: IzhikevichLayer,
}
