"""User-defined surrogate spike functions: classification of the classes and the sigma' helper (no GPU needed)."""
import numpy as np
import pytest
import torch

from snnimageclassification_b200 import _cabi
from snnimageclassification_b200.modules import functional as F_
from snnimageclassification_b200.modules.spike_funcs import (
	HeavisidePhiApprox, HeavisideSigmoidApprox, SpikeFunction, fused_surrogate)
from snnimageclassification_b200.modules.spiking_layers import ALIFLayer, IzhikevichLayer, LIFLayer

CPU = torch.device("cpu")


class Arctan(SpikeFunction):
	@staticmethod
	def backward(ctx, grad):
		v, thr, gamma = ctx.saved_tensors
		return grad / (1.0 + (np.pi * gamma * (v - thr)) ** 2), None, None


class OwnForward(SpikeFunction):
	@staticmethod
	def forward(ctx, inputs, threshold=torch.tensor(1.0), gamma=torch.tensor(0.3)):
		return torch.sigmoid(inputs - threshold)

	@staticmethod
	def backward(ctx, grad):
		return grad, None, None


class WrongShape(SpikeFunction):
	@staticmethod
	def backward(ctx, grad):
		v, thr, gamma = ctx.saved_tensors
		return (grad * v)[..., :1], None, None


def test_classification_of_spike_function_classes():
	assert fused_surrogate(HeavisideSigmoidApprox) == _cabi.SNNK_FAST_SIGMOID
	assert fused_surrogate(HeavisidePhiApprox) == _cabi.SNNK_PHI
	assert fused_surrogate(Arctan) == _cabi.SNNK_SURROGATE_TRACE == 2
	# the base class keeps its place on the trace path: inference runs, its backward raises NotImplementedError
	assert fused_surrogate(SpikeFunction) == _cabi.SNNK_SURROGATE_TRACE
	with pytest.raises(NotImplementedError, match="OwnForward"):
		fused_surrogate(OwnForward)
	with pytest.raises(TypeError):
		fused_surrogate(torch.sigmoid)


@pytest.mark.parametrize("layer_cls", [LIFLayer, ALIFLayer, IzhikevichLayer])
def test_layer_constants_carry_the_class(layer_cls):
	c = layer_cls(8, 32, spike_func=Arctan, device=CPU).snnk_consts()
	assert c.surrogate == _cabi.SNNK_SURROGATE_TRACE and c.spike_func is Arctan
	assert F_.make_desc(c, 2, 3, 8, 32, 10, True).surrogate == 2
	c = layer_cls(8, 32, spike_func=HeavisidePhiApprox, device=CPU).snnk_consts()
	assert c.surrogate == _cabi.SNNK_PHI
	with pytest.raises(NotImplementedError, match="OwnForward"):
		layer_cls(8, 32, spike_func=OwnForward, device=CPU).snnk_consts()


def _traces(shape=(3, 5, 32), seed=0):
	g = torch.Generator().manual_seed(seed)
	V = torch.randn(shape, generator=g) * 0.05
	a = torch.rand(shape, generator=g) * 0.1
	return V, a


def test_sigma_trace_lif_matches_the_formula():
	V, _ = _traces()
	c = LIFLayer(8, 32, spike_func=Arctan, device=CPU).snnk_consts()
	sg = F_.surrogate_trace(c, V, None, None)
	assert sg.shape == V.shape and sg.dtype == torch.float32 and sg.is_contiguous()
	theta, gamma = np.float32(c.theta), np.float32(c.gamma)
	want = 1.0 / (1.0 + (np.pi * gamma * (V.double().numpy() - theta)) ** 2)
	assert np.abs(sg.numpy() - want).max() <= 1e-6


def test_sigma_trace_alif_uses_the_per_step_threshold():
	V, a = _traces(seed=1)
	layer = ALIFLayer(8, 32, spike_func=Arctan, device=CPU)
	c = layer.snnk_consts()
	beta = layer.beta.reshape(1)
	sg = F_.surrogate_trace(c, V, a, beta)
	# theta + beta a_t with two fp32 roundings, as the kernels form the threshold
	thr = (beta * a) + torch.tensor(c.theta, dtype=torch.float32)
	want = 1.0 / (1.0 + (np.float32(np.pi) * np.float32(c.gamma) * (V - thr).numpy()) ** 2)
	assert np.abs(sg.numpy() - want).max() <= 1e-6
	# the adaptation matters: with the threshold held at theta the result differs
	assert np.abs(F_.surrogate_trace(c, V, torch.zeros_like(a), beta).numpy() - want).max() > 1e-3


def test_sigma_trace_izhikevich_uses_v_peak():
	layer = IzhikevichLayer(8, 32, spike_func=Arctan, device=CPU)
	c = layer.snnk_consts()
	V = torch.linspace(-70.0, 40.0, 3 * 5 * 32).reshape(3, 5, 32)
	sg = F_.surrogate_trace(c, V, torch.zeros_like(V), None)
	want = 1.0 / (1.0 + (np.pi * float(layer.gamma) * (V.double().numpy() - float(layer.v_peak))) ** 2)
	assert np.abs(sg.numpy() - want).max() <= 1e-6
	assert float(sg.max()) > 0.5      # the peak of the surrogate sits at v_peak


def test_sigma_trace_restated_fast_sigmoid_is_bit_identical_to_the_formula_in_fp32():
	class Restated(SpikeFunction):
		@staticmethod
		def backward(ctx, grad):
			v, thr, gamma = ctx.saved_tensors
			return grad / (gamma * (v - thr).abs() + 1.0) ** 2, None, None
	V, a = _traces(seed=2)
	layer = ALIFLayer(8, 32, spike_func=Restated, device=CPU)
	c = layer.snnk_consts()
	sg = F_.surrogate_trace(c, V, a, layer.beta.reshape(1))
	f = np.float32
	thr = f(c.theta) + f(layer.beta.item()) * a.numpy()
	d = f(c.gamma) * np.abs(V.numpy() - thr) + f(1.0)
	assert np.array_equal(sg.numpy(), f(1.0) / (d * d))


def test_sigma_trace_refuses_bad_results_and_the_base_class():
	V, _ = _traces()
	c = LIFLayer(8, 32, spike_func=WrongShape, device=CPU).snnk_consts()
	with pytest.raises(TypeError, match="WrongShape"):
		F_.surrogate_trace(c, V, None, None)
	c = LIFLayer(8, 32, spike_func=SpikeFunction, device=CPU).snnk_consts()
	with pytest.raises(NotImplementedError):
		F_.surrogate_trace(c, V, None, None)
