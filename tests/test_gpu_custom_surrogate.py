"""User-defined surrogate spike functions on every BPTT kernel family.

A ``SpikeFunction`` subclass with its own ``backward`` trains through the fused kernels: its ``backward`` is evaluated
once over the saved membrane trace and the sweep streams that sigma' trace (SNNK_SURROGATE_TRACE).

(a) ``RestatedFastSigmoid`` / ``RestatedPhi`` restate the built-in formulas in PyTorch operations, each one correctly
    rounded as in ``surrogate_grad`` (csrc/common.cuh), so in fp32 mode the gradients are bit-identical to the built-in
    classes'.  The tensor-core recurrence evaluates the built-ins with a hardware reciprocal (1 ulp), and tensor-core mode
    is held to the gradient tolerance of the other tensor-core tests.  Every case checks from the launched kernels that
    the family it targets ran with the trace instantiation.
(b) Surrogates the built-ins cannot express (arctan, Gaussian) against the PyTorch restatement of the reference.
(c) Training through ``_exec_batch`` (eager and graphed) and ``fit``.
(d) Stacked layers.
"""
import math
import re

import numpy as np
import pytest
import torch
from torch.autograd import DeviceType

from oracle import torch_port
from oracle.torch_port import TorchPortSNN
from _util import rel_err

pytestmark = pytest.mark.gpu

from snnimageclassification_b200 import LayerType, SNN, ToSpikes  # noqa: E402
from snnimageclassification_b200.modules.spike_funcs import (  # noqa: E402
	HeavisidePhiApprox, HeavisideSigmoidApprox, SpikeFunction)

DEV = torch.device("cuda:0")


def npy(t):
	return t.detach().cpu().numpy()


# ---- surrogates ------------------------------------------------------------------------------------------------------
class RestatedFastSigmoid(SpikeFunction):
	"""HeavisideSigmoidApprox's derivative written as oracle/torch_port.py writes it."""

	@staticmethod
	def backward(ctx, grad):
		v, thr, gamma = ctx.saved_tensors
		return grad / (gamma * (v - thr).abs() + 1.0) ** 2, None, None


class RestatedPhi(SpikeFunction):
	"""HeavisidePhiApprox's derivative written as oracle/torch_port.py writes it."""

	@staticmethod
	def backward(ctx, grad):
		v, thr, gamma = ctx.saved_tensors
		te = thr + 1e-5
		return grad * (gamma / te) * torch.clamp(1 - ((v - thr) / te).abs(), min=0.0), None, None


def arctan_f(v, thr, gamma):
	return 1.0 / (1.0 + (math.pi * gamma * (v - thr)) ** 2)


def gauss_f(v, thr, gamma):
	return torch.exp(-(gamma * (v - thr)) ** 2)


class ArctanSpike(SpikeFunction):
	@staticmethod
	def backward(ctx, grad):
		v, thr, gamma = ctx.saved_tensors
		return grad * arctan_f(v, thr, gamma), None, None


class GaussSpike(SpikeFunction):
	@staticmethod
	def backward(ctx, grad):
		v, thr, gamma = ctx.saved_tensors
		return grad * gauss_f(v, thr, gamma), None, None


def cpu_twin(f):
	"""The same surrogate as a plain autograd Function for the CPU restatement of the reference."""
	class Twin(torch.autograd.Function):
		@staticmethod
		def forward(ctx, v, thr, gamma):
			ctx.save_for_backward(v, thr, gamma)
			return (v >= thr).to(v.dtype)

		@staticmethod
		def backward(ctx, g):
			v, thr, gamma = ctx.saved_tensors
			return g * f(v, thr, gamma), None, None
	return Twin


# ---- which kernels ran (as tests/test_gpu_readout_width.py) ------------------------------------------------------------
def launched(fn):
	torch.cuda.synchronize()
	with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
		res = fn()
		torch.cuda.synchronize()
	names = [e.name for e in prof.events() if e.device_type == DeviceType.CUDA]
	assert any("snnk::" in n for n in names), f"the profiler reports no kernel of the library: {names[:8]}"
	return res, names


def bwd_kernels(names):
	"""{(kernel, template arguments)} of the BPTT sweeps that ran."""
	out = set()
	for n in names:
		m = re.search(r"(k_recur_bwd|k_recur_bwd_lean|k_recur_bwd_tc|k_nonrec_bwd|k_wide_bwd|k_recur_bwd_gen)<([^<>]*)>", n)
		if m:
			out.add((m.group(1), tuple(s.strip() for s in m.group(2).split(","))))
	return out


# ---- (a) restated built-ins on every family ------------------------------------------------------------------------------
def make_net(spike_func, H, layer, rec, tc, T, seed, N=64, O=10, **kw):
	torch.manual_seed(seed)
	dt = 1.0 if layer == LayerType.Izhikevich else 1e-3
	net = SNN(N, O, H, use_recurrent_connection=rec, int_time_steps=T, dt=dt, spike_func=spike_func,
		hidden_layer_type=layer, device=DEV, tensor_core=tc, cuda_graphs=False, **kw)
	if layer == LayerType.Izhikevich:      # drive that makes an Izhikevich layer spike (tests/test_gpu_readout_width.py)
		L = net.layers["input"]
		with torch.no_grad():
			L.forward_weights.mul_(25.0).add_(20.0)
			if rec:
				L.recurrent_weights.mul_(5.0)
	elif H > 128 and rec:
		with torch.no_grad():
			net.layers["input"].recurrent_weights.div_(4.0)
	net.train()
	return net


def grads(net):
	L, R = net.layers[list(net.layers)[-2]], net.layers["readout"]
	out = {"dW_in": L.forward_weights.grad, "dW_out": R.forward_weights.grad, "db": R.bias_weights.grad}
	if L.recurrent_weights is not None:
		out["dW_rec"] = L.recurrent_weights.grad
	for name in list(net.layers)[:-2]:
		out[name + ".dW_in"] = net.layers[name].forward_weights.grad
	return out


def train_step(net, x, y):
	loss = net.batch_loss(x, y)
	net.zero_grad()
	loss.backward()
	return loss.detach().clone()


# family: (H, layer types, recurrent, tensor_core, B, T, SNNK_MMA_RECUR, encoder input with a run table)
FAMILIES = {
	"simt_r1_h32": (32, "LA", (True, False), False, 24, 16, "0", False),
	"simt_r1_h64": (64, "LA", (True, False), False, 24, 16, "0", False),
	"simt_r2": (128, "LA", (True, False), False, 1030, 6, "0", False),
	"lean_fp32": (128, "LA", (True,), False, 48, 20, "0", False),
	"lean_planes": (128, "LA", (True,), True, 48, 20, "0", False),
	"lean_runs": (128, "LA", (True,), True, 48, 20, "0", True),
	"tc_recur": (128, "LA", (True,), True, 1024, 12, None, False),
	"nonrec": (128, "LA", (False,), True, 48, 20, "0", False),
	"wide_tc_256": (256, "LA", (True,), True, 12, 10, "0", False),
	"wide_tc_512": (512, "LA", (True,), True, 12, 10, "0", False),
	"wide_gen": (256, "LA", (True, False), False, 12, 10, "0", False),
	"izh_simt": (128, "I", (True, False), False, 12, 25, "0", False),
	"izh_gen": (256, "I", (True, False), False, 12, 25, "0", False),
}
LAYERS = {"L": LayerType.LIF, "A": LayerType.ALIF, "I": LayerType.Izhikevich}


def expected_sweep(family, H, rec, B, lt, trace, sid):
	"""(kernel, template arguments) the dispatcher must launch.  With the sigma' trace (SURR = 2) ALIF runs the LIF-mode
	instantiation: the trace replaces the only read of its threshold."""
	alif = lt == "A" and not trace
	s, a, r = ("2" if trace else str(sid)), ("true" if alif else "false"), ("true" if rec else "false")
	if family.startswith("simt") or family == "izh_simt":
		return ("k_recur_bwd", (str(H), "2" if B > 1024 else "1", r, "2" if lt == "I" else ("1" if alif else "0"), s))
	if family.startswith("lean"):
		return ("k_recur_bwd_lean", (a, s, "false" if family == "lean_fp32" else "true",
			"true" if family == "lean_runs" else "false", "12"))
	if family == "tc_recur":
		return ("k_recur_bwd_tc", (a, s))
	if family == "nonrec":
		return ("k_nonrec_bwd", (str(H), a, s))
	if family.startswith("wide_tc"):
		return ("k_wide_bwd", None, (a, s))
	return ("k_recur_bwd_gen", None, (r, "true" if trace else "false"))


def check_sweep(names, want):
	got = bwd_kernels(names)
	assert len(got) == 1, got
	(kern, args), = got
	assert kern == want[0], (got, want)
	if len(want) == 2:
		assert args == want[1], (got, want)
	else:      # leading NSM / NPT, R arguments depend on the width
		assert args[-len(want[2]):] == want[2], (got, want)


@pytest.mark.parametrize("family", list(FAMILIES))
def test_restated_builtins_match_builtins(family, monkeypatch):
	H, layers, recs, tc, B, T, mma, encoded = FAMILIES[family]
	monkeypatch.delenv("SNNK_LEAN", raising=False)
	if mma is None:
		monkeypatch.delenv("SNNK_MMA_RECUR", raising=False)
	else:
		monkeypatch.setenv("SNNK_MMA_RECUR", mma)
	for lt in layers:
		layer = LAYERS[lt]
		for rec in recs:
			for builtin, restated in ((HeavisideSigmoidApprox, RestatedFastSigmoid), (HeavisidePhiApprox, RestatedPhi)):
				if family in ("tc_recur", "simt_r2", "wide_tc_512") and builtin is HeavisidePhiApprox:
					continue      # the largest geometries: one surrogate is enough
				seed = sum(map(ord, f"{family}{lt}{rec}{builtin.__name__}"))
				g = torch.Generator().manual_seed(seed)
				N = 64
				if encoded:
					img = (torch.randint(1, 256, (B, N), generator=g).float() / 255.0) * (torch.rand(B, N, generator=g) < 0.3)
					x = ToSpikes(T, use_periods=True).encode_batch(img.to(DEV))
				else:
					x = (torch.rand(B, T, N, generator=g) < 0.2).float().to(DEV)
				y = torch.randint(0, 10, (B,), generator=g).to(DEV)
				res = {}
				for func in (builtin, restated):
					net = make_net(func, H, layer, rec, tc, T, seed)
					loss, names = launched(lambda: train_step(net, x, y))
					check_sweep(names, expected_sweep(family, H, rec, B, lt, func is restated, builtin.SURROGATE_ID))
					res[func] = (loss, grads(net))
				(l0, g0), (l1, g1) = res[builtin], res[restated]
				assert torch.equal(l0, l1)
				assert float(g0["dW_out"].abs().max()) > 0
				for k in g0:
					if tc:
						assert rel_err(npy(g1[k]), npy(g0[k])) <= 1e-4, (k, rel_err(npy(g1[k]), npy(g0[k])))
					else:
						assert torch.equal(g0[k], g1[k]), (k, rel_err(npy(g1[k]), npy(g0[k])))


# ---- (b) new surrogates against the PyTorch restatement of the reference --------------------------------------------------
def port_for(net, layer_type, surrogate_key, rec, T, learn_beta=False):
	L, R = net.layers["input"], net.layers["readout"]
	H, O, N = L.output_size, R.output_size, L.input_size
	kw = dict(dt=float(L.dt)) if layer_type == 2 else {}
	port = TorchPortSNN(N, H, O, T, layer_type=layer_type, surrogate=surrogate_key, recurrent=rec, seed=0,
		learn_beta=learn_beta, **kw)
	port.load(npy(L.forward_weights), npy(L.recurrent_weights) if rec else None, npy(R.forward_weights),
		npy(R.bias_weights), beta=float(L.beta) if layer_type == 1 else None)
	return port


def check_vs_port(net, port, x, y, rec):
	loss = train_step(net, x, y)
	lp = port.exec_batch(x.float().cpu(), y.cpu())
	assert abs(float(loss) - lp) <= 1e-4 * abs(lp), (float(loss), lp)
	L, R = net.layers["input"], net.layers["readout"]
	pairs = [(L.forward_weights, port.W_in), (R.forward_weights, port.W_out), (R.bias_weights, port.b_out)]
	if rec:
		pairs.append((L.recurrent_weights, port.W_rec))
	assert float(port.W_out.grad.abs().max()) > 0
	for mine, theirs in pairs:
		assert rel_err(npy(mine.grad), npy(theirs.grad)) <= 1e-4, rel_err(npy(mine.grad), npy(theirs.grad))


SURR = {"arctan": (ArctanSpike, arctan_f), "gauss": (GaussSpike, gauss_f)}


@pytest.mark.parametrize("H", [128, 256])
@pytest.mark.parametrize("rec", [True, False])
@pytest.mark.parametrize("lt", ["L", "A", "I"])
@pytest.mark.parametrize("surr", list(SURR))
def test_new_surrogates_vs_torch_port(surr, lt, rec, H, monkeypatch):
	cls, f = SURR[surr]
	monkeypatch.setitem(torch_port.SURROGATES, surr, cpu_twin(f))
	B, T, N = 16, 25 if lt == "I" else 20, 64
	net = make_net(cls, H, LAYERS[lt], rec, False, T, seed=7 + H)
	port = port_for(net, "LAI".index(lt), surr, rec, T)
	g = torch.Generator().manual_seed(H + 3)
	x = (torch.rand(B, T, N, generator=g) < 0.2).float()
	y = torch.randint(0, 10, (B,), generator=g)
	check_vs_port(net, port, x.to(DEV), y.to(DEV), rec)


@pytest.mark.parametrize("surr", list(SURR))
def test_new_surrogate_on_the_bench_workload(surr, monkeypatch):
	"""ALIF 784-128-10, recurrent, learn_beta, periodic encoder, B = 256, T = 100 (bench.py's training step)."""
	cls, f = SURR[surr]
	monkeypatch.setitem(torch_port.SURROGATES, surr, cpu_twin(f))
	B, T, N = 256, 100, 784
	torch.manual_seed(0)
	enc = ToSpikes(T, use_periods=True)
	net = SNN(N, 10, 128, use_recurrent_connection=True, int_time_steps=T, spike_func=cls, hidden_layer_type=LayerType.ALIF,
		device=DEV, learn_beta=True, input_encoder=enc, cuda_graphs=False)
	net.train()
	port = port_for(net, 1, surr, True, T, learn_beta=True)
	g = torch.Generator().manual_seed(11)
	img = (torch.randint(1, 256, (B, N), generator=g).float() / 255.0) * (torch.rand(B, N, generator=g) < 0.19)
	y = torch.randint(0, 10, (B,), generator=g)
	x = enc.encode_batch(img.to(DEV))
	check_vs_port(net, port, x, y.to(DEV), True)
	assert net.layers["input"].beta.grad is None


# ---- (c) training ---------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("lt", ["L", "A"])
def test_exec_batch_eager_and_graphed_are_bit_identical(lt):
	B, T, N, steps = 32, 16, 784, 4

	def make():
		torch.manual_seed(5)
		net = SNN(N, 10, 128, use_recurrent_connection=True, int_time_steps=T, spike_func=GaussSpike,
			hidden_layer_type=LAYERS[lt], device=DEV)
		net.train()
		return net, torch.optim.SGD(net.parameters(), lr=0.05)
	(eager, oe), (graphed, og) = make(), make()
	eager.cuda_graphs = False
	g = torch.Generator().manual_seed(9)
	crit = torch.nn.NLLLoss()
	for it in range(steps):
		x = (torch.rand(B, T, N, generator=g) < 0.1).float()
		y = torch.randint(0, 10, (B,), generator=g)
		le = eager._exec_batch(x, y, crit, oe)
		lg = graphed._exec_batch(x, y, crit, og)
		assert np.isfinite(le) and le == lg, (it, le, lg)
	assert len(graphed._graphed_steps) == 1
	for pe, pg in zip(eager.parameters(), graphed.parameters()):
		assert torch.equal(pe, pg)


def test_fit_runs_an_epoch_with_a_custom_surrogate(tmp_path):
	from snnimageclassification_b200.datasets.datasets import SyntheticSpikeImages
	torch.manual_seed(0)
	T = 20
	net = SNN(784, 10, 128, use_recurrent_connection=True, int_time_steps=T, spike_func=ArctanSpike,
		hidden_layer_type=LayerType.ALIF, device=DEV, learn_beta=True, input_encoder=ToSpikes(T, use_periods=True, tau=20.0),
		checkpoint_folder=str(tmp_path / "ck"))
	ds = SyntheticSpikeImages(256, seed=1)
	train = torch.utils.data.DataLoader(ds, batch_size=64, shuffle=False)
	before = [p.detach().clone() for p in net.parameters()]
	hist = net.fit(train, train, nb_epochs=1, force_overwrite=True, verbose=False)
	assert len(hist["train"]) == 1 and np.isfinite(hist["train"][-1])
	assert any(not torch.equal(b, p) for b, p in zip(before, net.parameters()))


def test_base_spike_function_infers_but_does_not_train():
	net = make_net(SpikeFunction, 64, LayerType.LIF, True, False, 8, seed=1)
	x = (torch.rand(4, 8, 64) < 0.2).float().to(DEV)
	with torch.no_grad():
		y, _ = net(x)
	assert torch.isfinite(y).all()
	loss = net.batch_loss(x, torch.zeros(4, dtype=torch.long, device=DEV))
	with pytest.raises(NotImplementedError):
		loss.backward()


# ---- (d) stacked layers -----------------------------------------------------------------------------------------------
@pytest.mark.parametrize("tc", [False, True])
def test_stacked_layers_restated_matches_builtin(tc):
	B, T, N = 24, 16, 64
	g = torch.Generator().manual_seed(3)
	x = (torch.rand(B, T, N, generator=g) < 0.3).float().to(DEV)
	y = torch.randint(0, 10, (B,), generator=g).to(DEV)
	res = {}
	for func in (HeavisideSigmoidApprox, RestatedFastSigmoid):
		torch.manual_seed(2)
		net = SNN(N, 10, [128, 128], use_recurrent_connection=True, int_time_steps=T, spike_func=func,
			hidden_layer_type=LayerType.ALIF, device=DEV, tensor_core=tc, cuda_graphs=False)
		net.train()
		res[func] = (train_step(net, x, y), grads(net))
	(l0, g0), (l1, g1) = res.values()
	assert torch.equal(l0, l1) and "input.dW_in" in g0
	assert float(g0["input.dW_in"].abs().max()) > 0
	for k in g0:
		if tc:
			assert rel_err(npy(g1[k]), npy(g0[k])) <= 1e-4, k
		else:
			assert torch.equal(g0[k], g1[k]), k
