"""The fused training kernel (recur_lean.cuh, k_train_lean): forward, head and BPTT sweep of a row in one CTA.

The captured training step (GraphedTrainStep) runs it where the lean forward and sweep kernels would run; everywhere
else, and for any backward gradient other than the step's own root gradient, the two kernels run as before.  The fused
kernel does the same arithmetic in the same order, so everything here is compared bit for bit.
"""
import ctypes
import re

import numpy as np
import pytest
import torch
from torch.autograd import DeviceType

pytestmark = pytest.mark.gpu

from snnimageclassification_b200 import SNN, FusedAdam, LayerType, SpikeFuncType, ToSpikes, _cabi  # noqa: E402
from snnimageclassification_b200.modules import functional as F_  # noqa: E402

from test_gpu_guardbands import Guarded  # noqa: E402

DEV = torch.device("cuda:0")
N, H = 784, 128


def _net(layer, spike, O, T, tc):
	torch.manual_seed(0)
	alif = layer == "ALIF"
	return SNN(N, O, H, use_recurrent_connection=True, int_time_steps=T, device=DEV, tensor_core=tc,
		spike_func=SpikeFuncType.FastSigmoid if spike == "fs" else SpikeFuncType.Phi,
		hidden_layer_type=LayerType.ALIF if alif else LayerType.LIF, **({"learn_beta": True} if alif else {}))


def _batch(B, T, O, dedup, seed=7):
	g = torch.Generator().manual_seed(seed)
	labels = torch.randint(0, O, (B,), generator=g).to(DEV)
	if dedup:      # encoder output with its run table: the frame-dedup kernels
		img = (torch.randint(1, 256, (B, N), generator=g).float() / 255.0) * (torch.rand(B, N, generator=g) < 0.19)
		x = ToSpikes(T, use_periods=True).encode_batch(img.to(DEV))
		assert F_.get_runs(x) is not None
	else:          # a dense binary raster without a table
		x = F_.mark_binary((torch.rand(B, T, N, generator=g) < 0.2).float().to(DEV))
	return x, labels


def _kernels(fn):
	torch.cuda.synchronize()
	with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
		fn()
		torch.cuda.synchronize()
	names = [e.name for e in prof.events() if e.device_type == DeviceType.CUDA]
	assert any("snnk::" in n for n in names), f"the profiler reports no kernel of the library: {names[:8]}"
	return names


def _ran(names, pattern):
	return any(re.search(pattern, n) for n in names)


CASES = {
	"alif_fs_tc_dedup_o10": ("ALIF", "fs", 10, 100, True, True),
	"lif_phi_tc_dense_o12": ("LIF", "phi", 12, 23, True, False),
	"alif_phi_fp32_dense_o1": ("ALIF", "phi", 1, 23, False, False),
	"lif_fs_tc_dedup_o1_t37": ("LIF", "fs", 1, 37, True, True),
	"alif_fs_fp32_dense_o12_t10": ("ALIF", "fs", 12, 10, False, False),
	"alif_phi_tc_dedup_o12_t51": ("ALIF", "phi", 12, 51, True, True),
}


@pytest.mark.parametrize("case", list(CASES))
def test_graphed_step_matches_eager(case):
	"""Several captured steps (fused kernel) against the same steps run eagerly (lean forward + lean sweep): loss and
	every updated parameter bit-identical after each step."""
	layer, spike, O, T, tc, dedup = CASES[case]
	B = 37
	x, y = _batch(B, T, O, dedup)
	crit = torch.nn.NLLLoss()
	ref, net = _net(layer, spike, O, T, tc), _net(layer, spike, O, T, tc)
	opt_ref = FusedAdam(ref.parameters(), lr=1e-3, weight_decay=1e-5)
	opt = FusedAdam(net.parameters(), lr=1e-3, weight_decay=1e-5)
	ref.train(); net.train()
	step = net.graphed_train_step(x, y, crit, opt, static_inputs=True)
	names = _kernels(step)
	assert _ran(names, r"k_train_lean<") and not _ran(names, r"k_recur_bwd_lean<"), names
	# the profiled replay was step 1 of the captured arm
	for k in range(4):
		if k > 0:
			step()
		loss_ref = ref.batch_loss(x, y, crit)
		opt_ref.zero_grad()
		loss_ref.backward()
		opt_ref.step()
		assert float(step.loss) == float(loss_ref), (k, float(step.loss), float(loss_ref))
		for (name, p), q in zip(ref.named_parameters(), net.parameters()):
			assert torch.equal(p, q), f"step {k}: {name} differs"


def test_logp_and_gradients_of_the_fused_forward():
	"""Outside a graph: a forward on the fused path whose backward receives the published root gradient gives the
	eager path's loss, log-probabilities and gradients."""
	x, y = _batch(29, 41, 10, True)
	ref, net = _net("ALIF", "fs", 10, 41, True), _net("ALIF", "fs", 10, 41, True)
	ws = (ref._weights(), net._weights())
	root = F_._const_scalar(1.0, DEV)
	loss_r, logp_r, *_ = F_.SpikingSequenceNLL.apply(ref._consts(), x, y, *ws[0], False)
	loss_r.backward(gradient=root)
	F_.SWEEP_SCALE = root
	try:
		names = _kernels(lambda: F_.SpikingSequenceNLL.apply(net._consts(), x, y, *ws[1], False))
		assert _ran(names, r"k_train_lean<"), names
		loss, logp, *_ = F_.SpikingSequenceNLL.apply(net._consts(), x, y, *ws[1], False)
	finally:
		F_.SWEEP_SCALE = None
	names = _kernels(lambda: loss.backward(gradient=root))
	assert not _ran(names, r"k_recur_bwd_lean<|k_recur_fwd"), names
	assert float(loss) == float(loss_r) and torch.equal(logp, logp_r)
	for (name, p), q in zip(ref.named_parameters(), net.parameters()):
		assert (p.grad is None) == (q.grad is None), name
		if p.grad is not None:
			assert torch.equal(p.grad, q.grad), f"{name}.grad differs"


def test_other_gradient_falls_back_to_the_regular_sweep():
	"""A forward on the fused path followed by loss.backward(2.0): the sweep it ran was for 1.0, so the backward
	recomputes the traces and runs the regular sweep -- and matches the eager result."""
	x, y = _batch(33, 23, 10, True)
	ref, net = _net("ALIF", "fs", 10, 23, True), _net("ALIF", "fs", 10, 23, True)
	two = torch.tensor(2.0, device=DEV)
	ref.batch_loss(x, y).backward(gradient=two)
	F_.SWEEP_SCALE = F_._const_scalar(1.0, DEV)
	try:
		loss = net.batch_loss(x, y)
	finally:
		F_.SWEEP_SCALE = None
	names = _kernels(lambda: loss.backward(gradient=two))
	assert _ran(names, r"k_recur_bwd_lean<"), names
	for (name, p), q in zip(ref.named_parameters(), net.parameters()):
		if p.grad is not None:
			assert torch.equal(p.grad, q.grad), f"{name}.grad differs"


@pytest.mark.parametrize("O,fused", [(12, True), (13, False)])
def test_selection_at_the_readout_threshold(O, fused):
	"""The graph replay runs the fused kernel up to 12 classes and the forward + sweep pair from 13 on."""
	x, y = _batch(37, 23, O, True)
	net = _net("ALIF", "fs", O, 23, True)
	net.train()
	step = net.graphed_train_step(x, y, torch.nn.NLLLoss(), FusedAdam(net.parameters(), lr=1e-3), static_inputs=True)
	names = _kernels(step)
	assert _ran(names, r"k_train_lean<") == fused, names
	assert _ran(names, r"k_recur_bwd_lean<") != fused, names


@pytest.mark.parametrize("B,T,layer,tc,dedup", [(37, 23, 1, True, True), (21, 10, 0, True, False), (9, 37, 1, False, False)])
def test_sweep_entry_guard_bands_and_parity(B, T, layer, tc, dedup):
	"""snnk_forward_nll_sweep + snnk_backward(SNNK_F_SWEEP_DONE) with every output and both workspaces between guard
	bands: nothing written outside them, every output written, and all of it bit-identical to snnk_forward_nll +
	snnk_backward of the same inputs."""
	O, Nx = 10, 64
	g = torch.Generator().manual_seed(B * 100 + T)
	theta = 0.03 if layer else 1.0
	consts = F_.LayerConsts(layer, 0, True, float(np.float32(np.exp(-1 / 20))), float(np.float32(np.exp(-1 / 200))), theta,
		0.3 if layer else 1.0, float(np.float32(np.exp(-1 / 10))), tensor_core=tc)
	if dedup:
		img = (torch.randint(1, 256, (B, Nx), generator=g).float() / 255.0) * (torch.rand(B, Nx, generator=g) < 0.3)
		x = ToSpikes(T, use_periods=True).encode_batch(img.to(DEV))
	else:
		x = F_.mark_binary((torch.rand(B, T, Nx, generator=g) < 0.15).float().to(DEV))
	W_in = (torch.randn(Nx, H, generator=g) * theta).to(DEV)
	W_rec = (torch.randn(H, H, generator=g) * theta).to(DEV)
	mask = (1 - torch.eye(H)).to(DEV)
	W_out = torch.randn(H, O, generator=g).to(DEV)
	b_out = (torch.randn(O, generator=g) * 0.1).to(DEV)
	beta = torch.tensor([1.6], device=DEV) if layer else None
	labels = torch.randint(0, O, (B,), generator=g).to(DEV)
	scale = torch.tensor([0.75], device=DEV)
	runs = F_.get_runs(x)
	lib, p = _cabi.lib(), _cabi.ptr
	desc = F_.make_desc(consts, B, T, Nx, H, O, False, binary=True)
	fwd_bytes = max(int(lib.snnk_forward_workspace_bytes(ctypes.byref(desc))), 16)
	bwd_bytes = max(int(lib.snnk_backward_workspace_bytes(ctypes.byref(desc))), 16)

	def outputs():
		return {"Z": Guarded((B, T, H)), "zbits": Guarded((B, T, H // 32), torch.int32), "y": Guarded((B, T, O)),
			"logits": Guarded((B, O)), "tstar": Guarded((B, O), torch.int32), "logp": Guarded((B, O)), "loss": Guarded((1,)),
			"g_logits": Guarded((B, O)), "dW_in": Guarded((Nx, H)), "dW_rec": Guarded((H, H)), "dW_out": Guarded((H, O)),
			"db": Guarded((O,))}

	def backward(G, desc_b, ws_b, V, a, W_effT):
		rc = lib.snnk_backward(ctypes.byref(desc_b), p(x), p(W_rec), p(mask), p(beta), p(W_out), None, p(V), p(a),
			p(G["Z"].t), p(G["zbits"].t), None, p(G["g_logits"].t), p(G["tstar"].t), p(scale), None, None, p(G["dW_in"].t),
			p(G["dW_rec"].t), p(G["dW_out"].t), p(G["db"].t), p(ws_b), ws_b.numel(), p(runs), p(W_effT), _cabi.stream_ptr())
		_cabi.check(rc, "snnk_backward")

	# reference: forward with traces + head, then the regular backward
	R = outputs()
	desc_t = F_.make_desc(consts, B, T, Nx, H, O, True, binary=True)
	V = torch.empty((B, T, H), device=DEV)
	a = torch.empty((B, T, H), device=DEV) if layer else None
	W_effT = torch.empty((H, H), device=DEV)
	ws_f = torch.empty(fwd_bytes, dtype=torch.uint8, device=DEV)
	head_ws = torch.zeros(B + 1, dtype=torch.int32, device=DEV)
	rc = lib.snnk_forward_nll(ctypes.byref(desc_t), p(x), p(W_in), p(W_rec), p(mask), p(beta), p(W_out), p(b_out), None, None,
		None, p(V), p(a), p(R["Z"].t), p(R["zbits"].t), p(R["y"].t), p(R["logits"].t), p(R["tstar"].t), p(ws_f), fwd_bytes,
		p(runs), p(W_effT), p(labels), p(R["logp"].t), p(R["loss"].t), p(R["g_logits"].t), p(head_ws), None, None,
		_cabi.stream_ptr())
	_cabi.check(rc, "snnk_forward_nll")
	backward(R, desc_t, torch.empty(bwd_bytes, dtype=torch.uint8, device=DEV), V, a, W_effT)

	# fused: forward + head + sweep, then the rest of the backward
	G = outputs()
	ws_fg = Guarded((fwd_bytes,), torch.uint8)
	ws_bg = Guarded((bwd_bytes,), torch.uint8)
	names = _kernels(lambda: _cabi.check(lib.snnk_forward_nll_sweep(ctypes.byref(desc), p(x), p(W_in), p(W_rec), p(mask),
		p(beta), p(W_out), p(b_out), None, None, None, None, None, p(G["Z"].t), p(G["zbits"].t), p(G["y"].t), p(G["logits"].t),
		p(G["tstar"].t), p(ws_fg.t), fwd_bytes, p(runs), None, p(labels), p(G["logp"].t), p(G["loss"].t), p(G["g_logits"].t),
		p(head_ws), None, None, p(scale), p(ws_bg.t), bwd_bytes, _cabi.stream_ptr()), "snnk_forward_nll_sweep"))
	assert _ran(names, r"k_train_lean<"), names
	desc_d = F_.make_desc(consts, B, T, Nx, H, O, True, binary=True)
	desc_d.flags |= _cabi.SNNK_F_SWEEP_DONE
	backward(G, desc_d, ws_bg.t, None, None, None)
	torch.cuda.synchronize()
	for k, gb in G.items():
		gb.check(k, written=k not in ("zbits", "tstar"))
		assert torch.equal(gb.t, R[k].t), f"{k} differs from snnk_forward_nll + snnk_backward"
	ws_fg.check("forward workspace", written=False)
	ws_bg.check("backward workspace", written=False)


def test_sweep_entry_refuses_what_it_does_not_fuse():
	"""Not eligible (here: a user-defined surrogate, and a request for the V / a traces): SNNK_ERR_UNSUPPORTED, and
	nothing was launched -- the outputs keep their sentinel."""
	B, T, O, Nx = 8, 12, 10, 64
	lib, p = _cabi.lib(), _cabi.ptr
	x = F_.mark_binary(torch.zeros(B, T, Nx, device=DEV))
	W_in, W_rec = torch.zeros(Nx, H, device=DEV), torch.zeros(H, H, device=DEV)
	W_out, b_out, beta = torch.zeros(H, O, device=DEV), torch.zeros(O, device=DEV), torch.ones(1, device=DEV)
	labels = torch.zeros(B, dtype=torch.int64, device=DEV)
	for surrogate, traces in ((_cabi.SNNK_SURROGATE_TRACE, False), (_cabi.SNNK_FAST_SIGMOID, True)):
		consts = F_.LayerConsts(1, surrogate, True, 0.9, 0.99, 0.1, 0.3, 0.9, tensor_core=True)
		desc = F_.make_desc(consts, B, T, Nx, H, O, traces, binary=True)
		ws_f = torch.empty(int(lib.snnk_forward_workspace_bytes(ctypes.byref(desc))), dtype=torch.uint8, device=DEV)
		ws_b = torch.empty(int(lib.snnk_backward_workspace_bytes(ctypes.byref(desc))), dtype=torch.uint8, device=DEV)
		out = {k: torch.full(s, -7.0, device=DEV) for k, s in (("V", (B, T, H)), ("a", (B, T, H)), ("Z", (B, T, H)),
			("y", (B, T, O)), ("logits", (B, O)), ("logp", (B, O)), ("loss", (1,)), ("g", (B, O)))}
		zbits = torch.zeros((B, T, H // 32), dtype=torch.int32, device=DEV)
		tstar = torch.zeros((B, O), dtype=torch.int32, device=DEV)
		rc = lib.snnk_forward_nll_sweep(ctypes.byref(desc), p(x), p(W_in), p(W_rec), None, p(beta), p(W_out), p(b_out), None,
			None, None, p(out["V"]), p(out["a"]), p(out["Z"]), p(zbits), p(out["y"]), p(out["logits"]), p(tstar), p(ws_f),
			ws_f.numel(), None, None, p(labels), p(out["logp"]), p(out["loss"]), p(out["g"]),
			p(torch.zeros(B + 1, dtype=torch.int32, device=DEV)), None, None, p(torch.ones(1, device=DEV)), p(ws_b),
			ws_b.numel(), _cabi.stream_ptr())
		assert rc == _cabi.SNNK_ERR_UNSUPPORTED
		torch.cuda.synchronize()
		for k, t in out.items():
			assert bool((t == -7.0).all()), f"{k} was written"
