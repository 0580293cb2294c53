"""Autograd glue between the PyTorch-facing modules and the C ABI (include/snnk.h).

Two ``torch.autograd.Function``s wrap one hidden spiking layer + leaky readout over all T steps:

* ``SpikingSequence``      -- returns the output trace and the hidden traces, differentiable w.r.t. the weights;
  any PyTorch head / criterion can follow (the generic path of ``SNN.forward``, reference snn.py:201-219).
* ``SpikingSequenceNLL``   -- the fused training path of ``SNN._exec_batch`` (reference snn.py:384-415 with the
  default ``nn.NLLLoss``): max-over-time, log_softmax and the loss are evaluated by the library and the backward
  receives its seeds in sparse form.

PyTorch is plumbing here (device memory, streams, autograd bookkeeping); every FLOP of the path is issued by
libsnnk.so.  Nothing in this file has a CPU or eager fallback.
"""
from __future__ import annotations

import ctypes
import types
from dataclasses import dataclass
from typing import Optional, Tuple

import torch

from .. import _cabi


@dataclass(frozen=True)
class LayerConsts:
	"""Scalar constants of the hidden layer + readout (python floats, rounded to fp32 by the ABI struct)."""
	layer_type: int      # _cabi.SNNK_LIF | SNNK_ALIF | SNNK_IZHIKEVICH
	surrogate: int       # _cabi.SNNK_FAST_SIGMOID | SNNK_PHI | SNNK_SURROGATE_TRACE (spike_funcs.fused_surrogate)
	recurrent: bool
	alpha: float
	rho: float
	theta: float
	gamma: float
	kappa: float
	tensor_core: bool = False
	izh: Optional[Tuple[float, ...]] = None    # Izhikevich only: (dt, C, v_rest, v_th, k, a, b, c, d, v_peak)
	spike_func: Optional[type] = None          # the SpikeFunction class; its backward gives sigma' for SNNK_SURROGATE_TRACE


BINARY_TAG = "_snnk_binary"   # python attribute on tensors known to hold exactly {0,1} (encoder output, spike traces)


RUNS_TAG = "_snnk_runs"       # python attribute: the int32 run table of an encoded batch (include/snnk.h, snnk_encode_runs)


BITS_TAG = "_snnk_bits"       # python attribute on a BIT-PACKED raster (B, T, ceil(N/32)) int32: its feature count N


def mark_bits(t: torch.Tensor, n_pix: int) -> torch.Tensor:
	"""Tags an int32 tensor as the packed raster of ``n_pix`` features (SNNK_F_INPUT_BITS, include/snnk.h): the
	projection and weight-gradient kernels then expand the words in shared memory instead of reading fp32 rows."""
	if t.dtype != torch.int32 or t.ndim != 3 or t.shape[-1] != (n_pix + 31) // 32:
		raise ValueError("a packed raster is an int32 tensor (B, T, ceil(n_pix / 32))")
	setattr(t, BITS_TAG, int(n_pix))
	return t


def bits_width(t) -> Optional[int]:
	"""Feature count of a packed raster, None for anything else."""
	n = getattr(t, BITS_TAG, None)
	if n is None or t.dtype != torch.int32 or t.ndim != 3 or t.shape[-1] != (n + 31) // 32:
		return None
	return n


def bits_eligible(n_pix: int, tensor_core: bool) -> bool:
	"""Whether snnk_forward / snnk_backward take a packed raster of this width directly (else: unpack first)."""
	return bool(tensor_core) and n_pix % 4 == 0


def mark_binary(t: torch.Tensor, runs: Optional[torch.Tensor] = None) -> torch.Tensor:
	setattr(t, BINARY_TAG, True)
	if runs is not None:
		setattr(t, RUNS_TAG, runs)
	return t


def is_binary(t) -> bool:
	return bool(getattr(t, BINARY_TAG, False))


def get_runs(t) -> Optional[torch.Tensor]:
	"""The frame-run table riding on an encoder output, if it still describes ``t`` (same rows, same device)."""
	runs = getattr(t, RUNS_TAG, None)
	if runs is None or not is_binary(t) or t.ndim != 3:
		return None
	need = _cabi.lib().snnk_run_table_bytes(t.shape[0], t.shape[1]) // 4
	if runs.dtype != torch.int32 or runs.device != t.device or need == 0:
		return None
	if runs.numel() != need and not runs_tiled(t):
		return None
	return runs


def runs_tiled(t) -> bool:
	"""Whether the run table riding on ``t`` is followed by the tiled compact rows (snnk_run_table_tiled_bytes)."""
	runs = getattr(t, RUNS_TAG, None)
	if runs is None or t.ndim != 3 or t.dtype != torch.float32:
		return False
	need = _cabi.lib().snnk_run_table_tiled_bytes(t.shape[0], t.shape[1], t.shape[2]) // 4
	return need != 0 and runs.numel() == need


def make_desc(c: LayerConsts, B: int, T: int, N: int, H: int, O: int, traces: bool, binary: bool = False,
		bits: bool = False, tiled: bool = False) -> _cabi.SnnkDesc:
	flags = (_cabi.SNNK_F_TRACES if traces else 0) | (_cabi.SNNK_F_TENSOR_CORE if c.tensor_core else 0) | (
		_cabi.SNNK_F_INPUT_BINARY if (binary or bits) else 0) | (_cabi.SNNK_F_INPUT_BITS if bits else 0) | (
		_cabi.SNNK_F_RUNS_TILED if tiled else 0)
	izh = tuple(c.izh) if c.izh is not None else (0.0,) * 10
	return _cabi.SnnkDesc(
		B, T, N, H, O, c.layer_type, c.surrogate, int(c.recurrent), c.alpha, c.rho, c.theta, c.gamma, c.kappa, flags,
		*izh)


def padded_width(H: int) -> int:
	"""Hidden widths the kernels are instantiated for: 32, 64, 128 (register-resident recurrent weights) and the
	multiples of 128 up to 2048 (wide path).  Any other width (the reference's sweeps use 100 and 200,
	training.py:37) is zero-padded to the next one: padded neurons have no incoming, recurrent or outgoing weights,
	so they change nothing for the real ones and their traces / gradients are sliced away."""
	for h in (32, 64, 128):
		if H <= h:
			return h
	hp = (H + 127) // 128 * 128
	if hp > 2048:
		raise NotImplementedError(f"hidden width {H} > 2048 is not supported by the B200 path")
	return hp


def _pad_hidden(H: int, Hp: int, W_in, W_rec, rec_mask, W_out):
	if Hp == H:
		return W_in, W_rec, rec_mask, W_out
	pad = Hp - H
	P = torch.nn.functional.pad
	return (P(W_in, (0, pad)), None if W_rec is None else P(W_rec, (0, pad, 0, pad)),
		None if rec_mask is None else P(rec_mask, (0, pad, 0, pad)), P(W_out, (0, 0, 0, pad)))


_CONST = {}


def _const_scalar(value: float, device) -> torch.Tensor:
	"""A cached 0-d fp32 constant per device: placeholders and the root gradient of ``loss.backward()`` would otherwise
	each cost a fill kernel in every training step."""
	key = (float(value), str(device))
	t = _CONST.get(key)
	if t is None:
		t = _CONST[key] = torch.full((), float(value), dtype=torch.float32, device=device)
	return t


def _workspace(nbytes: int, device) -> torch.Tensor:
	return torch.empty(max(int(nbytes), 16), dtype=torch.uint8, device=device)


def _c(t: Optional[torch.Tensor]) -> Optional[torch.Tensor]:
	if t is None:
		return None
	r = t.detach()
	if bits_width(t) is not None:      # packed raster: stays int32 words
		return mark_bits(r if r.is_contiguous() else r.contiguous(), bits_width(t))
	if r.dtype != torch.float32:
		r = r.float()
	r = r if r.is_contiguous() else r.contiguous()
	if is_binary(t):
		mark_binary(r, getattr(t, RUNS_TAG, None))
	return r


_HEAD_WS = {}     # (device, B) -> zeroed scratch of snnk_forward_nll (per-row NLL terms + ticket word)


def _head_scratch(dev, B: int) -> torch.Tensor:
	"""One scratch per device and batch size, allocated (zeroed) on first use and kept: launches that use it are
	expected to be ordered, as the steps of one training loop are (include/snnk.h, snnk_forward_nll)."""
	key = (dev.index, B)
	ws = _HEAD_WS.get(key)
	if ws is None:
		ws = _HEAD_WS[key] = torch.zeros(B + 1, dtype=torch.int32, device=dev)
	return ws


def run_forward(
		c: LayerConsts, x, W_in, W_rec, rec_mask, beta, W_out, b_out, traces: bool = True,
		state: Optional[Tuple[Optional[torch.Tensor], ...]] = None, labels: Optional[torch.Tensor] = None,
		want_head_grad: bool = True, sweep_scale: Optional[torch.Tensor] = None,
):
	"""Calls ``snnk_forward`` -- or, with ``labels``, ``snnk_forward_nll`` (forward + fused log_softmax / NLL head).
	Returns dict(y, V, a, Z, zbits, logits, tstar, I_in, desc[, loss, logp, g_logits]).

	With ``sweep_scale`` (labels given, no traces): ``snnk_forward_nll_sweep``, which also runs the BPTT sweep for the
	loss gradient ``sweep_scale`` and leaves its results in the returned ``sweep_ws`` (for ``run_backward``); V and a
	are not produced.  Returns None when the library has no such kernel for this layer."""
	lib = _cabi.lib()
	_cabi.require_b200(x.device)
	B, T, N = x.shape
	nbits = bits_width(x)
	if nbits is not None:
		N = nbits
	H, O = W_out.shape
	if W_in.shape != (N, H):
		raise RuntimeError(f"forward_weights has shape {tuple(W_in.shape)}, expected {(N, H)}")
	runs = get_runs(x) if nbits is None else None
	desc = make_desc(c, B, T, N, H, O, traces, binary=is_binary(x), bits=nbits is not None,
		tiled=runs is not None and runs_tiled(x))
	dev = x.device
	f32 = dict(dtype=torch.float32, device=dev)
	alif = c.layer_type != _cabi.SNNK_LIF     # three-state layers: ALIF (V, a, Z) and Izhikevich (V, u, Z)
	sweep = sweep_scale is not None
	V = torch.empty((B, T, H), **f32) if traces else None
	Z = torch.empty((B, T, H), **f32) if (traces or sweep) else None
	a = torch.empty((B, T, H), **f32) if (traces and alif) else None
	zbits = torch.empty((B, T, H // 32), dtype=torch.int32, device=dev)
	y = torch.empty((B, T, O), **f32)
	logits = torch.empty((B, O), **f32)
	tstar = torch.empty((B, O), dtype=torch.int32, device=dev)
	ws = _workspace(lib.snnk_forward_workspace_bytes(ctypes.byref(desc)), dev)
	# the transposed masked recurrent matrix the backward sweep needs is prepared here, off the critical path
	W_effT = torch.empty((H, H), **f32) if (traces and W_rec is not None) else None
	V0 = a0 = Z0 = None
	if state is not None:
		if alif:
			V0, a0, Z0 = (_c(s) for s in state)
		else:
			V0, Z0 = (_c(s) for s in state)
	common = (
		ctypes.byref(desc), _cabi.ptr(x), _cabi.ptr(W_in), _cabi.ptr(W_rec), _cabi.ptr(rec_mask),
		_cabi.ptr(beta), _cabi.ptr(W_out), _cabi.ptr(b_out), _cabi.ptr(V0), _cabi.ptr(a0), _cabi.ptr(Z0),
		_cabi.ptr(V), _cabi.ptr(a), _cabi.ptr(Z), _cabi.ptr(zbits), _cabi.ptr(y), _cabi.ptr(logits),
		_cabi.ptr(tstar), _cabi.ptr(ws), ws.numel(), _cabi.ptr(runs), _cabi.ptr(W_effT))
	head = {}
	with torch.cuda.device(dev):
		if labels is None:
			rc = lib.snnk_forward(*common, _cabi.stream_ptr())
		else:
			labels = labels.to(device=dev, dtype=torch.int64).contiguous()
			logp = torch.empty((B, O), **f32)
			loss = torch.empty((), **f32)
			g = torch.empty((B, O), **f32) if want_head_grad else None
			box = LOSS_MAILBOX if (LOSS_MAILBOX is not None and LOSS_MAILBOX[1].device == dev) else None
			head_args = (_cabi.ptr(labels), _cabi.ptr(logp), _cabi.ptr(loss), _cabi.ptr(g), _cabi.ptr(_head_scratch(dev, B)),
				ctypes.c_void_p(box[0].data_ptr()) if box else None, _cabi.ptr(box[1]) if box else None)
			if sweep:
				sweep_ws = _workspace(lib.snnk_backward_workspace_bytes(ctypes.byref(desc)), dev)
				rc = lib.snnk_forward_nll_sweep(*common, *head_args, _cabi.ptr(sweep_scale), _cabi.ptr(sweep_ws),
					sweep_ws.numel(), _cabi.stream_ptr())
				if rc == _cabi.SNNK_ERR_UNSUPPORTED:
					return None
				head["sweep_ws"] = sweep_ws
			else:
				rc = lib.snnk_forward_nll(*common, *head_args, _cabi.stream_ptr())
			head.update(loss=loss, logp=logp, g_logits=g)
	_cabi.check(rc, "snnk_forward" if labels is None else "snnk_forward_nll_sweep" if sweep else "snnk_forward_nll")
	I_in = ws[: B * T * H * 4].view(torch.float32).view(B, T, H)
	return dict(y=y, V=V, a=a, Z=Z, zbits=zbits, logits=logits, tstar=tstar, I_in=I_in, desc=desc, Z0=Z0, W_effT=W_effT,
		**head)


def run_backward(
		c: LayerConsts, x, W_rec, rec_mask, beta, W_out, V, a, zbits, g_y=None, g_logits=None, tstar=None,
		g_V=None, g_Z=None, Z0=None, Z=None, g_scale=None, binary_input: bool = False, runs=None, W_effT=None,
		sweep_ws=None,
):
	"""Calls ``snnk_backward``.  Returns dict(dW_in, dW_rec, dW_out, db, gI) -- ``gI`` is a zero-argument callable
	(the tensor-core mode stores it as two planes; summing them is only worth it when somebody asks).  For a
	user-defined surrogate the ``a`` argument of the call is sigma' (surrogate_trace) instead of the saved ``a``.
	``sweep_ws``: the workspace in which ``run_forward(sweep_scale=...)`` already ran the sweep (SNNK_F_SWEEP_DONE)."""
	lib = _cabi.lib()
	if c.surrogate == _cabi.SNNK_SURROGATE_TRACE:
		a = surrogate_trace(c, V, a, beta)
	B, T, N = x.shape
	nbits = bits_width(x)
	if nbits is not None:
		N, runs = nbits, None
	H, O = W_out.shape
	desc = make_desc(c, B, T, N, H, O, True, binary=binary_input or is_binary(x), bits=nbits is not None)
	dev = x.device
	f32 = dict(dtype=torch.float32, device=dev)
	dW_in = torch.empty((N, H), **f32)
	dW_rec = torch.empty((H, H), **f32) if c.recurrent else None
	dW_out = torch.empty((H, O), **f32)
	db = torch.empty((O,), **f32)
	if sweep_ws is not None:
		desc.flags |= _cabi.SNNK_F_SWEEP_DONE
		ws = sweep_ws
	else:
		ws = _workspace(lib.snnk_backward_workspace_bytes(ctypes.byref(desc)), dev)
	with torch.cuda.device(dev):
		rc = lib.snnk_backward(
			ctypes.byref(desc), _cabi.ptr(x), _cabi.ptr(W_rec), _cabi.ptr(rec_mask), _cabi.ptr(beta),
			_cabi.ptr(W_out), _cabi.ptr(Z0), _cabi.ptr(V), _cabi.ptr(a), _cabi.ptr(Z), _cabi.ptr(zbits), _cabi.ptr(g_y),
			_cabi.ptr(g_logits), _cabi.ptr(tstar), _cabi.ptr(g_scale), _cabi.ptr(g_V), _cabi.ptr(g_Z), _cabi.ptr(dW_in),
			_cabi.ptr(dW_rec), _cabi.ptr(dW_out), _cabi.ptr(db), _cabi.ptr(ws), ws.numel(),
			_cabi.ptr(runs if (runs is not None or nbits is not None) else get_runs(x)), _cabi.ptr(W_effT), _cabi.stream_ptr())
	_cabi.check(rc, "snnk_backward")
	n = B * T * H * 4
	planes = c.tensor_core and N % 4 == 0   # stored as two tf32 planes (high, exact remainder); see include/snnk.h

	def gI():
		hi = ws[:n].view(torch.float32).view(B, T, H)
		if not planes:
			return hi
		off = (n + 255) // 256 * 256
		return hi + ws[off: off + n].view(torch.float32).view(B, T, H)
	return dict(dW_in=dW_in, dW_rec=dW_rec, dW_out=dW_out, db=db, gI=gI)


def run_input_grad(c: LayerConsts, gI: torch.Tensor, W_in: torch.Tensor) -> torch.Tensor:
	"""Calls ``snnk_input_grad``: gX (B,T,N) = gI (B,T,H) @ W_in^T  (W_in is (N,H))."""
	lib = _cabi.lib()
	B, T, H = gI.shape
	N = W_in.shape[0]
	desc = make_desc(c, B, T, N, H, 1, True)
	gX = torch.empty((B, T, N), dtype=torch.float32, device=gI.device)
	gI = gI.contiguous()
	with torch.cuda.device(gI.device):
		rc = lib.snnk_input_grad(ctypes.byref(desc), _cabi.ptr(gI), _cabi.ptr(W_in), _cabi.ptr(gX), _cabi.stream_ptr())
	_cabi.check(rc, "snnk_input_grad")
	return gX


# (pinned host int64 word, device int32 counter) while a graphed training step is being built: the head kernel then
# also posts the loss to the host word (include/snnk.h, snnk_head_nll); see modules/graphed.py
LOSS_MAILBOX = None

# The root gradient (a 0-d device tensor) of the backward call that follows while a graphed training step runs its body
# (modules/graphed.py): SpikingSequenceNLL then runs the BPTT sweep for that gradient in its forward
# (snnk_forward_nll_sweep), and its backward keeps the result if it receives that very tensor.
SWEEP_SCALE = None


def run_head_nll(logits: torch.Tensor, labels: torch.Tensor, want_grad: bool = True):
	"""Calls ``snnk_head_nll``.  Returns (loss (), logp (B,O), g_logits (B,O) | None)."""
	lib = _cabi.lib()
	B, O = logits.shape
	dev = logits.device
	labels = labels.to(device=dev, dtype=torch.int64).contiguous()
	logp = torch.empty_like(logits)
	loss = torch.empty((), dtype=torch.float32, device=dev)
	g = torch.empty_like(logits) if want_grad else None
	box = LOSS_MAILBOX if (LOSS_MAILBOX is not None and LOSS_MAILBOX[1].device == dev) else None
	with torch.cuda.device(dev):
		rc = lib.snnk_head_nll(
			B, O, _cabi.ptr(logits), _cabi.ptr(labels), _cabi.ptr(logp), _cabi.ptr(loss), _cabi.ptr(g),
			ctypes.c_void_p(box[0].data_ptr()) if box else None, _cabi.ptr(box[1]) if box else None,
			_cabi.stream_ptr())
	_cabi.check(rc, "snnk_head_nll")
	return loss, logp, g


def surrogate_trace(c: LayerConsts, V: torch.Tensor, a: Optional[torch.Tensor], beta: Optional[torch.Tensor]):
	"""sigma'_t = dZ_t/dV_t (B,T,H) of the user-defined surrogate ``c.spike_func`` over the saved traces, for the
	``a`` argument of ``snnk_backward`` with SNNK_SURROGATE_TRACE: its ``backward`` is called once on a stand-in ctx
	holding (V, threshold, gamma), as SpikeFunction.forward saves them, with an all-ones gradient.  The threshold is
	theta (LIF), theta + beta a_t rounded twice as the kernels do (ALIF) or v_peak (Izhikevich, ``c.theta``).  Nothing
	here waits for the device, so a captured training step records the user's operations too."""
	dev = V.device
	thr = _const_scalar(c.theta, dev)
	if c.layer_type == _cabi.SNNK_ALIF:
		thr = thr + beta * a
	ctx = types.SimpleNamespace(saved_tensors=(V, thr, _const_scalar(c.gamma, dev).reshape(1)))
	out = c.spike_func.backward(ctx, _const_scalar(1.0, dev).expand(V.shape))
	sg = out[0] if isinstance(out, (tuple, list)) else out
	if not isinstance(sg, torch.Tensor) or sg.shape != V.shape or sg.dtype != torch.float32 or sg.device != dev:
		got = f"{tuple(sg.shape)} {sg.dtype} on {sg.device}" if isinstance(sg, torch.Tensor) else type(sg).__name__
		raise TypeError(f"{c.spike_func.__name__}.backward must return a float32 tensor of the input's shape "
			f"{tuple(V.shape)} on {dev} as its first element, got {got}")
	return sg.detach().contiguous()


class SpikingSequence(torch.autograd.Function):
	"""(x, weights) -> (y, V, a, Z): generic differentiable forward over all T steps."""

	@staticmethod
	def forward(ctx, consts: LayerConsts, x, W_in, W_rec, rec_mask, beta, W_out, b_out):
		xc, Wi, Wr, M, be, Wo, bo = (_c(t) for t in (x, W_in, W_rec, rec_mask, beta, W_out, b_out))
		H = Wo.shape[0]
		Hp = padded_width(H)
		Wi, Wr, M, Wo = _pad_hidden(H, Hp, Wi, Wr, M, Wo)
		out = run_forward(consts, xc, Wi, Wr, M, be, Wo, bo, traces=True)
		ctx.consts, ctx.H, ctx.Hp = consts, H, Hp
		ctx.set_materialize_grads(False)                     # absent seeds stay None instead of (B,T,H) zero fills
		ctx.binary, ctx.runs, ctx.W_effT = is_binary(xc), get_runs(xc), out["W_effT"]
		ctx.Wi = Wi if ctx.needs_input_grad[1] else None      # stacked layers: the input is the spike trace below
		ctx.save_for_backward(xc, Wr, M, be, Wo, out["V"], out["a"], out["zbits"], out["Z"])
		alif = consts.layer_type != _cabi.SNNK_LIF
		a = out["a"][..., :H] if alif else _const_scalar(0.0, out["V"].device)
		ctx.mark_non_differentiable(a)
		return out["y"], out["V"][..., :H], a, out["Z"][..., :H]

	@staticmethod
	def backward(ctx, g_y, g_V, g_a, g_Z):
		xc, Wr, M, be, Wo, V, a, zbits, Z = ctx.saved_tensors
		if g_y is None:
			g_y = torch.zeros((V.shape[0], V.shape[1], Wo.shape[1]), dtype=torch.float32, device=V.device)
		H, Hp = ctx.H, ctx.Hp
		g_V, g_Z = _c(g_V), _c(g_Z)
		if Hp != H:
			g_V = None if g_V is None else torch.nn.functional.pad(g_V, (0, Hp - H))
			g_Z = None if g_Z is None else torch.nn.functional.pad(g_Z, (0, Hp - H))
		g = run_backward(ctx.consts, xc, Wr, M, be, Wo, V, a, zbits, g_y=_c(g_y), g_V=g_V, g_Z=g_Z, Z=Z,
			binary_input=ctx.binary, runs=ctx.runs, W_effT=ctx.W_effT)
		# (consts, x, W_in, W_rec, rec_mask, beta, W_out, b_out); beta gets no gradient -- the threshold input of
		# the reference's spike function returns None (spike_funcs.py:62/79)
		gX = run_input_grad(ctx.consts, g["gI"](), ctx.Wi) if ctx.Wi is not None else None
		return (None, gX, g["dW_in"][:, :H], None if g["dW_rec"] is None else g["dW_rec"][:H, :H], None, None,
			g["dW_out"][:H], g["db"])


class SpikingSequenceNLL(torch.autograd.Function):
	"""(x, labels, weights) -> (loss, logp, y, V, a, Z) with the head fused (snn.py:228, :258, :297)."""

	@staticmethod
	def forward(ctx, consts: LayerConsts, x, labels, W_in, W_rec, rec_mask, beta, W_out, b_out, traces: bool):
		xc, Wi, Wr, M, be, Wo, bo = (_c(t) for t in (x, W_in, W_rec, rec_mask, beta, W_out, b_out))
		H = Wo.shape[0]
		Hp = padded_width(H)
		Wi, Wr, M, Wo = _pad_hidden(H, Hp, Wi, Wr, M, Wo)
		need_grad = any(ctx.needs_input_grad)
		scale = SWEEP_SCALE
		out = None
		if need_grad and not traces and scale is not None and scale.device == xc.device:
			out = run_forward(consts, xc, Wi, Wr, M, be, Wo, bo, traces=False, labels=labels, sweep_scale=scale)
		# the sweep ran for `scale`; any other gradient recomputes the traces (same kernels, same values) in backward
		ctx.sweep = (scale, out["sweep_ws"], Wi, bo) if out is not None else None
		if out is None:
			out = run_forward(consts, xc, Wi, Wr, M, be, Wo, bo, traces=traces or need_grad, labels=labels,
				want_head_grad=need_grad)
		loss, logp, g_logits = out["loss"], out["logp"], out["g_logits"]
		ctx.consts, ctx.H = consts, H
		ctx.set_materialize_grads(False)
		ctx.binary, ctx.runs, ctx.W_effT = is_binary(xc), get_runs(xc), out["W_effT"]
		ctx.Wi = Wi if ctx.needs_input_grad[1] else None
		if need_grad:
			ctx.save_for_backward(xc, Wr, M, be, Wo, out["V"], out["a"], out["zbits"], g_logits, out["tstar"], out["Z"])
		empty = _const_scalar(0.0, logp.device)
		extras = tuple(
			(out[k] if k == "y" else out[k][..., :H]) if out[k] is not None else empty for k in ("y", "V", "a", "Z"))
		ctx.mark_non_differentiable(logp, *extras)
		return (loss, logp) + extras

	@staticmethod
	def backward(ctx, g_loss, *_):
		xc, Wr, M, be, Wo, V, a, zbits, g_logits, tstar, Z = ctx.saved_tensors
		if g_loss is None:
			return (None,) * 10
		sweep_ws, W_effT = None, ctx.W_effT
		if ctx.sweep is not None:
			scale, ws, Wi, bo = ctx.sweep
			if g_loss.dtype == torch.float32 and g_loss.data_ptr() == scale.data_ptr():
				sweep_ws = ws
			else:
				f = run_forward(ctx.consts, xc, Wi, Wr, M, be, Wo, bo, traces=True)
				V, a, zbits, Z, W_effT = f["V"], f["a"], f["zbits"], f["Z"], f["W_effT"]
		g = run_backward(
			ctx.consts, xc, Wr, M, be, Wo, V, a, zbits, g_logits=g_logits, tstar=tstar, Z=Z,
			g_scale=g_loss.detach().float().reshape(1), binary_input=ctx.binary, runs=ctx.runs, W_effT=W_effT,
			sweep_ws=sweep_ws)
		H = ctx.H
		gX = run_input_grad(ctx.consts, g["gI"](), ctx.Wi) if ctx.Wi is not None else None
		return (None, gX, None, g["dW_in"][:, :H], None if g["dW_rec"] is None else g["dW_rec"][:H, :H], None, None,
			g["dW_out"][:H], g["db"], None)
