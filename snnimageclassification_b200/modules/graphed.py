"""CUDA-graph capture of one training step (reference snn.py:384-415: forward, loss, backward, [all-reduce],
optimizer step).

At the reference's batch size the B200 kernels of a step run for a few hundred microseconds in total, less than
the Python/launch overhead of issuing them one by one, so ``SNN._exec_batch`` captures the whole step once per
input geometry and replays it: the host then does two small copies into static buffers and one graph launch.
"""
from __future__ import annotations

import gc
import weakref
from typing import Optional

import numpy as np
import torch

from . import functional as F_
from .functional import _const_scalar


def _optimizer_is_capturable(optimizer) -> bool:
	groups = getattr(optimizer, "param_groups", None)
	return bool(groups) and all(g.get("capturable", False) for g in groups)


class GraphedTrainStep:
	"""``step(x, y) -> loss`` (0-d device tensor, overwritten by the next call) replaying a captured CUDA graph.

	``x``/``y`` may live on the host (pinned memory makes the copy asynchronous) or on the device; they are
	copied into static buffers.  The optimizer step is part of the graph when the optimizer is capturable
	(``torch.optim.Adam(..., capturable=True)``), otherwise it runs eagerly after the replay.
	"""

	def __init__(self, net, x_example: torch.Tensor, y_example: torch.Tensor, criterion, optimizer, warmup: int = 3,
			static_inputs: bool = False):
		# The network caches its graphed steps, so a strong reference back would be a cycle: a discarded network (and its
		# CUDA graphs) would then be freed by the cyclic collector at an arbitrary later moment -- possibly in the middle
		# of ANOTHER capture, which destroying a graph invalidates.  Weak reference + an explicit collection before capture.
		self._net = weakref.ref(net)
		self.optimizer, self.criterion = optimizer, criterion
		dev = net.device
		self.static_inputs = static_inputs
		if static_inputs:
			# the caller's device tensors ARE the graph inputs (data resident in HBM: nothing to copy per step)
			assert x_example.is_cuda and y_example.is_cuda
			self.x, self.y = x_example, y_example
		else:
			self.x = torch.empty(x_example.shape, dtype=x_example.dtype, device=dev)
			self.y = torch.empty(y_example.shape, dtype=y_example.dtype, device=dev)
			self.x.copy_(x_example, non_blocking=True)
			self.y.copy_(y_example, non_blocking=True)
			# Host batches are staged through two device buffers on a copy stream: with the loss mailbox the caller is
			# back with the next batch while this step's backward pass still runs, so its H2D copy overlaps that work;
			# the compute stream then only does a device-to-device copy into the graph's input buffers.
			self._copy_stream = torch.cuda.Stream(device=dev)
			self._xs = [torch.empty_like(self.x) for _ in range(2)]
			self._ys = [torch.empty_like(self.y) for _ in range(2)]
			self._staged = [torch.cuda.Event() for _ in range(2)]
			self._consumed = [torch.cuda.Event() for _ in range(2)]
			self._flip = 0
		# Image batches that the network's own GPU encoder turns into spike trains (``input_encoder``): the encoder of the
		# NEXT batch is replayed on the copy stream, behind that batch's H2D copy, while the compute stream still runs
		# the current step (whose recurrence kernels leave SMs idle) -- two sets of encoder outputs, two captured steps.
		self._pre = (not static_inputs and getattr(net, "input_encoder", None) is not None and x_example.ndim == 2
			and not x_example.is_cuda)
		self.step_in_graph = _optimizer_is_capturable(optimizer)
		self.loss: Optional[torch.Tensor] = None
		# Loss mailbox: the fused head posts {launch number, loss} into this pinned host word, so the host reads the
		# loss of a replay by polling for its launch number -- it does not wait for the backward pass and can enqueue
		# the next batch meanwhile (``wait_loss``).  Only the fused-head path (plain NLLLoss) posts.
		self._mail = torch.zeros(1, dtype=torch.int64).pin_memory()
		self._mail_np = self._mail.numpy().view(np.uint64)
		self._mail_counter = torch.zeros(1, dtype=torch.int32, device=dev)
		self._expected = 0
		self._posts = False
		self._warmup = warmup
		self._capture()

	def _hyper_signature(self):
		sig = getattr(self.optimizer, "hyper_signature", None)
		return sig() if (callable(sig) and self.step_in_graph) else None

	def _capture(self):
		"""Warm-up + capture.  Runs at construction and again whenever the optimizer's by-value hyper-parameters (lr,
		betas, eps, weight decay -- kernel scalar arguments frozen into the graph) or its state tensors have changed."""
		net, optimizer, warmup = self.net, self.optimizer, self._warmup
		dev = net.device
		self._sig = self._hyper_signature()
		# Snapshot what the warm-up iterations would change: capture must not advance the training state.
		params = [p for p in net.parameters()]
		saved_params = [p.detach().clone() for p in params]
		saved_opt = _clone_state(optimizer.state_dict()) if self.step_in_graph else None

		side = torch.cuda.Stream(device=dev)
		side.wait_stream(torch.cuda.current_stream(dev))
		F_.LOSS_MAILBOX = (self._mail, self._mail_counter)
		try:
			if self._pre:
				for k in range(2):
					self._xs[k].copy_(self.x)
					self._ys[k].copy_(self.y)
				side.wait_stream(torch.cuda.current_stream(dev))
			with torch.cuda.stream(side):
				for _ in range(warmup):
					if self._pre:
						self._body(net._encode_if_needed(self._xs[0]), self._ys[0])
					else:
						self._body()
			torch.cuda.current_stream(dev).wait_stream(side)
			torch.cuda.synchronize(dev)
			self._expected = int(self._mail_counter.item())       # launches so far (warm-up); 0 if the head never posted
			self._posts = self._expected > 0

			if self._pre:
				self._enc_graphs, self._step_graphs, self._losses, self._grads = [], [], [], []
				for k in range(2):
					optimizer.zero_grad(set_to_none=True)
					gc.collect()
					ge = torch.cuda.CUDAGraph()
					with torch.cuda.graph(ge):
						xr = net._encode_if_needed(self._xs[k])
					gs = torch.cuda.CUDAGraph()
					with torch.cuda.graph(gs):
						loss = self._body(xr, self._ys[k])
					self._enc_graphs.append(ge)
					self._step_graphs.append(gs)
					self._losses.append(loss)
					self._grads.append([p.grad for p in params])
				self._rasters = xr      # keep-alive is the graph's pool; the attribute only documents the hand-over
				self.graph, self.loss = self._step_graphs[0], self._losses[0]
			else:
				optimizer.zero_grad(set_to_none=True)
				gc.collect()
				self.graph = torch.cuda.CUDAGraph()
				with torch.cuda.graph(self.graph):
					self.loss = self._body()
		finally:
			F_.LOSS_MAILBOX = None
		with torch.no_grad():
			for p, s in zip(params, saved_params):
				p.copy_(s)
		if saved_opt is not None:
			_restore_state(optimizer, saved_opt)

	@property
	def net(self):
		net = self._net()
		if net is None:
			raise RuntimeError("the network of this graphed training step no longer exists")
		return net

	def _body(self, x=None, y=None) -> torch.Tensor:
		net = self.net
		x = self.x if x is None else x
		root = _const_scalar(1.0, x.device)      # cached root gradient: no ones_like fill per step
		# published while the body runs: the fused training path of the loss runs the BPTT sweep for this gradient in its
		# forward kernel, and its backward uses that sweep when it receives this tensor
		F_.SWEEP_SCALE = root
		try:
			loss = net.batch_loss(x, self.y if y is None else y, self.criterion)
			self.optimizer.zero_grad(set_to_none=True)
			loss.backward(gradient=root)
		finally:
			F_.SWEEP_SCALE = None
		net._allreduce_gradients(self.optimizer)
		if self.step_in_graph:
			self.optimizer.step()
		return loss

	def _call_pre(self, x: torch.Tensor, y: torch.Tensor) -> torch.Tensor:
		"""Encoder of this batch on the copy stream (overlapping the previous step), then the step on the compute stream."""
		if self.step_in_graph and self._sig is not None and self._hyper_signature() != self._sig:
			torch.cuda.synchronize(self.x.device)
			self._capture()
		k = self._flip
		self._flip ^= 1
		main = torch.cuda.current_stream(self.x.device)
		cs = self._copy_stream if not (x.is_cuda or y.is_cuda) else main
		if cs is not main:
			cs.wait_event(self._consumed[k])          # the step that read this set of encoder outputs (two calls ago) is done
		with torch.cuda.stream(cs):
			self._xs[k].copy_(x, non_blocking=True)
			self._ys[k].copy_(y, non_blocking=True)
			self._enc_graphs[k].replay()
			if cs is not main:
				self._staged[k].record(cs)
		if cs is not main:
			main.wait_event(self._staged[k])
		self._step_graphs[k].replay()
		self._consumed[k].record(main)
		self._expected = (self._expected + 1) & 0xFFFFFFFF
		self.loss = self._losses[k]
		for p, g in zip(self.net.parameters(), self._grads[k]):
			p.grad = g
		if not self.step_in_graph:
			self.optimizer.step()
		return self.loss

	def __call__(self, x: Optional[torch.Tensor] = None, y: Optional[torch.Tensor] = None) -> torch.Tensor:
		if self._pre:
			return self._call_pre(x, y)
		if not self.static_inputs:
			if x.is_cuda or y.is_cuda:     # device inputs are ordered on the compute stream: copy there
				self.x.copy_(x, non_blocking=True)
				self.y.copy_(y, non_blocking=True)
			else:
				k = self._flip
				self._flip ^= 1
				main = torch.cuda.current_stream(self.x.device)
				cs = self._copy_stream
				cs.wait_event(self._consumed[k])          # the compute stream has taken what was staged here two calls ago
				with torch.cuda.stream(cs):
					self._xs[k].copy_(x, non_blocking=True)
					self._ys[k].copy_(y, non_blocking=True)
					self._staged[k].record(cs)
				main.wait_event(self._staged[k])
				self.x.copy_(self._xs[k], non_blocking=True)
				self.y.copy_(self._ys[k], non_blocking=True)
				self._consumed[k].record(main)
		if self.step_in_graph and self._sig is not None and self._hyper_signature() != self._sig:
			torch.cuda.current_stream(self.x.device).synchronize()
			self._capture()       # e.g. an LR scheduler stepped: the captured launch still carries the old scalars
		self.graph.replay()
		self._expected = (self._expected + 1) & 0xFFFFFFFF
		if not self.step_in_graph:
			self.optimizer.step()
		return self.loss

	def wait_loss(self) -> float:
		"""Python float of the latest replay's loss.  With the mailbox: polls the pinned host word for this replay's
		launch number (the rest of the step may still be running); otherwise synchronises and reads the device scalar."""
		if self._posts:
			target, word = self._expected, self._mail_np
			for _ in range(5_000_000):
				w = int(word[0])
				if (w >> 32) == target:
					return float(np.uint32(w & 0xFFFFFFFF).view(np.float32))
		return float(self.loss.item())


def _clone_state(sd):
	out = {"param_groups": [dict(g) for g in sd["param_groups"]], "state": {}}
	for k, st in sd["state"].items():
		out["state"][k] = {n: (v.detach().clone() if torch.is_tensor(v) else v) for n, v in st.items()}
	return out


def _restore_state(optimizer, saved):
	"""In-place restore: the graph holds pointers to the optimizer's state tensors, so they must not be replaced."""
	cur = optimizer.state_dict()["state"]
	with torch.no_grad():
		for k, st in cur.items():
			for n, v in st.items():
				if torch.is_tensor(v):
					if k in saved["state"] and n in saved["state"][k]:
						v.copy_(saved["state"][k][n])
					else:
						v.zero_()
