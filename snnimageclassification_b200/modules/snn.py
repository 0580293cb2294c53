"""``SNN`` -- mirror of the reference's src/modules/snn.py with the hot path on B200 kernels.

Same constructor, parameter names, ``state_dict`` layout, return values of ``forward`` /
``get_prediction_*`` / ``fit`` and checkpoint files as the reference.  What changes underneath:

* ``forward`` (reference snn.py:201-219, a Python loop of T x layers small matmuls and elementwise ops) makes ONE
  call into libsnnk.so: projection GEMM for all T steps, persistent fused recurrence + readout kernel.
* ``_exec_batch`` (reference snn.py:384-415) with the default ``nn.NLLLoss`` uses the fused head and the fused
  reverse-time BPTT kernels; any other criterion goes through ordinary autograd on top of the same kernels.
* data-parallel training: when ``torch.distributed`` is initialised, ``_exec_batch`` all-reduces (averages) the
  gradients over the ranks before the optimizer step -- one flat NCCL call.

Extra constructor keywords (all optional, the reference ignores unknown kwargs the same way):
``input_encoder`` (a ``ToSpikes`` applied on the GPU to (B, F) image batches) and ``tensor_core``.
"""
from __future__ import annotations

import enum
import json
import logging
import os
import shutil
from typing import Any, Dict, Iterable, List, Optional, Tuple, Type, Union

import numpy as np
import torch
import torch.nn.functional as F
from torch import Tensor, nn
from torch.utils.data import DataLoader

from .. import _cabi
from . import functional as F_
from .spike_funcs import HeavisideSigmoidApprox, SpikeFuncType, SpikeFuncType2Func, SpikeFunction
from .spiking_layers import ALIFLayer, IzhikevichLayer, LayerType, LayerType2Layer, LIFLayer, ReadoutLayer
from .utils import LossHistory, mapping_update_recursively

try:  # progress bars are cosmetic
	from tqdm.auto import tqdm
except ImportError:  # pragma: no cover
	def tqdm(it=None, **kw):
		return it


class ReadoutMth(enum.Enum):
	RNN = 0


class ForwardMth(enum.Enum):
	LAYER_THEN_TIME = 0
	TIME_THEN_LAYER = 1


class LoadCheckpointMode(enum.Enum):
	BEST_EPOCH = enum.auto()
	LAST_EPOCH = enum.auto()


class SNN(torch.nn.Module):
	SAVE_EXT = ".pth"
	SUFFIX_SEP = "-"
	CHECKPOINTS_META_SUFFIX = "checkpoints"
	CHECKPOINT_SAVE_PATH_KEY = "save_path"
	CHECKPOINT_BEST_KEY = "best"
	CHECKPOINT_EPOCHS_KEY = "epochs"
	CHECKPOINT_EPOCH_KEY = "epoch"
	CHECKPOINT_LOSS_KEY = "loss"
	CHECKPOINT_OPTIMIZER_STATE_DICT_KEY = "optimizer_state_dict"
	CHECKPOINT_STATE_DICT_KEY = "model_state_dict"
	CHECKPOINT_FILE_STRUCT: Dict[str, Union[str, Dict[int, str]]] = {
		CHECKPOINT_BEST_KEY: CHECKPOINT_SAVE_PATH_KEY,
		CHECKPOINT_EPOCHS_KEY: {0: CHECKPOINT_SAVE_PATH_KEY},
	}
	load_mode_to_suffix = {mode: mode.name for mode in list(LoadCheckpointMode)}

	def __init__(
			self,
			inputs_size: int,
			output_size: int,
			n_hidden_neurons: Iterable[int] = None,
			use_recurrent_connection: Union[bool, Iterable[bool]] = True,
			dt=1e-3,
			int_time_steps=100,
			spike_func: Union[Type[SpikeFunction], SpikeFuncType] = HeavisideSigmoidApprox,
			hidden_layer_type: Union[Type[LIFLayer], LayerType] = LIFLayer,
			device=None,
			checkpoint_folder: str = "checkpoints",
			model_name: str = "snn",
			**kwargs
	):
		super().__init__()
		# the fused readout / head kernels hold the class dimension in 16 lanes: refuse a wider readout here rather
		# than at the first forward call
		if not 1 <= int(output_size) <= _cabi.SNNK_MAX_CLASSES:
			raise ValueError(f"output_size={output_size}: the B200 kernels support readouts of 1 to "
				f"{_cabi.SNNK_MAX_CLASSES} classes")
		self.input_size = inputs_size
		self.output_size = output_size
		# keywords of the B200 build; everything else is threaded to the layers exactly as in the reference
		self.input_encoder = kwargs.pop("input_encoder", None)
		# tcgen05 GEMMs by default (exact for spike inputs, automatic fp32 fallback otherwise); SNNK_TENSOR_CORE=0 or
		# tensor_core=False selects the fp32 CUDA-core GEMMs, which are bit-identical to the CPU oracle
		self.tensor_core = bool(kwargs.pop("tensor_core", os.environ.get("SNNK_TENSOR_CORE", "1") != "0"))
		# replay a captured CUDA graph for training steps whose input geometry repeats (see modules/graphed.py)
		self.cuda_graphs = bool(kwargs.pop("cuda_graphs", os.environ.get("SNNK_CUDA_GRAPHS", "1") != "0"))
		self._graphed_steps: Dict[Any, Any] = {}
		self._graph_seen: Dict[Any, int] = {}
		self.last_eval_accuracy = float("nan")     # accuracy counted by the latest eval-mode _exec_epoch
		self._last_graphed_step = None
		self.kwargs = kwargs

		# device, time grid and the two enum-or-class arguments (reference snn.py:68-84)
		if device is None:
			self.device = None
			self._set_default_device_()
			device = self.device
		self.device = torch.device(device)
		self.dt, self.int_time_steps = dt, int_time_steps
		self.spike_func = SpikeFuncType2Func[spike_func] if isinstance(spike_func, SpikeFuncType) else spike_func
		self.hidden_layer_type = (
			LayerType2Layer[hidden_layer_type] if isinstance(hidden_layer_type, LayerType) else hidden_layer_type)
		self.checkpoint_folder, self.model_name = checkpoint_folder, model_name
		# an int is one hidden layer, None is a readout-only model
		widths = [n_hidden_neurons] if isinstance(n_hidden_neurons, int) else n_hidden_neurons
		self.n_hidden_neurons = [] if widths is None else widths
		self.use_recurrent_connection = use_recurrent_connection
		self.layers = nn.ModuleDict()
		self._add_layers_()
		self.initialize_weights_()
		self.loss_history = LossHistory()
		self._consts_cache: Optional[F_.LayerConsts] = None

	# ---- construction (reference snn.py:96-157) -----------------------------------------------------------------
	@property
	def checkpoints_meta_path(self) -> str:
		return f"{self.checkpoint_folder}/{self.model_name}{SNN.SUFFIX_SEP}{SNN.CHECKPOINTS_META_SUFFIX}.json"

	def _set_default_device_(self):
		self.device = torch.device("cuda") if torch.cuda.is_available() else torch.device("cpu")

	def _spiking_layer(self, n_in: int, n_out: int):
		"""One hidden layer of the configured type; every extra keyword of the constructor is handed on, as the
		reference does (snn.py:103-128)."""
		return self.hidden_layer_type(
			input_size=n_in, output_size=n_out, use_recurrent_connection=self.use_recurrent_connection, dt=self.dt,
			spike_func=self.spike_func, device=self.device, **self.kwargs)

	def _add_input_layer_(self):
		if self.n_hidden_neurons:
			self.layers["input"] = self._spiking_layer(self.input_size, self.n_hidden_neurons[0])

	def _add_hidden_layers_(self):
		widths = list(self.n_hidden_neurons)
		for i, (n_in, n_out) in enumerate(zip(widths[:-1], widths[1:])):
			self.layers[f"hidden_{i}"] = self._spiking_layer(n_in, n_out)

	def _add_readout_layer(self):
		n_in = self.n_hidden_neurons[-1] if self.n_hidden_neurons else self.input_size
		self.layers["readout"] = ReadoutLayer(
			input_size=n_in, output_size=self.output_size, dt=self.dt, spike_func=self.spike_func, device=self.device,
			**self.kwargs)

	def _add_layers_(self):
		for add in (self._add_input_layer_, self._add_hidden_layers_, self._add_readout_layer):
			add()

	def initialize_weights_(self):
		# Same order as the reference (snn.py:149-157): every parameter is re-drawn ~N(0,1) -- including a learnable
		# beta -- and then each layer applies its own initialiser, so a given torch seed yields the same weights.
		for p in self.parameters():
			(torch.nn.init.xavier_normal_ if p.ndim > 2 else torch.nn.init.normal_)(p)
		for layer in self.layers.values():
			init = getattr(layer, "initialize_weights_", None)
			if callable(init):
				init()

	# ---- input formatting (reference snn.py:159-184) ------------------------------------------------------------
	def _format_inputs(self, inputs: torch.Tensor) -> torch.Tensor:
		"""(B, F) -> repeated over int_time_steps; (B, T' <= T, F) -> zero-padded to T; cast to float32."""
		if F_.bits_width(inputs) is not None:      # packed raster kept packed by _encode_if_needed: T already matches
			return inputs
		with torch.no_grad():
			if inputs.ndim == 2:
				inputs = torch.unsqueeze(inputs, 1).repeat(1, self.int_time_steps, 1)
			assert inputs.ndim == 3, \
				"shape of inputs must be (batch_size, time_steps, nb_features) or (batch_size, nb_features)"
			t_diff = self.int_time_steps - inputs.shape[1]
			assert t_diff >= 0, "inputs time steps must me less or equal to int_time_steps"
			if t_diff > 0:
				pad = torch.zeros((inputs.shape[0], t_diff, inputs.shape[-1]), dtype=torch.float32, device=inputs.device)
				inputs = torch.cat([inputs.float(), pad], dim=1)
		return inputs.float().contiguous()

	def _encode_if_needed(self, inputs: torch.Tensor) -> torch.Tensor:
		"""Image batches (B, F) are turned into spike trains on the GPU when an ``input_encoder`` was given; bit-packed
		rasters (int32, last dimension ceil(F/32): ``ToSpikes.encode_batch_bits``) are unpacked on the device."""
		if inputs.dtype == torch.int32 and inputs.ndim == 3 and inputs.shape[-1] == (self.input_size + 31) // 32 \
				and inputs.shape[-1] != self.input_size:
			inputs = inputs.to(self.device, non_blocking=True)
			# the tensor-core GEMMs expand the words inside their shared-memory tiles (SNNK_F_INPUT_BITS): the fp32
			# raster is never materialised.  Otherwise (fp32 mode, ragged width, fewer steps than int_time_steps,
			# SNNK_PACKED_GEMM=0) the words are unpacked on the device first.
			if (F_.bits_eligible(self.input_size, self.tensor_core) and inputs.shape[1] == self.int_time_steps
					and os.environ.get("SNNK_PACKED_GEMM", "1") != "0"):
				return F_.mark_bits(inputs.contiguous(), self.input_size)
			from ..datasets.datasets import unpack_raster
			return unpack_raster(inputs, self.input_size)
		if self.input_encoder is not None and inputs.ndim == 2:
			# the raster is an intermediate nobody but the first layer's kernels reads: with the frame-dedup variant
			# active those read only the first row of every run, so the rest need not be written (lazy raster)
			# (only where snnk_forward / snnk_backward take the variant: tensor-core GEMMs, first layer <= 128 wide,
			# TMA-addressable input width -- include/snnk.h; otherwise the dense kernels read every row)
			lazy = (self.tensor_core and self.input_encoder.n_steps == self.int_time_steps
				and bool(self.n_hidden_neurons) and F_.padded_width(int(self.n_hidden_neurons[0])) <= 128
				and inputs.shape[1] % 4 == 0 and os.environ.get("SNNK_LAZY_RASTER", "1") != "0")
			return self.input_encoder.encode_batch(inputs, lazy=lazy)
		return inputs

	# ---- the fused path -------------------------------------------------------------------------------------------
	def _hidden_chain(self) -> List[Tuple[str, LIFLayer]]:
		"""The spiking layers in execution order ("input", "hidden_0", ...; reference snn.py:103-128)."""
		if not self.n_hidden_neurons:
			raise NotImplementedError(
				"the B200 path needs at least one hidden spiking layer (n_hidden_neurons=None is a readout-only model, "
				"which no published configuration of the reference uses); there is no eager fallback")
		chain = [(name, layer) for name, layer in self.layers.items() if name != "readout"]
		for name, layer in chain:
			if not isinstance(layer, (LIFLayer, IzhikevichLayer)):
				raise NotImplementedError(
					f"{type(layer).__name__} is not supported by the B200 path (LIF, ALIF and Izhikevich are fused)")
		return chain

	def _hot_layers(self) -> Tuple[LIFLayer, ReadoutLayer]:
		"""(last hidden layer, readout): the pair the fused recurrence + readout kernel runs."""
		return self._hidden_chain()[-1][1], self.layers["readout"]

	def refresh_constants(self):
		"""Re-reads alpha/rho/theta/gamma/kappa from the layers (call after editing them by hand)."""
		self._consts_cache = None
		self._inner_cache = {}

	def _consts(self) -> F_.LayerConsts:
		if self._consts_cache is None:
			layer, readout = self._hot_layers()
			self._consts_cache = layer.snnk_consts(kappa=float(readout.kappa), tensor_core=self.tensor_core)
		return self._consts_cache

	@staticmethod
	def _layer_weights(layer: LIFLayer):
		beta = layer.beta.reshape(1) if isinstance(layer, ALIFLayer) else None
		return layer.forward_weights, layer.recurrent_weights, layer.rec_mask, beta

	def _weights(self):
		layer, readout = self._hot_layers()
		return (*self._layer_weights(layer), readout.forward_weights, readout.bias_weights)

	def _run_inner_layers(self, x: torch.Tensor, hidden: Optional[dict] = None) -> torch.Tensor:
		"""Stacked hidden layers (snn.py:116-128): every layer but the last runs the same fused kernels with a null
		readout; its spike trace is the input of the next layer.  (Time-then-layer, as the reference loops, and
		layer-then-time, as here, are the same computation: layer l at step t only sees layer l-1 at step t.)"""
		if not hasattr(self, "_inner_cache"):
			self._inner_cache = {}
		for name, layer in self._hidden_chain()[:-1]:
			if name not in self._inner_cache:
				H = layer.output_size
				self._inner_cache[name] = (
					layer.snnk_consts(kappa=0.0, tensor_core=self.tensor_core),
					torch.zeros((H, 1), dtype=torch.float32, device=self.device),
					torch.zeros((1,), dtype=torch.float32, device=self.device))
			consts, w0, b0 = self._inner_cache[name]
			_, V, a, Z = F_.SpikingSequence.apply(consts, x, *self._layer_weights(layer), w0, b0)
			if hidden is not None:
				hidden[name] = (V, a, Z) if isinstance(layer, (ALIFLayer, IzhikevichLayer)) else (V, Z)
			x = F_.mark_binary(Z)      # a spike trace is exactly {0,1}
		return x

	def forward(self, inputs):
		"""-> (outputs_trace (B,T,O), {"input": (V,[a],Z), ["hidden_i": ...], "readout": (y,)}), as snn.py:201-219."""
		layer, _ = self._hot_layers()
		inputs = self._format_inputs(self._encode_if_needed(inputs.to(self.device, non_blocking=True)))
		hidden_states = {}
		inputs = self._run_inner_layers(inputs, hidden_states)
		y, V, a, Z = F_.SpikingSequence.apply(self._consts(), inputs, *self._weights())
		hidden_states[self._hidden_chain()[-1][0]] = (V, a, Z) if isinstance(layer, (ALIFLayer, IzhikevichLayer)) else (V, Z)
		hidden_states["readout"] = (y,)
		return y, hidden_states

	def _infer_logits(self, inputs: torch.Tensor) -> torch.Tensor:
		"""Forward without materialising the last layer's traces; the max over time comes out of the kernel."""
		inputs = self._format_inputs(self._encode_if_needed(inputs))
		inputs = self._run_inner_layers(inputs)
		Wi, Wr, M, be, Wo, bo = (F_._c(w) for w in self._weights())
		H = Wo.shape[0]
		Wi, Wr, M, Wo = F_._pad_hidden(H, F_.padded_width(H), Wi, Wr, M, Wo)
		return F_.run_forward(self._consts(), F_._c(inputs), Wi, Wr, M, be, Wo, bo, traces=False)["logits"]

	# ---- prediction heads (reference snn.py:221-259) --------------------------------------------------------------
	def get_prediction_logits(self, inputs: torch.Tensor, re_outputs_trace: bool = True, re_hidden_states: bool = True):
		inputs = inputs.to(self.device)
		if not re_outputs_trace and not re_hidden_states and not torch.is_grad_enabled():
			return self._infer_logits(inputs)
		outputs_trace, hidden_states = self(inputs)
		logits, _ = torch.max(outputs_trace, dim=1)
		if re_outputs_trace and re_hidden_states:
			return logits, outputs_trace, hidden_states
		elif re_outputs_trace:
			return logits, outputs_trace
		elif re_hidden_states:
			return logits, hidden_states
		return logits

	def get_prediction_proba(self, inputs: torch.Tensor, re_outputs_trace: bool = True, re_hidden_states: bool = True):
		if re_outputs_trace or re_hidden_states:
			m, *outs = self.get_prediction_logits(inputs, re_outputs_trace, re_hidden_states)
			return (F.softmax(m, dim=-1), *outs)
		# the reference returns the raw logits in this branch (snn.py:246-248); kept
		return self.get_prediction_logits(inputs, re_outputs_trace, re_hidden_states)

	def get_prediction_log_proba(self, inputs: torch.Tensor, re_outputs_trace: bool = True, re_hidden_states: bool = True):
		if re_outputs_trace or re_hidden_states:
			m, *outs = self.get_prediction_logits(inputs, re_outputs_trace, re_hidden_states)
			return (F.log_softmax(m, dim=-1), *outs)
		return self.get_prediction_logits(inputs, re_outputs_trace, re_hidden_states)

	def get_spikes_count_per_neuron(self, hidden_states: Dict[str, List[torch.Tensor]]) -> torch.Tensor:
		counts = []
		for l_name, traces in hidden_states.items():
			if isinstance(self.layers[l_name], LIFLayer):
				counts.extend(traces[-1].sum(dim=(0, 1)).tolist())
		return torch.tensor(counts, dtype=torch.float32, device=self.device)

	def _check_early_stopping(self, patience: int, tol: float = 1e-2) -> bool:
		losses = self.loss_history["val"][-patience:]
		return bool(np.all(np.abs(np.diff(losses)) < tol))

	def _prepare_run(self, optimizer, load_checkpoint_mode, force_overwrite: bool, verbose: bool) -> int:
		"""First epoch to run.  Fresh run (no load mode): the reference's guard is kept as it is (snn.py:301-306 -- it
		insists on ``force_overwrite`` when there is NO checkpoint index yet, although its message says the opposite) and
		an existing checkpoint folder is removed.  Resume: weights, optimizer state and loss history come back from the
		chosen checkpoint; a missing one means starting from scratch."""
		meta = self.checkpoints_meta_path
		if load_checkpoint_mode is None:
			have_meta = os.path.exists(meta)
			assert have_meta or force_overwrite, (
				f"{meta} already exists. Set force_overwrite flag to True to overwrite existing saves.")
			if have_meta and force_overwrite and self._is_writer():
				shutil.rmtree(self.checkpoint_folder)
			self._dp_barrier()      # nobody runs ahead (and writes) while rank 0 is still removing the old folder
			return 0
		try:
			ck = self.load_checkpoint(load_checkpoint_mode)       # also loads the weights
		except FileNotFoundError:
			if verbose:
				logging.warning("No such checkpoint. Fit from beginning.")
			return 0
		optimizer.load_state_dict(ck[SNN.CHECKPOINT_OPTIMIZER_STATE_DICT_KEY])
		self.loss_history = self.get_checkpoints_loss_history()
		return int(ck[SNN.CHECKPOINT_EPOCH_KEY]) + 1

	# ---- training loop (reference snn.py:280-415) -----------------------------------------------------------------
	def fit(
			self,
			train_dataloader: DataLoader,
			val_dataloader: DataLoader,
			lr=1e-3,
			nb_epochs=15,
			criterion=None,
			optimizer=None,
			load_checkpoint_mode: LoadCheckpointMode = None,
			force_overwrite: bool = False,
			early_stopping: bool = False,
			early_stopping_patience: int = 5,
			verbose: bool = True,
			p_bar_position: Optional[int] = None,
			p_bar_leave: Optional[bool] = None,
	):
		if criterion is None:
			criterion = nn.NLLLoss()
		if optimizer is None:
			# same hyper-parameters as the reference (snn.py:299); on the GPU the multi-tensor capturable variant is
			# (libsnnk's one-launch step) is used so that the step can live inside the captured training graph
			if self.device.type == "cuda":
				from .optim import FusedAdam
				optimizer = FusedAdam(self.parameters(), lr=lr, weight_decay=1e-5)
				if os.environ.get("SNNK_DP_FUSED", "1") != "0":
					optimizer.enable_data_parallel()    # no-op on one rank: gradient mean rides in the Adam launch
			else:
				optimizer = torch.optim.Adam(self.parameters(), lr=lr, weight_decay=1e-5)

		start_epoch = self._prepare_run(optimizer, load_checkpoint_mode, force_overwrite, verbose)
		if start_epoch >= nb_epochs:
			return self.loss_history

		best_loss = self.loss_history.min("val")
		p_bar = tqdm(
			range(start_epoch, nb_epochs), desc="Training", disable=not verbose, position=p_bar_position,
			unit="epoch", leave=p_bar_leave)
		for epoch in p_bar:
			epoch_loss = self._exec_phase(train_dataloader, val_dataloader, criterion, optimizer)
			# data parallel: every rank sees the same (mean) epoch losses, so is_best, the checkpoint index and the
			# early-stopping break are decided identically everywhere (a rank leaving the loop alone would leave the
			# others waiting in the gradient exchange)
			epoch_loss, self.last_eval_accuracy = self._dp_mean_epoch_stats(epoch_loss, self.last_eval_accuracy)
			epoch_val_acc = self.last_eval_accuracy     # counted in the validation pass that produced the loss
			self.loss_history.concat(epoch_loss)
			is_best = epoch_loss["val"] < best_loss
			self.save_checkpoint(optimizer, epoch, epoch_loss, is_best)
			if is_best:
				best_loss = epoch_loss["val"]
			if hasattr(p_bar, "set_postfix"):
				p_bar.set_postfix(
					train_loss=f"{epoch_loss['train']:.5e}", val_loss=f"{epoch_loss['val']:.5e}",
					val_acc=f"{epoch_val_acc:.5f}")
			if early_stopping and self._check_early_stopping(early_stopping_patience):
				if verbose:
					logging.info(f"Early stopping stopped the training at epoch {epoch}.")
				break
		if hasattr(p_bar, "close"):
			p_bar.close()
		self.plot_loss_history(show=False)
		return self.loss_history

	@staticmethod
	def _dp_world() -> int:
		import torch.distributed as dist
		return dist.get_world_size() if (dist.is_available() and dist.is_initialized()) else 1

	def _dp_barrier(self):
		if self._dp_world() > 1:
			import torch.distributed as dist
			dist.barrier()

	def _dp_mean_epoch_stats(self, epoch_loss: Dict[str, float], acc: float):
		"""Mean over the ranks of the epoch's train / validation loss and validation accuracy (SURVEY.md 8e: the loss
		for logging is the all-reduce mean).  One tiny collective per epoch; identity on a single rank."""
		world = self._dp_world()
		if world == 1:
			return epoch_loss, acc
		import torch.distributed as dist
		keys = sorted(epoch_loss)
		dev = self.device if dist.get_backend() == "nccl" else torch.device("cpu")
		t = torch.tensor([float(epoch_loss[k]) for k in keys] + [float(acc)], dtype=torch.float64, device=dev)
		dist.all_reduce(t, op=dist.ReduceOp.SUM)
		t = (t / world).tolist()
		return {k: v for k, v in zip(keys, t[:-1])}, t[-1]

	def _exec_phase(self, train_dataloader, val_dataloader, criterion, optimizer):
		self.train()
		train_loss = self._exec_epoch(train_dataloader, criterion, optimizer)
		self.eval()
		val_loss = self._exec_epoch(val_dataloader, criterion, optimizer)
		return dict(train=train_loss, val=val_loss)

	def _exec_epoch(self, dataloader, criterion, optimizer):
		"""Mean batch loss of one pass over ``dataloader`` (reference snn.py:376-382), accumulated on the device in
		float64 and read back once.  In eval mode the same pass also counts correct predictions
		(``self.last_eval_accuracy``), which ``fit`` reports instead of running the validation set a second time."""
		total = torch.zeros((), dtype=torch.float64, device=self.device)
		correct = torch.zeros((), dtype=torch.float64, device=self.device)
		n_batches = n_samples = 0
		for x_batch, y_batch in dataloader:
			if self.training:
				loss = self._exec_batch_device(x_batch, y_batch, criterion, optimizer)
			else:
				loss, c = self._eval_batch_device(x_batch, y_batch, criterion)
				correct += c
				n_samples += int(y_batch.shape[0])
			total += loss.double()
			n_batches += 1
		if not self.training:
			self.last_eval_accuracy = float(correct.item() / n_samples) if n_samples else float("nan")
		return float(total.item() / n_batches) if n_batches else float("nan")

	@staticmethod
	def _is_plain_nll(criterion) -> bool:
		return (
			type(criterion) is nn.NLLLoss and criterion.weight is None and criterion.reduction == "mean"
			and criterion.ignore_index == -100)

	def batch_loss(self, x_batch, y_batch, criterion=None, traces: bool = False) -> torch.Tensor:
		"""Loss tensor of one batch (on the device, attached to the graph in train mode).

		With the default criterion (``nn.NLLLoss`` mean) the fused head + fused BPTT kernels are used; any other
		criterion receives log-probabilities exactly as in the reference and is differentiated by autograd.
		"""
		x = self._encode_if_needed(x_batch.to(self.device, non_blocking=True))
		y = y_batch.to(self.device, non_blocking=True)
		if criterion is None or self._is_plain_nll(criterion):
			x = self._run_inner_layers(self._format_inputs(x))
			loss, *_ = F_.SpikingSequenceNLL.apply(self._consts(), x, y.long(), *self._weights(), traces)
			return loss
		log_p_y, out, h_states = self.get_prediction_log_proba(x, re_outputs_trace=True, re_hidden_states=True)
		return criterion(log_p_y, y.long())

	def graphed_train_step(self, x_example, y_example, criterion, optimizer, static_inputs: bool = False):
		"""Captures (once per input geometry) and returns the CUDA-graph version of one training step.

		With ``static_inputs`` the given device tensors themselves are the graph's inputs (call the step without
		arguments); otherwise every call copies its batch into the graph's static buffers first."""
		from .graphed import GraphedTrainStep
		key = (tuple(x_example.shape), x_example.dtype, tuple(y_example.shape), y_example.dtype, id(optimizer), id(criterion),
			(x_example.data_ptr(), y_example.data_ptr()) if static_inputs else None)
		step = self._graphed_steps.get(key)
		if step is None:
			step = GraphedTrainStep(self, x_example, y_example, criterion, optimizer, static_inputs=static_inputs)
			self._graphed_steps[key] = step
		return step

	def _exec_batch_device(self, x_batch, y_batch, criterion, optimizer) -> torch.Tensor:
		"""``_exec_batch`` without the host read-back: the batch loss as a 0-d device tensor (valid until the next
		call).  The epoch loop accumulates these on the device and synchronises once per epoch (SURVEY.md 8f.4)."""
		if self.training and self.cuda_graphs and self.device.type == "cuda":
			key = (tuple(x_batch.shape), x_batch.dtype, tuple(y_batch.shape), y_batch.dtype, id(optimizer), id(criterion))
			seen = self._graph_seen.get(key, 0)
			self._graph_seen[key] = seen + 1
			if seen >= 1:   # a geometry that repeats (every full batch of an epoch): capture once, replay afterwards
				step = self.graphed_train_step(x_batch, y_batch, criterion, optimizer)
				self._last_graphed_step = step
				return step(x_batch, y_batch)
		self._last_graphed_step = None
		if self.training:
			batch_loss = self.batch_loss(x_batch, y_batch, criterion)
			optimizer.zero_grad()
			batch_loss.backward()
			self._allreduce_gradients(optimizer)
			optimizer.step()
		else:
			with torch.no_grad():
				batch_loss = self.batch_loss(x_batch, y_batch, criterion)
		return batch_loss.detach()

	def _exec_batch(self, x_batch, y_batch, criterion, optimizer):
		"""forward (+ backward + optimizer step in train mode) -> python float (reference snn.py:384-415)."""
		loss = self._exec_batch_device(x_batch, y_batch, criterion, optimizer)
		step = self._last_graphed_step
		if step is not None and loss is step.loss:
			return step.wait_loss()      # posted to pinned host memory by the head kernel: no stream synchronisation
		return loss.item()

	def _eval_batch_device(self, x_batch, y_batch, criterion):
		"""Validation batch in ONE pass: (loss, number of correct predictions) as device tensors.  The reference runs
		the validation set twice per epoch (loss in ``_exec_phase``, accuracy in ``compute_classification_accuracy``,
		snn.py:333-334); the fused head already yields the log-probabilities the accuracy needs."""
		with torch.no_grad():
			x = self._encode_if_needed(x_batch.to(self.device, non_blocking=True))
			y = y_batch.to(self.device, non_blocking=True).long()
			if criterion is None or self._is_plain_nll(criterion):
				x = self._run_inner_layers(self._format_inputs(x))
				loss, logp, *_ = F_.SpikingSequenceNLL.apply(self._consts(), x, y, *self._weights(), False)
			else:
				logp, out, h_states = self.get_prediction_log_proba(x, re_outputs_trace=True, re_hidden_states=True)
				loss = criterion(logp, y)
			return loss.detach(), torch.eq(torch.argmax(logp, dim=-1), y).sum()

	def _allreduce_gradients(self, optimizer=None):
		"""Data-parallel training: average the (small) gradients over the ranks with one flat NCCL all-reduce --
		unless the optimizer does the exchange itself (``FusedAdam.enable_data_parallel``)."""
		if getattr(optimizer, "reduces_gradients", False):
			return
		from ..distributed import allreduce_mean_
		allreduce_mean_(p.grad for p in self.parameters())

	# ---- checkpoints (reference snn.py:417-505; same files and index layout, so checkpoints interchange) -------------
	# On disk: one "<model>-epoch<N>.pth" per epoch ({epoch, model_state_dict, optimizer_state_dict, loss}) and the index
	# "<model>-checkpoints.json" = {"epochs": {"<N>": path, ...}, "best": path}.
	def _folder(self) -> str:
		# the reference writes "./{checkpoint_folder}/..." (snn.py:421, :425); absolute folders are kept usable here
		f = str(self.checkpoint_folder)
		return f if os.path.isabs(f) else f"./{f}"

	@staticmethod
	def _is_writer() -> bool:
		"""In a data-parallel run (one process per GPU, identical replicas) only rank 0 touches the checkpoint folder."""
		import torch.distributed as dist
		return not (dist.is_available() and dist.is_initialized()) or dist.get_rank() == 0

	def _read_index(self) -> dict:
		with open(self.checkpoints_meta_path, "r") as fh:
			return json.load(fh)

	def _load_file(self, path: str) -> dict:
		"""Checkpoints written here hold tensors and plain Python numbers only, so they load under torch's safe
		``weights_only`` unpickler; files written by the reference (numpy scalars in the loss entry, snn.py:443-448,
		which torch >= 2.6 refuses by default, :481) are retried with exactly those numpy types allow-listed; anything that
		still needs the unrestricted unpickler is refused unless SNNK_TRUST_CHECKPOINTS=1 (it can run arbitrary code)."""
		import pickle
		import warnings
		try:
			return torch.load(path, map_location=self.device, weights_only=True)
		except pickle.UnpicklingError:
			pass       # only the safe unpickler's refusal is retried; I/O errors and corrupt files propagate
		# reference-written files: the loss entry holds numpy scalars (snn.py:443-448) -- allow exactly those types
		allowed = [np.dtype, np.ndarray, np.float64, np.float32, np.int64, type(np.dtype(np.float64)),
			type(np.dtype(np.float32)), type(np.dtype(np.int64))]
		core = getattr(np, "_core", None) or getattr(np, "core")
		allowed += [core.multiarray.scalar, core.multiarray._reconstruct]
		try:
			with torch.serialization.safe_globals(allowed):
				return torch.load(path, map_location=self.device, weights_only=True)
		except pickle.UnpicklingError as e:
			if os.environ.get("SNNK_TRUST_CHECKPOINTS", "0") != "1":
				raise RuntimeError(
					f"{path} needs the unrestricted unpickler ({e}); it can execute arbitrary code. Set "
					"SNNK_TRUST_CHECKPOINTS=1 to load files you trust.") from e
			warnings.warn(f"loading {path} with the unrestricted unpickler (SNNK_TRUST_CHECKPOINTS=1)")
			return torch.load(path, map_location=self.device, weights_only=False)

	def plot_loss_history(self, loss_history: LossHistory = None, show=False):
		history = self.loss_history if loss_history is None else loss_history
		if not self._is_writer():
			return
		os.makedirs(self._folder(), exist_ok=True)
		history.plot(os.path.join(self._folder(), "loss_history.png"), show)

	def _create_checkpoint_path(self, epoch: int = -1):
		name = f"{self.model_name}{SNN.SUFFIX_SEP}{SNN.CHECKPOINT_EPOCH_KEY}{epoch}{SNN.SAVE_EXT}"
		return f"{self._folder()}/{name}"

	def _create_new_checkpoint_meta(self, epoch: int, best: bool = False) -> dict:
		path = self._create_checkpoint_path(epoch)
		entry = {SNN.CHECKPOINT_EPOCHS_KEY: {epoch: path}}
		return {**entry, SNN.CHECKPOINT_BEST_KEY: path} if best else entry

	def save_checkpoints_meta(self, new_info: dict):
		index = self._read_index() if os.path.exists(self.checkpoints_meta_path) else {}
		mapping_update_recursively(index, new_info)
		with open(self.checkpoints_meta_path, "w") as fh:
			json.dump(index, fh, indent=4)

	def save_checkpoint(self, optimizer, epoch: int, epoch_losses: Dict[str, Any], best: bool = False):
		if not self._is_writer():
			return
		os.makedirs(self.checkpoint_folder, exist_ok=True)
		payload = {
			SNN.CHECKPOINT_EPOCH_KEY: epoch,
			SNN.CHECKPOINT_STATE_DICT_KEY: self.state_dict(),
			SNN.CHECKPOINT_OPTIMIZER_STATE_DICT_KEY: optimizer.state_dict(),
			SNN.CHECKPOINT_LOSS_KEY: {phase: float(v) for phase, v in epoch_losses.items()},     # plain floats: weights_only-safe
		}
		torch.save(payload, self._create_checkpoint_path(epoch))
		self.save_checkpoints_meta(self._create_new_checkpoint_meta(epoch, best))

	@staticmethod
	def get_save_path_from_checkpoints(
			checkpoints_meta: Dict[str, Union[str, Dict[Any, str]]],
			load_checkpoint_mode: LoadCheckpointMode = LoadCheckpointMode.BEST_EPOCH
	) -> str:
		if load_checkpoint_mode == LoadCheckpointMode.BEST_EPOCH:
			return checkpoints_meta[SNN.CHECKPOINT_BEST_KEY]
		if load_checkpoint_mode == LoadCheckpointMode.LAST_EPOCH:
			per_epoch = checkpoints_meta[SNN.CHECKPOINT_EPOCHS_KEY]       # json keys are strings
			return per_epoch[str(max(int(e) for e in per_epoch))]
		raise ValueError()

	def get_checkpoints_loss_history(self) -> LossHistory:
		history = LossHistory()
		for path in self._read_index()[SNN.CHECKPOINT_EPOCHS_KEY].values():
			history.concat(self._load_file(path)[SNN.CHECKPOINT_LOSS_KEY])
		return history

	def load_checkpoint(self, load_checkpoint_mode: LoadCheckpointMode = LoadCheckpointMode.BEST_EPOCH) -> dict:
		"""Loads the chosen checkpoint's weights into the model and returns the whole checkpoint dict."""
		ck = self._load_file(self.get_save_path_from_checkpoints(self._read_index(), load_checkpoint_mode))
		self.load_state_dict(ck[SNN.CHECKPOINT_STATE_DICT_KEY], strict=True)
		return ck

	# ---- evaluation (reference snn.py:507-555) ---------------------------------------------------------------------
	def compute_classification_accuracy(self, dataloader: DataLoader, verbose: bool = False, desc: Optional[str] = None) -> float:
		"""Accuracy over a dataloader; the per-batch comparison stays on the device, one host read at the end."""
		self.eval()
		correct = torch.zeros((), dtype=torch.float64, device=self.device)
		total = 0
		with torch.no_grad():
			for inputs, classes in tqdm(dataloader, total=len(dataloader), desc=desc, disable=not verbose):
				classes = classes.to(self.device)
				outputs = self.get_prediction_logits(inputs, re_outputs_trace=False, re_hidden_states=False)
				_, preds = torch.max(outputs, -1)
				correct += torch.eq(preds, classes).sum()
				total += classes.numel()
		return (correct / max(total, 1)).item()

	def compute_confusion_matrix(self, nb_classes: int, dataloaders: Dict[str, DataLoader], fit=False, fit_kwargs=None,
			load_checkpoint_mode: LoadCheckpointMode = None):
		if fit_kwargs is None:
			fit_kwargs = {}
		if fit:
			self.fit(dataloaders["train"], dataloaders["val"], **fit_kwargs)
		if load_checkpoint_mode is not None:
			self.load_checkpoint(load_checkpoint_mode)
		return {key: self._compute_single_confusion_matrix(nb_classes, d) for key, d in dataloaders.items()}

	def _compute_single_confusion_matrix(self, nb_classes: int, dataloader: DataLoader) -> np.ndarray:
		self.eval()
		cm = torch.zeros((nb_classes, nb_classes), dtype=torch.int64, device=self.device)
		with torch.no_grad():
			for inputs, classes in dataloader:
				classes = classes.to(self.device).view(-1).long()
				outputs = self.get_prediction_logits(inputs, re_outputs_trace=False, re_hidden_states=False)
				preds = torch.max(outputs, -1)[1].view(-1)
				cm.view(-1).index_add_(0, classes * nb_classes + preds, torch.ones_like(preds))
		return cm.cpu().numpy().astype(np.float64)
