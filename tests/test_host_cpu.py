"""CPU-side checks: the Python mirror of the reference interface, and that the C-ABI library loads and exports
every symbol include/snnk.h declares (no compute calls: there is no GPU here)."""
import ctypes
import os
import re

import numpy as np
import pytest
import torch

from snnimageclassification_b200 import _cabi
from snnimageclassification_b200 import (
	ALIFLayer, LayerType, LayerType2Layer, LIFLayer, LoadCheckpointMode, ReadoutLayer, SNN, SpikeFuncType,
	SpikeFuncType2Func, HeavisidePhiApprox, HeavisideSigmoidApprox, ToSpikes)
from snnimageclassification_b200.modules.utils import LossHistory, batchwise_temporal_filter
from _util import load

CPU = torch.device("cpu")


def test_library_exports_every_declared_symbol():
	_cabi.build_extension()
	header = open(_cabi.INCLUDE).read()
	declared = sorted(set(re.findall(r"\b(snnk_[a-z_0-9]+)\s*\(", header)))
	assert declared, "no entry points parsed from include/snnk.h"
	lib = ctypes.CDLL(_cabi.LIB_PATH)
	for name in declared:
		assert hasattr(lib, name), f"{name} declared in snnk.h but not exported by libsnnk.so"
	assert sorted(_cabi.EXPORTS) == declared, "python binding and header disagree on the entry points"
	assert _cabi.lib().snnk_abi_version() == 8
	assert b"sm_100" in _cabi.lib().snnk_strerror(-3)


def test_desc_struct_matches_header_layout():
	assert ctypes.sizeof(_cabi.SnnkDesc) == 24 * 4
	assert _cabi.SnnkDesc.alpha.offset == 32 and _cabi.SnnkDesc.flags.offset == 52


SPECS = {
	"alif_rec_lb": dict(hidden_layer_type=LayerType.ALIF, use_recurrent_connection=True, learn_beta=True),
	"alif_nonrec": dict(hidden_layer_type=LayerType.ALIF, use_recurrent_connection=False, learn_beta=False),
	"lif_rec": dict(hidden_layer_type=LayerType.LIF, use_recurrent_connection=True),
	"lif_two_hidden": dict(hidden_layer_type=LayerType.LIF, use_recurrent_connection=True),
}


@pytest.mark.parametrize("name", list(SPECS))
def test_same_seed_same_weights_as_reference(name):
	"""Parameter names, order, shapes and the RNG consumption order match the reference's SNN (snn.py:93, :149-157)."""
	z = load("init_golden.npz")
	torch.manual_seed(42)
	hidden = [24, 16] if name == "lif_two_hidden" else 24
	net = SNN(20, 10, hidden, int_time_steps=5, spike_func=SpikeFuncType.FastSigmoid, device=CPU, **SPECS[name])
	assert list(net.state_dict().keys()) == list(z[f"{name}/__keys__"])
	assert [n for n, _ in net.named_parameters()] == list(z[f"{name}/__params__"])
	for k, v in net.state_dict().items():
		assert np.array_equal(v.numpy(), z[f"{name}/{k}"]), k


def test_reference_quirks_are_kept():
	torch.manual_seed(0)
	net = SNN(16, 10, 32, hidden_layer_type=LayerType.ALIF, spike_func=SpikeFuncType.FastSigmoid, device=CPU,
		learn_beta=True)
	L = net.layers["input"]
	assert isinstance(L, ALIFLayer) and isinstance(L.beta, torch.nn.Parameter)
	assert abs(float(L.beta)) < 0.5          # re-drawn ~N(0, 0.03^2), not 1.6 (SURVEY 0.5)
	assert float(L.gamma) == pytest.approx(0.3) and float(L.threshold) == pytest.approx(0.03)
	assert float(L.alpha) == pytest.approx(np.exp(-1 / 20), rel=1e-6)
	assert float(L.rho) == pytest.approx(np.exp(-1 / 200), rel=1e-6)
	assert float(net.layers["readout"].kappa) == pytest.approx(np.exp(-1 / 10), rel=1e-6)
	assert torch.equal(L.rec_mask, 1 - torch.eye(32))
	assert "rec_mask" not in dict(L.named_buffers())
	lif = LIFLayer(8, 32, device=CPU)
	assert float(lif.gamma) == 1.0 and float(lif.threshold) == 1.0
	assert float(lif.alpha) == pytest.approx(np.exp(-1 / 10), rel=1e-6)
	assert LayerType2Layer[LayerType.ALIF] is ALIFLayer
	assert SpikeFuncType2Func[SpikeFuncType.Phi] is HeavisidePhiApprox
	assert SpikeFuncType2Func[SpikeFuncType.FastSigmoid] is HeavisideSigmoidApprox
	assert HeavisidePhiApprox.epsilon == 1e-5
	assert [m.name for m in LoadCheckpointMode] == ["BEST_EPOCH", "LAST_EPOCH"]


def test_no_cpu_fallback():
	net = SNN(16, 10, 32, hidden_layer_type=LayerType.LIF, device=CPU, int_time_steps=4)
	with pytest.raises(RuntimeError, match="no CPU fallback"):
		net(torch.zeros(2, 4, 16))
	with pytest.raises(RuntimeError, match="no CPU fallback"):
		HeavisideSigmoidApprox.apply(torch.zeros(4), torch.tensor(1.0), torch.tensor(1.0))
	if not torch.cuda.is_available():
		with pytest.raises(RuntimeError, match="no CPU fallback"):
			ToSpikes(10)(np.zeros(4))
	izh = SNN(16, 10, 32, hidden_layer_type=LayerType.Izhikevich, device=CPU, int_time_steps=4)
	with pytest.raises(RuntimeError, match="no CPU fallback"):
		izh(torch.zeros(2, 4, 16))
	wide = SNN(16, 10, 256, hidden_layer_type=LayerType.Izhikevich, device=CPU, int_time_steps=4)
	with pytest.raises(RuntimeError, match="no CPU fallback"):      # wide Izhikevich layers are supported -- on the GPU
		wide(torch.zeros(2, 4, 16))
	V, u, Z = izh.layers["input"].create_empty_state(3)           # reference spiking_layers.py:308-328
	assert float(V.min()) == float(V.max()) == -60.0 and float(u.abs().max()) == 0.0 and float(Z.abs().max()) == 0.0


def test_readout_wider_than_16_classes_is_refused_at_construction():
	for O in (1, 16):
		assert SNN(16, O, 32, device=CPU, int_time_steps=4).layers["readout"].forward_weights.shape == (32, O)
	for O in (17, 0):
		with pytest.raises(ValueError, match="1 to 16 classes"):
			SNN(16, O, 32, device=CPU, int_time_steps=4)


def test_format_inputs():
	net = SNN(6, 10, 32, device=CPU, int_time_steps=5)
	x = torch.arange(12, dtype=torch.float64).reshape(2, 6)
	f = net._format_inputs(x)
	assert f.shape == (2, 5, 6) and f.dtype == torch.float32
	assert torch.equal(f[:, 3], x.float())
	f = net._format_inputs(torch.ones(2, 3, 6))
	assert f.shape == (2, 5, 6) and f[:, 3:].abs().sum() == 0 and f[:, :3].sum() == 36
	with pytest.raises(AssertionError):
		net._format_inputs(torch.ones(2, 6, 6))


def test_checkpoint_files_interchange(tmp_path):
	net = SNN(6, 10, 32, hidden_layer_type=LayerType.ALIF, device=CPU, int_time_steps=5, learn_beta=True,
		checkpoint_folder=str(tmp_path / "ck"), model_name="m")
	opt = torch.optim.Adam(net.parameters(), lr=1e-3, weight_decay=1e-5)
	net.save_checkpoint(opt, 0, dict(train=1.0, val=2.0), best=True)
	net.save_checkpoint(opt, 1, dict(train=0.5, val=2.5), best=False)
	assert net.checkpoints_meta_path.endswith("ck/m-checkpoints.json")
	assert os.path.exists(tmp_path / "ck" / "m-epoch1.pth")
	w = net.layers["input"].forward_weights.detach().clone()
	with torch.no_grad():
		net.layers["input"].forward_weights.zero_()
	ck = net.load_checkpoint(LoadCheckpointMode.LAST_EPOCH)
	assert ck["epoch"] == 1 and torch.equal(net.layers["input"].forward_weights, w)
	assert net.load_checkpoint(LoadCheckpointMode.BEST_EPOCH)["epoch"] == 0
	hist = net.get_checkpoints_loss_history()
	assert hist["val"] == [2.0, 2.5] and hist.min("val") == 2.0


def test_loss_history_and_temporal_filter():
	h = LossHistory()
	assert h.min("val") == np.inf
	h.concat(dict(train=1.0, val=3.0)); h.concat(dict(train=[0.5], val=[2.0]))
	assert h["train"] == [1.0, 0.5] and h.min_item("val") == dict(train=0.5, val=2.0)
	# known answers of the reference's test/test_temporal_filter.py
	x = torch.ones(1, 3, 1)
	assert torch.allclose(batchwise_temporal_filter(x, 0.5), torch.tensor([[1.75]]))


def test_host_side_size_queries():
	"""Pure host entry points of the C ABI (no device needed): run-table and exchange-buffer sizes."""
	lib = _cabi.lib()
	B, T = 256, 100
	cap = max(128, (B * T // 4 + 127) // 128 * 128)
	assert lib.snnk_run_table_bytes(B, T) == 4 * (4 + B * T + 2 * cap + B)
	assert lib.snnk_run_table_bytes(3, 5) == 4 * (4 + 15 + 2 * 128 + 3)
	assert lib.snnk_run_table_bytes(0, 5) == 0 and lib.snnk_run_table_bytes(1 << 28, 100) == 0
	n = ctypes.c_size_t(0)
	assert lib.snnk_adam_dp_buffer_bytes(8, 118026, ctypes.byref(n)) == 0 and n.value == 2 * 8 * 118026 * 8
	assert lib.snnk_adam_dp_buffer_bytes(17, 10, ctypes.byref(n)) != 0 and lib.snnk_adam_dp_buffer_bytes(0, 10, ctypes.byref(n)) != 0


def test_fused_adam_data_parallel_needs_a_process_group():
	from snnimageclassification_b200 import FusedAdam
	p = torch.nn.Parameter(torch.zeros(4))
	opt = FusedAdam([p], lr=1e-3)
	assert opt.enable_data_parallel() is False and opt.reduces_gradients is False
	p.grad = torch.ones(4)
	with pytest.raises(RuntimeError, match="no CPU fallback"):
		opt.step()


def test_run_table_tag_is_validated():
	from snnimageclassification_b200.modules.functional import get_runs, mark_binary
	x = torch.zeros(2, 5, 8)
	assert get_runs(x) is None
	mark_binary(x, runs=torch.zeros(7, dtype=torch.int32))          # wrong size for (2, 5): ignored
	assert get_runs(x) is None
	need = _cabi.lib().snnk_run_table_bytes(2, 5) // 4
	mark_binary(x, runs=torch.zeros(need, dtype=torch.int32))
	assert get_runs(x) is not None
	assert get_runs(mark_binary(torch.zeros(2, 5, 8), runs=torch.zeros(need, dtype=torch.int64))) is None
	# a table followed by the tiled compact rows (snnk_run_table_tiled_bytes) is accepted too, and recognised as such
	from snnimageclassification_b200.modules.functional import runs_tiled
	tiled = _cabi.lib().snnk_run_table_tiled_bytes(2, 5, 8) // 4
	assert tiled > need and _cabi.lib().snnk_run_table_tiled_bytes(2, 5, 6) == 0          # n_pix % 4 != 0: no tiled form
	assert not runs_tiled(x)
	y = mark_binary(torch.zeros(2, 5, 8), runs=torch.zeros(tiled, dtype=torch.int32))
	assert get_runs(y) is not None and runs_tiled(y)
	assert get_runs(mark_binary(torch.zeros(2, 5, 8), runs=torch.zeros(tiled - 1, dtype=torch.int32))) is None


def test_fused_adam_load_state_dict_normalises_foreign_state():
	"""Loading a plain torch.optim.Adam state (ADVICE r1): capturable groups, float32 0-d step tensors on the parameter's
	device -- checked on CPU parameters (step() itself needs the GPU and is covered by the gpu tests)."""
	from snnimageclassification_b200 import FusedAdam
	ps = [torch.randn(4, 3, requires_grad=True), torch.randn(3, requires_grad=True)]
	ref = torch.optim.Adam(ps, lr=2e-3, weight_decay=1e-5)
	for p in ps:
		p.grad = torch.randn_like(p)
	ref.step(); ref.step()
	mine = FusedAdam([p.detach().clone().requires_grad_() for p in ps], lr=1e-3)
	v0 = mine.hyper_signature()
	mine.load_state_dict(ref.state_dict())
	assert mine.hyper_signature() != v0             # a captured graph would be re-captured
	for g in mine.param_groups:
		assert g["capturable"] is True and g["foreach"] is False and g["lr"] == 2e-3
	for p in mine.param_groups[0]["params"]:
		st = mine.state[p]
		assert st["step"].dtype == torch.float32 and st["step"].ndim == 0 and float(st["step"]) == 2.0


def test_reference_style_checkpoint_loads_without_full_unpickling(tmp_path):
	"""A checkpoint as the reference writes it (numpy scalars in the loss entry, snn.py:443-448) loads through the
	allow-listed safe unpickler; a file that needs arbitrary globals is refused unless explicitly trusted."""
	net = SNN(6, 10, 32, hidden_layer_type=LayerType.LIF, device=CPU, int_time_steps=5,
		checkpoint_folder=str(tmp_path / "ck"), model_name="m")
	path = str(tmp_path / "ref.pth")
	torch.save({"epoch": 3, "model_state_dict": net.state_dict(), "optimizer_state_dict": {},
		"loss": {"train": np.float64(0.25), "val": np.float32(0.5)}}, path)
	ck = net._load_file(path)
	assert ck["epoch"] == 3 and float(ck["loss"]["train"]) == 0.25

	class Evil:
		def __reduce__(self):
			return (os.getcwd, ())
	bad = str(tmp_path / "bad.pth")
	torch.save({"epoch": 0, "payload": Evil()}, bad)
	with pytest.raises(RuntimeError, match="SNNK_TRUST_CHECKPOINTS"):
		net._load_file(bad)
	with pytest.raises(FileNotFoundError):
		net._load_file(str(tmp_path / "missing.pth"))


def test_packed_raster_tagging_and_passthrough():
	"""Host logic of SNNK_F_INPUT_BITS: which int32 tensors count as packed rasters, when SNN keeps them packed."""
	from snnimageclassification_b200.modules import functional as F_
	bits = torch.zeros(2, 5, 25, dtype=torch.int32)
	assert F_.bits_width(bits) is None
	assert F_.bits_width(F_.mark_bits(bits, 784)) == 784
	assert F_.bits_width(F_._c(bits)) == 784 and F_._c(bits).dtype == torch.int32      # stays packed through the glue
	with pytest.raises(ValueError):
		F_.mark_bits(torch.zeros(2, 5, 24, dtype=torch.int32), 784)       # 784 features are 25 words
	with pytest.raises(ValueError):
		F_.mark_bits(torch.zeros(2, 5, 25), 784)                          # not int32
	assert F_.bits_eligible(784, True) and not F_.bits_eligible(784, False) and not F_.bits_eligible(786, True)
	net = SNN(784, 10, 32, device=CPU, int_time_steps=5)
	kept = net._encode_if_needed(torch.zeros(2, 5, 25, dtype=torch.int32))
	assert F_.bits_width(kept) == 784 and net._format_inputs(kept) is kept
	# fewer steps than int_time_steps: must be unpacked (and zero-padded) -- on the GPU; here the unpack refuses the CPU
	with pytest.raises(RuntimeError, match="no CPU fallback|CUDA"):
		net._encode_if_needed(torch.zeros(2, 3, 25, dtype=torch.int32))
	fp32 = SNN(784, 10, 32, device=CPU, int_time_steps=5, tensor_core=False)
	with pytest.raises(RuntimeError, match="no CPU fallback|CUDA"):
		fp32._encode_if_needed(torch.zeros(2, 5, 25, dtype=torch.int32))


def _bench_module():
	import importlib.util
	root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
	spec = importlib.util.spec_from_file_location("bench_mod", os.path.join(root, "bench.py"))
	bench = importlib.util.module_from_spec(spec)
	spec.loader.exec_module(bench)
	return bench


def test_bench_parses_the_committed_ncu_summary():
	"""bench.py takes `roofline.traffic` / `roofline.smem_frac` from profiles/r02_ncu_full_summary.csv (unit row respected):
	the headline kernels' rows must be found (lean kernels first) and carry sane numbers."""
	bench = _bench_module()
	k3 = bench.ncu_evidence("K3")
	assert k3 is not None and "k_recur_bwd_lean" in k3["kernel"]
	assert 20e6 < k3["traffic"] < 60e6                     # bytes per launch: V, a read once (26 MB), gI mostly stays in L2
	assert 30.0 < k3["ncu_duration_us"] < 100.0            # microseconds, not nanoseconds
	assert k3["smem_wavefronts"] > 1e6
	k2 = bench.ncu_evidence("K2")
	assert k2 is not None and "k_recur_fwd_lean" in k2["kernel"]
	assert bench.ncu_evidence("K1") is not None and bench.ncu_evidence("nope") is None
	flops, byts = bench.per_sample_work(128, True, True, True)
	assert abs(flops - 50.7e6) < 0.5e6 and abs(byts - 942e3) < 5e3      # SURVEY.md 8d: c2 = 50.7 MFLOP, 942 KB per sample


def test_bench_dump_outputs_writes_loss_and_parameters(tmp_path):
	"""bench.py --dump-outputs: the loss and every parameter, one float32 .npy file each, values unchanged."""
	bench = _bench_module()
	torch.manual_seed(0)
	net = SNN(20, 10, 24, hidden_layer_type=LayerType.ALIF, use_recurrent_connection=True, learn_beta=True, device=CPU,
		int_time_steps=5)
	out = tmp_path / "out"
	bench.dump_outputs(str(out), torch.tensor(1.25), net)
	params = dict(net.named_parameters())
	assert sorted(os.listdir(out)) == sorted(["loss.npy"] + [f"param.{n}.npy" for n in params])
	assert np.load(out / "loss.npy").tolist() == [1.25]
	for n, p in params.items():
		a = np.load(out / f"param.{n}.npy")
		assert a.dtype == np.float32 and np.array_equal(a, p.detach().numpy()), n
