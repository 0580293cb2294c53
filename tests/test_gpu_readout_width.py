"""Oracle parity across the supported readout widths (O = 1 to 16) in every kernel family.

Several code paths depend on the readout width: the lean forward keeps W_out at a pitch of kLeanOP = 12 and takes
O <= 12; the lean BPTT sweep is instantiated with OP = 12 (O <= 12) and OP = 16 (O = 13 to 16); the tensor-core
recurrence packs the spike bits into row 15 of its readout MMA and takes O <= 15; the scans behind the tensor-core,
non-recurrent and wide kernels pad the readout adjoint to 16 columns.  Every case here states which kernel family it
targets and checks, from the CUDA kernels the profiler saw, that the dispatcher launched it; the widths are chosen on
both sides of each threshold.

The readout data are chosen so that a column mix-up cannot cancel out: column c of W_out is scaled by (1 + c), the
biases are distinct, the reference gradient of the last class is non-zero and the arg-max steps are not constant.
"""
import re

import numpy as np
import pytest
import torch

import oracle
from oracle import OracleCfg
from oracle.torch_port import TorchPortSNN
from _util import elementwise_err, launched, ran, rel_err, unexplained_forks

pytestmark = pytest.mark.gpu

from snnimageclassification_b200 import LayerType, SNN, SpikeFuncType, ToSpikes  # noqa: E402
from snnimageclassification_b200.modules import functional as F_  # noqa: E402

DEV = torch.device("cuda:0")
WIDTHS = [1, 2, 12, 13, 15, 16]
ALPHA, RHO, KAPPA = (float(np.float32(np.exp(-1 / k))) for k in (20, 200, 10))


def npy(t):
	return None if t is None else t.detach().cpu().numpy()


def _targ(s):
	s = s.strip()
	return int(s == "true") if s in ("true", "false") else int(re.sub(r"\D", "", s))


def lean_bwd_variants(names):
	"""(ALIF, SURR, PLANES, RUNS, OP) of every k_recur_bwd_lean launch."""
	out = set()
	for n in names:
		m = re.search(r"k_recur_bwd_lean<([^<>]*)>", n)
		if m:
			out.add(tuple(_targ(v) for v in m.group(1).split(",")))
	return out


# ---- data ------------------------------------------------------------------------------------------------------------
class Case:
	"""Inputs, weights and constants of one layer + readout of width O; W_out column c scaled by (1 + c)."""

	def __init__(self, B, T, N, H, O, layer, rec, phi=0, tc=False, density=0.2, dedup=False, seed=0, wscale=1.0):
		g = torch.Generator().manual_seed(seed)
		self.B, self.T, self.N, self.H, self.O, self.layer, self.rec, self.phi = B, T, N, H, O, layer, rec, phi
		self.theta = theta = 0.03 if layer else 1.0
		if dedup:
			img = (torch.randint(1, 256, (B, N), generator=g).float() / 255.0) * (torch.rand(B, N, generator=g) < 0.3)
			self.x = ToSpikes(T, use_periods=True).encode_batch(img.to(DEV))
			assert F_.get_runs(self.x) is not None
		else:
			self.x = F_.mark_binary((torch.rand(B, T, N, generator=g) < density).float().to(DEV))
		self.W_in = (torch.randn(N, H, generator=g) * theta).to(DEV)
		self.W_rec = (torch.randn(H, H, generator=g) * theta / (4 if H > 128 else 1)).to(DEV) if rec else None
		self.mask = (1 - torch.eye(H)).to(DEV) if rec else None
		self.W_out = (torch.randn(H, O, generator=g) * (1.0 + torch.arange(O)) * wscale).to(DEV)
		self.b_out = (torch.randn(O, generator=g) * 0.1 + 0.05 * torch.arange(O)).to(DEV)
		assert len(set(npy(self.b_out).tolist())) == O
		self.beta = torch.tensor([1.6], device=DEV) if layer else None
		self.labels = torch.randint(0, O, (B,), generator=g).to(DEV)      # over all O classes
		self.seeds = (torch.randn(B, O, generator=g) / B).to(DEV)          # sweep seeds where the head's are all zero
		self.g_y = torch.randn(B, T, O, generator=g).to(DEV)               # dense seeds
		self.c = F_.LayerConsts(layer, phi, rec, ALPHA, RHO, theta, 0.3 if layer else 1.0, KAPPA, tensor_core=tc)
		self.cfg = OracleCfg(B, T, N, H, O, layer_type=layer, surrogate=phi, recurrent=int(rec), alpha=ALPHA, rho=RHO,
			theta=theta, gamma=0.3 if layer else 1.0, kappa=KAPPA, beta=1.6)

	def forward(self, labels=True, traces=True):
		return F_.run_forward(self.c, self.x, self.W_in, self.W_rec, self.mask, self.beta, self.W_out, self.b_out,
			traces=traces, labels=self.labels if labels else None)

	def backward(self, f, **kw):
		return F_.run_backward(self.c, self.x, self.W_rec, self.mask, self.beta, self.W_out, f["V"], f["a"], f["zbits"],
			Z=f["Z"], **kw)

	def sparse_seeds(self, f):
		"""g_logits for the sweep: the fused head's, except at O = 1 where they are exactly zero (then random ones)."""
		if self.O == 1:
			assert float(f["g_logits"].abs().max()) == 0.0 and float(f["loss"]) == 0.0
			return self.seeds
		return f["g_logits"]

	def oracle_forward(self):
		return oracle.forward(self.cfg, npy(self.x), npy(self.W_in), npy(self.W_rec), npy(self.mask), npy(self.W_out),
			npy(self.b_out))

	def oracle_backward(self, V, a, Z, g_y):
		return oracle.backward(self.cfg, npy(self.x), npy(self.W_rec), npy(self.mask), npy(self.W_out), V, a, Z, g_y)


def scatter_seeds(g_logits, tstar, T):
	"""The dense readout adjoint of sparse seeds: g_logits[b, c] at step tstar[b, c]."""
	gl, ts = npy(g_logits), npy(tstar).astype(np.int64)
	B, O = gl.shape
	g_y = np.zeros((B, T, O), np.float32)
	g_y[np.arange(B)[:, None], ts, np.arange(O)[None, :]] = gl
	return g_y


def check_columns(case, gref, tstar):
	"""The data can tell the classes apart: the last class has a gradient, the arg-max steps vary."""
	O = case.O
	assert np.abs(gref["dW_out"][:, O - 1]).max() > 0 and gref["db"][O - 1] != 0
	assert len(np.unique(npy(tstar))) > 1, "constant arg-max steps"


WEIGHTS = ("dW_in", "dW_out", "db")


def check_grads(case, g, gref, gI_tol, w_tol, elem_tol=None):
	assert rel_err(npy(g["gI"]()), gref["gI"]) <= gI_tol
	for k in WEIGHTS + (("dW_rec",) if case.rec else ()):
		assert rel_err(npy(g[k]), gref[k]) <= w_tol, (k, rel_err(npy(g[k]), gref[k]))
		if elem_tol is not None:
			assert elementwise_err(npy(g[k]), gref[k]) <= elem_tol, (k, elementwise_err(npy(g[k]), gref[k]))
	if case.rec:
		assert np.all(np.diag(npy(g["dW_rec"])) == 0.0)


def check_forward_exact(case, f, ref):
	for k in ("I_in", "V", "Z", "y") + (("a",) if case.layer else ()):
		assert np.array_equal(npy(f[k]), ref[k]), k
	assert 0.001 < ref["Z"].mean() < 0.999
	h = oracle.head(ref["y"], npy(case.labels))
	assert np.array_equal(npy(f["logits"]), h["logits"]) and np.array_equal(npy(f["tstar"]), h["tstar"])
	if "loss" in f:
		assert abs(float(f["loss"]) - h["loss"]) <= 1e-5 * abs(h["loss"])
		assert rel_err(npy(f["logp"]), h["logp"]) <= 1e-5
	return h


def check_forward_forks(case, f, ref, max_fork_frac=0.03):
	"""Tensor-core forward against the oracle: rasters up to forks at near-ties, state on the samples that did not fork,
	and the readout tail consistent with the kernel's own output trace."""
	if F_.get_runs(case.x) is None:         # with a run table the workspace holds the compact rows, not I_in
		assert rel_err(npy(f["I_in"]), ref["I_in"]) <= 1e-5
	thr = case.theta + (1.6 * ref["a"] if case.layer else 0.0)
	forked, unexplained = unexplained_forks(npy(f["Z"]), ref["Z"], ref["V"], thr)
	assert unexplained == 0, f"{unexplained} of {forked} forked samples differ first at a spike that is no near-tie"
	ok = ~(npy(f["Z"]) != ref["Z"]).any(axis=(1, 2))
	assert ok.mean() >= 1 - max_fork_frac, f"{forked} of {case.B} samples forked"
	for k in ("V", "y") + (("a",) if case.layer else ()):
		assert rel_err(npy(f[k])[ok], ref[k][ok]) <= 1e-5, k
	h = oracle.head(npy(f["y"]), npy(case.labels))
	assert np.array_equal(npy(f["logits"]), h["logits"]) and np.array_equal(npy(f["tstar"]), h["tstar"])
	assert abs(float(f["loss"]) - h["loss"]) <= 1e-5 * abs(h["loss"])
	return h


def dense_step(case):
	f = case.forward()
	return f, case.backward(f, g_y=case.g_y)


# ---- SIMT recurrences (recur_fwd.cuh / recur_bwd.cuh), fp32: bit-exact forward ----------------------------------------
@pytest.mark.parametrize("O", WIDTHS)
@pytest.mark.parametrize("H", [32, 64, 128])
def test_simt_vs_oracle(O, H, monkeypatch):
	monkeypatch.setenv("SNNK_LEAN", "0")      # the general kernels also at H = 128, O <= 12
	for layer, phi in ((0, 0), (0, 1), (1, 0), (1, 1)):
		case = Case(13, 9, 64, H, O, layer, True, phi=phi, seed=100 * O + H + 10 * layer + phi)
		(f, g), names = launched(lambda: dense_step(case))
		assert ran(names, r"k_recur_fwd<") and ran(names, r"k_recur_bwd<") and not ran(names, r"_lean<")
		ref = case.oracle_forward()
		check_forward_exact(case, f, ref)
		gref = case.oracle_backward(ref["V"], ref["a"], ref["Z"], npy(case.g_y))
		check_columns(case, gref, f["tstar"])
		check_grads(case, g, gref, 1e-5, 1e-5)


@pytest.mark.parametrize("O", WIDTHS)
def test_simt_two_rows_per_cta_vs_oracle(O):
	"""B > 1024: two rows per CTA (R = 2); the lean kernels are never selected there."""
	case = Case(1030, 6, 64, 128, O, O % 2, True, phi=(O // 2) % 2, seed=O)
	(f, g), names = launched(lambda: dense_step(case))
	assert ran(names, r"k_recur_fwd<128, 2\b") and ran(names, r"k_recur_bwd<128, 2\b")
	ref = case.oracle_forward()
	check_forward_exact(case, f, ref)
	gref = case.oracle_backward(ref["V"], ref["a"], ref["Z"], npy(case.g_y))
	check_columns(case, gref, f["tstar"])
	check_grads(case, g, gref, 1e-5, 1e-5)


# ---- lean forward + lean BPTT (recur_lean.cuh) == general kernels, bit for bit; and the oracle -------------------------
@pytest.mark.parametrize("O", WIDTHS)
@pytest.mark.parametrize("mode", ["fp32", "tc", "dedup"])
def test_lean_kernels_vs_general_and_oracle(O, mode, monkeypatch):
	"""O <= 12: lean forward (W_out at pitch kLeanOP) and the OP = 12 sweep; O >= 13: the general forward and the OP = 16
	sweep.  fp32: PLANES = false; tc: PLANES = true; dedup (encoded input with a run table): PLANES = RUNS = true."""
	monkeypatch.delenv("SNNK_MMA_RECUR", raising=False)
	tc = mode != "fp32"
	for layer, phi in ((0, 0), (0, 1), (1, 0), (1, 1)):
		case = Case(96, 14, 64, 128, O, layer, True, phi=phi, tc=tc, dedup=mode == "dedup",
			seed=1000 + 10 * O + 2 * layer + phi)
		res = {}
		for lean in ("1", "0"):
			monkeypatch.setenv("SNNK_LEAN", lean)

			def step():
				f = case.forward()
				gl = case.sparse_seeds(f)
				g = case.backward(f, g_logits=gl, tstar=f["tstar"], W_effT=f["W_effT"])
				f2 = case.forward(labels=False, traces=False)
				return f, gl, g, f2
			(f, gl, g, f2), names = launched(step)
			if lean == "1":
				assert ran(names, r"k_recur_fwd_lean<") == (O <= 12)
				assert ran(names, r"k_recur_fwd<") == (O > 12)
				want = (layer, phi, int(tc), int(mode == "dedup"), 12 if O <= 12 else 16)
				assert lean_bwd_variants(names) == {want}, (lean_bwd_variants(names), want)
			else:
				assert not ran(names, r"_lean<") and ran(names, r"k_recur_fwd<") and ran(names, r"k_recur_bwd<")
			res[lean] = dict(V=f["V"], a=f["a"], Z=f["Z"], y=f["y"], zbits=f["zbits"], logits=f["logits"],
				tstar=f["tstar"], loss=f["loss"], logp=f["logp"], g_logits=f["g_logits"], gI=g["gI"]().clone(),
				dW_in=g["dW_in"], dW_rec=g["dW_rec"], dW_out=g["dW_out"], db=g["db"], logits_infer=f2["logits"])
		for k, v in res["1"].items():
			if v is not None:
				assert torch.equal(v, res["0"][k]), (k, layer, phi)
		ref = case.oracle_forward()
		if tc:
			check_forward_forks(case, f, ref, max_fork_frac=0.05)
		else:
			check_forward_exact(case, f, ref)
		gref = case.oracle_backward(npy(f["V"]), npy(f["a"]), npy(f["Z"]), scatter_seeds(gl, f["tstar"], case.T))
		check_columns(case, gref, f["tstar"])
		check_grads(case, g, gref, 1e-5, 1e-4 if tc else 1e-5)      # tc: the dW_in GEMM on tf32 planes


# ---- tensor-core recurrence (recur_tc.cuh), forced at small batch --------------------------------------------------
@pytest.mark.parametrize("O", WIDTHS)
def test_tensor_core_recurrence_vs_oracle(O, monkeypatch):
	"""Row 15 of the readout MMA carries the spike bits: O <= 15 runs recur_tc.cuh, O = 16 must not."""
	monkeypatch.setenv("SNNK_MMA_RECUR", "1")
	for layer in (1, 0):
		case = Case(128, 20, 64, 128, O, layer, True, tc=True, density=0.15, seed=2000 + 10 * O + layer)

		def step():
			f = case.forward()
			gl = case.sparse_seeds(f)
			return f, gl, case.backward(f, g_logits=gl, tstar=f["tstar"])
		(f, gl, g), names = launched(step)
		assert ran(names, r"k_recur_fwd_tc\b") == (O <= 15) and ran(names, r"k_recur_bwd_tc\b") == (O <= 15)
		if O == 16:
			assert ran(names, r"k_recur_fwd<") and lean_bwd_variants(names) == {(layer, 0, 1, 0, 16)}
		ref = case.oracle_forward()
		check_forward_forks(case, f, ref)
		# gradients unconditionally: the oracle's sweep over the GPU's own traces
		gref = case.oracle_backward(npy(f["V"]), npy(f["a"]), npy(f["Z"]), scatter_seeds(gl, f["tstar"], case.T))
		check_columns(case, gref, f["tstar"])
		check_grads(case, g, gref, 1e-5, 1e-4, elem_tol=1e-3)


# ---- non-recurrent scans (recur_nr.cuh) --------------------------------------------------------------------------------
@pytest.mark.parametrize("O", WIDTHS)
@pytest.mark.parametrize("H", [32, 128])
def test_nonrecurrent_scans_vs_oracle(O, H):
	for layer in (1, 0):
		case = Case(64, 16, 64, H, O, layer, False, phi=layer, tc=True, seed=3000 + 10 * O + H + layer)

		def step():
			f = case.forward()
			gl = case.sparse_seeds(f)
			return f, gl, case.backward(f, g_logits=gl, tstar=f["tstar"])
		(f, gl, g), names = launched(step)
		assert ran(names, r"k_nonrec_fwd<") and ran(names, r"k_nonrec_bwd<")
		ref = case.oracle_forward()
		check_forward_forks(case, f, ref, max_fork_frac=0.05)
		gref = case.oracle_backward(npy(f["V"]), npy(f["a"]), npy(f["Z"]), scatter_seeds(gl, f["tstar"], case.T))
		check_columns(case, gref, f["tstar"])
		check_grads(case, g, gref, 1e-5, 1e-5)


# ---- wide layers: weight-stationary tensor-core kernels (recur_wide.cuh) and generic fp32 kernels (recur_gen.cuh) -------
@pytest.mark.parametrize("O", WIDTHS)
def test_wide_layers_vs_oracle(O):
	for layer in (1, 0):
		case = Case(6, 10, 64, 256, O, layer, True, seed=4000 + 10 * O + layer, density=0.15, wscale=1 / 8)
		f, names = launched(lambda: case.forward())
		assert ran(names, r"k_recur_fwd_gen<") and ran(names, r"k_readout_scan\b") and not ran(names, r"k_wide_fwd<")
		ref = case.oracle_forward()
		check_forward_exact(case, f, ref)
		gl = case.sparse_seeds(f)
		gref = case.oracle_backward(ref["V"], ref["a"], ref["Z"], scatter_seeds(gl, f["tstar"], case.T))
		check_columns(case, gref, f["tstar"])
		for tc, kern in ((False, r"k_recur_bwd_gen<"), (True, r"k_wide_bwd<")):
			c = F_.LayerConsts(layer, 0, True, ALPHA, RHO, case.theta, case.c.gamma, KAPPA, tensor_core=tc)
			g, names = launched(lambda: F_.run_backward(c, case.x, case.W_rec, case.mask, case.beta, case.W_out, f["V"],
				f["a"], f["zbits"], g_logits=gl, tstar=f["tstar"], Z=f["Z"]))
			assert ran(names, kern) and ran(names, r"k_wout_grad\b"), tc
			check_grads(case, g, gref, 1e-5, 1e-4)
		# the weight-stationary forward: projection within 1e-5, readout tail consistent with its own trace
		case.c = F_.LayerConsts(layer, 0, True, ALPHA, RHO, case.theta, case.c.gamma, KAPPA, tensor_core=True)
		f2, names = launched(lambda: case.forward())
		assert ran(names, r"k_wide_fwd<") and ran(names, r"k_readout_scan\b")
		assert rel_err(npy(f2["I_in"]), ref["I_in"]) <= 1e-5
		h2 = oracle.head(npy(f2["y"]), npy(case.labels))
		assert np.array_equal(npy(f2["logits"]), h2["logits"]) and np.array_equal(npy(f2["tstar"]), h2["tstar"])


# ---- Izhikevich, fp32 kernels ----------------------------------------------------------------------------------------
@pytest.mark.parametrize("O,rec", [(1, True), (16, True), (16, False)])
def test_izhikevich_fp32_kernels_vs_oracle(O, rec):
	B, T, N, H = 6, 25, 48, 64
	torch.manual_seed(7 + O)
	net = SNN(N, O, H, use_recurrent_connection=rec, int_time_steps=T, dt=1.0, hidden_layer_type=LayerType.Izhikevich,
		spike_func=SpikeFuncType.FastSigmoid, device=DEV, tensor_core=False)
	L, R = net.layers["input"], net.layers["readout"]
	with torch.no_grad():
		L.forward_weights.mul_(25.0).add_(20.0)
		if rec:
			L.recurrent_weights.mul_(5.0)
		R.forward_weights.mul_(1.0 + torch.arange(O, device=DEV))
		R.bias_weights.copy_(torch.randn(O) * 0.1 + 0.05 * torch.arange(O))
	g = torch.Generator().manual_seed(4)
	x = (torch.rand(B, T, N, generator=g) < 0.2).float()
	lab = torch.randint(0, O, (B,), generator=g)
	cfg = OracleCfg(B, T, N, H, O, layer_type=2, surrogate=0, recurrent=int(rec), gamma=float(L.gamma), kappa=float(R.kappa),
		dt=float(L.dt), iz_C=float(L.C), iz_vr=float(L.v_rest), iz_vth=float(L.v_th), iz_k=float(L.k), iz_a=float(L.a),
		iz_b=float(L.b), iz_c=float(L.c), iz_d=float(L.d), iz_vpeak=float(L.v_peak))
	W_rec, mask = (npy(L.recurrent_weights), npy(L.rec_mask)) if rec else (None, None)
	f = oracle.forward(cfg, x.numpy(), npy(L.forward_weights), W_rec, mask, npy(R.forward_weights), npy(R.bias_weights))
	net.train()

	def step():
		out, hs = net(x.to(DEV))
		loss = net.batch_loss(x.to(DEV), lab.to(DEV), torch.nn.NLLLoss())
		net.zero_grad()
		loss.backward()
		return out, hs, loss
	(out, hs, loss), names = launched(step)
	assert ran(names, r"k_recur_fwd<64, 1, [^<>]+, 2>") and ran(names, r"k_recur_bwd<")
	V, u, Z = hs["input"]
	assert npy(Z).sum() > 0
	assert np.array_equal(npy(Z), f["Z"]) and np.array_equal(npy(V), f["V"]) and np.array_equal(npy(u), f["a"])
	assert np.array_equal(npy(out), f["y"])
	h = oracle.head(f["y"], lab.numpy())
	assert abs(loss.item() - h["loss"]) <= 1e-5 * max(abs(h["loss"]), 1e-30)
	if O > 1:
		gr = oracle.backward(cfg, x.numpy(), W_rec, mask, npy(R.forward_weights), f["V"], f["a"], f["Z"], h["g_y"])
		assert gr["db"][O - 1] != 0
		assert rel_err(npy(L.forward_weights.grad), gr["dW_in"]) <= 1e-4
		assert rel_err(npy(R.forward_weights.grad), gr["dW_out"]) <= 1e-4 and rel_err(npy(R.bias_weights.grad), gr["db"]) <= 1e-4
		if rec:
			assert rel_err(npy(L.recurrent_weights.grad), gr["dW_rec"]) <= 1e-4
	else:
		assert loss.item() == 0.0 and float(R.forward_weights.grad.abs().max()) == 0.0


# ---- head: fused == stand-alone at the edges of the width ------------------------------------------------------------
FAMILIES = {
	# name: (H, rec, tc, MMA_RECUR, B)
	"simt": (64, True, False, "0", 300),      # more rows than the stand-alone head's 256 threads
	"lean": (128, True, False, "0", 37),
	"tc_recur": (128, True, True, "1", 37),
	"nonrec": (128, False, True, "0", 37),
	"wide_tc": (256, True, True, "0", 11),
	"wide_fp32": (256, True, False, "0", 11),
}


@pytest.mark.parametrize("O", [1, 12, 13, 16])
@pytest.mark.parametrize("family", list(FAMILIES))
def test_fused_head_is_bit_identical_to_the_standalone_head(family, O, monkeypatch):
	H, rec, tc, mma, B = FAMILIES[family]
	monkeypatch.setenv("SNNK_MMA_RECUR", mma)
	case = Case(B, 7, 64, H, O, 1, rec, tc=tc, density=0.3, seed=5000 + 10 * O + H, wscale=1 / 8 if H > 128 else 1.0)
	c = case.c
	for variant in ("plain", "ignored", "bad"):
		lab = case.labels.clone()
		if variant == "ignored":
			lab[::3] = -100
		if variant == "bad":
			lab[B // 2] = O                      # the first invalid class
		for _ in range(2):      # twice: the ticket word must be back at zero after a launch
			f = F_.run_forward(c, case.x, case.W_in, case.W_rec, case.mask, case.beta, case.W_out, case.b_out, labels=lab)
		f0 = F_.run_forward(c, case.x, case.W_in, case.W_rec, case.mask, case.beta, case.W_out, case.b_out)
		loss, logp, gl = F_.run_head_nll(f0["logits"], lab)
		assert torch.equal(f["logits"], f0["logits"]) and torch.equal(f["tstar"], f0["tstar"])
		assert torch.equal(f["logp"], logp)
		assert torch.equal(f["loss"].isnan(), loss.isnan()) and (bool(loss.isnan()) or torch.equal(f["loss"], loss)), variant
		assert torch.equal(f["g_logits"].isnan(), gl.isnan())
		assert torch.equal(torch.nan_to_num(f["g_logits"]), torch.nan_to_num(gl)), variant
		if variant == "bad":
			assert bool(f["loss"].isnan()) and bool(gl[B // 2].isnan().all())
			assert not bool(gl[B // 2 + 1].isnan().any())
		if O == 1 and variant != "bad":
			assert float(loss) == 0.0 and float(logp.abs().max()) == 0.0 and float(gl.abs().max()) == 0.0


# ---- head: snnk_head_nll against float64 torch ---------------------------------------------------------------------
@pytest.mark.parametrize("O", [1, 16])
@pytest.mark.parametrize("B", [1, 300])
def test_head_nll_vs_float64(B, O):
	"""Logits spread over +-1e3: a log-softmax without the max subtraction overflows to inf / NaN."""
	g = torch.Generator().manual_seed(B * 100 + O)
	logits = (torch.rand(B, O, generator=g, dtype=torch.float64) * 2 - 1) * 1e3
	logits = logits.float()
	labels = torch.randint(0, O, (B,), generator=g)
	if B == 1:
		labels[0] = int(logits[0].argmin())      # a loss far from zero
	loss, logp, gl = F_.run_head_nll(logits.to(DEV), labels.to(DEV))
	lg = logits.double().requires_grad_()
	ref_logp = torch.log_softmax(lg, -1)
	ref = torch.nn.functional.nll_loss(ref_logp, labels)
	ref.backward()
	assert torch.isfinite(logp).all() and torch.isfinite(gl).all() and torch.isfinite(loss)
	if O == 1:
		assert float(loss) == 0.0 and float(logp.abs().max()) == 0.0 and float(gl.abs().max()) == 0.0
		return
	assert rel_err(npy(logp), ref_logp.detach().numpy()) <= 1e-6
	assert abs(loss.item() - ref.item()) <= 1e-6 * abs(ref.item())
	assert rel_err(npy(gl), lg.grad.numpy()) <= 1e-6


# ---- bounds at the new widths -----------------------------------------------------------------------------------------
GUARDED = {
	# family: (B, T, H, layer, rec, tc, dedup, MMA_RECUR, backward kernel)
	"lean": (37, 23, 128, 1, True, True, True, "0", r"k_recur_bwd_lean<"),
	"lean_fp32": (37, 23, 128, 0, True, False, False, "0", r"k_recur_bwd_lean<"),
	"tc_recur": (21, 10, 128, 1, True, True, True, "1", r"k_recur_bwd_tc\b"),
	"nonrec": (5, 7, 128, 0, False, True, True, "0", r"k_nonrec_bwd<"),
	"wide_tc": (21, 10, 256, 1, True, True, False, "0", r"k_wide_bwd<"),
}


@pytest.mark.parametrize("O", [1, 13, 15, 16])
@pytest.mark.parametrize("family", list(GUARDED))
def test_guard_bands_at_the_edges_of_the_width(family, O, monkeypatch):
	"""Every y, logits, dW_out and db element written, nothing written outside the buffers (tests/test_gpu_guardbands)."""
	from test_gpu_guardbands import _run
	B, T, H, layer, rec, tc, dedup, mma, kern = GUARDED[family]
	monkeypatch.setenv("SNNK_MMA_RECUR", mma)
	_, names = launched(lambda: _run(B, T, 64, H, O, layer, rec, tc, dedup))
	assert ran(names, kern) == (family != "tc_recur" or O <= 15)


# ---- module level -------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("O", [2, 13, 16])
def test_snn_training_steps_vs_torch_port(O):
	"""SNN(784, O, 128): a few SGD steps through _exec_batch, eagerly and graphed, against the PyTorch restatement of the
	reference -- the fused head and the lean sweep (OP = 16 from 13 classes on) end to end through the optimizer."""
	N, H, T, B, steps = 784, 128, 12, 16, 4

	def make():
		torch.manual_seed(O)
		net = SNN(N, O, H, use_recurrent_connection=True, int_time_steps=T, spike_func=SpikeFuncType.FastSigmoid,
			hidden_layer_type=LayerType.ALIF, device=DEV, learn_beta=False)
		net.train()
		return net, torch.optim.SGD(net.parameters(), lr=0.05)
	(eager, oe), (graphed, og) = make(), make()
	eager.cuda_graphs = False
	L, R = eager.layers["input"], eager.layers["readout"]
	with torch.no_grad():
		for net in (eager, graphed):
			net.layers["readout"].forward_weights.mul_(1.0 + torch.arange(O, device=DEV))
	port = TorchPortSNN(N, H, O, T, layer_type=1, surrogate=0, recurrent=True, seed=0)
	port.load(npy(L.forward_weights), npy(L.recurrent_weights), npy(R.forward_weights), npy(R.bias_weights),
		beta=float(L.beta))
	op = torch.optim.SGD(port.parameters(), lr=0.05)
	g = torch.Generator().manual_seed(O)
	xs = [(torch.rand(B, T, N, generator=g) < 0.1).float() for _ in range(steps)]
	ys = [torch.randint(0, O, (B,), generator=g) for _ in range(steps)]
	crit = torch.nn.NLLLoss()
	for it, (x, y) in enumerate(zip(xs, ys)):
		if it == 0:
			le, names = launched(lambda: eager._exec_batch(x, y, crit, oe))
			assert lean_bwd_variants(names) == {(1, 0, 1, 0, 12 if O <= 12 else 16)}
		else:
			le = eager._exec_batch(x, y, crit, oe)
		lg = graphed._exec_batch(x, y, crit, og)
		lp = port.exec_batch(x, y, op)
		assert abs(le - lp) <= 1e-4 * abs(lp), (it, le, lp)
		assert abs(lg - le) <= 1e-5 * abs(le), (it, lg, le)
	assert len(graphed._graphed_steps) == 1
	for pe, pg in zip(eager.parameters(), graphed.parameters()):
		assert rel_err(npy(pg), npy(pe)) <= 1e-5
	for mine, theirs in ((L.forward_weights, port.W_in), (L.recurrent_weights, port.W_rec), (R.forward_weights, port.W_out),
			(R.bias_weights, port.b_out)):
		assert rel_err(npy(mine), npy(theirs)) <= 1e-4
