"""Initial state, hidden-trace seeds and stacked layers against the C oracle in every kernel family.

Every recurrence family has code for the optional initial state (V0, a0, Z0 of the forward; Z0 again in the backward,
where it stands in for Z_{-1} in dW_rec and in the ALIF adaptation) and for the extra seeds g_V, g_Z on the hidden
traces -- the form in which a stacked network hands gX = gI W_in^T of layer l+1 down to layer l.  Each case here runs
one layer + readout with all of them given, asserts from the profiled kernel names which family ran, and compares with
oracle.forward / oracle.backward (the backward over the GPU's own traces, as in the other suites).  At T = 1, dW_rec is
exactly the Z0 term.  Every family also checks that all-zero state and seed tensors give the same bits as NULL.

The stacked cases compare SNN(N, O, [h1, h2]) with the oracle applied layer by layer, the lower layer selecting each
family in turn; the last section checks snnk_input_grad against float64.
"""
import numpy as np
import pytest
import torch

import oracle
from oracle import OracleCfg
from _util import Guarded, elementwise_err, launched, ran, rel_err
from test_gpu_readout_width import ALPHA, KAPPA, RHO, Case, check_forward_exact, check_forward_forks, scatter_seeds

pytestmark = pytest.mark.gpu

from snnimageclassification_b200 import LayerType, SNN, SpikeFuncType  # noqa: E402
from snnimageclassification_b200.modules import functional as F_  # noqa: E402

DEV = torch.device("cuda:0")


def npy(t):
	return None if t is None else t.detach().cpu().numpy()


def pack(x):
	"""(B,T,N) {0,1} -> the tagged bit-packed raster (SNNK_F_INPUT_BITS)."""
	B, T, N = x.shape
	W = (N + 31) // 32
	xp = np.zeros((B, T, W * 32), dtype=np.uint8)
	xp[..., :N] = npy(x).astype(np.uint8)
	words = np.packbits(xp.reshape(B, T, W, 32), axis=-1, bitorder="little").view(np.uint32).reshape(B, T, W)
	return F_.mark_bits(torch.from_numpy(words.view(np.int32)).to(DEV), N)


# ---- one layer + readout with state and seeds ---------------------------------------------------------------------------
def izh_case(B, T, N, H, O, rec, seed):
	"""A Case whose layer is Izhikevich (dt = 1, input weights large enough to spike; constants of IzhikevichLayer)."""
	case = Case(B, T, N, H, O, 1, rec, seed=seed)
	torch.manual_seed(seed)
	net = SNN(N, O, H, use_recurrent_connection=rec, int_time_steps=T, dt=1.0, hidden_layer_type=LayerType.Izhikevich,
		spike_func=SpikeFuncType.FastSigmoid, device=DEV, tensor_core=False)
	L, R = net.layers["input"], net.layers["readout"]
	case.W_in = (L.forward_weights.detach() * 25.0 + 20.0).contiguous()
	case.W_rec = (L.recurrent_weights.detach() * 5.0).contiguous() if rec else None
	case.beta, case.layer = None, 2
	case.c = L.snnk_consts(kappa=float(R.kappa))
	case.vr = float(L.v_rest)
	case.cfg = OracleCfg(B, T, N, H, O, layer_type=2, surrogate=0, recurrent=int(rec), gamma=float(L.gamma),
		kappa=float(R.kappa), dt=float(L.dt), iz_C=float(L.C), iz_vr=float(L.v_rest), iz_vth=float(L.v_th), iz_k=float(L.k),
		iz_a=float(L.a), iz_b=float(L.b), iz_c=float(L.c), iz_d=float(L.d), iz_vpeak=float(L.v_peak))
	return case


def make_state(case, seed):
	"""V0 spread around the threshold, a0 >= 0, Z0 a raster with ~30 % ones, dense g_V / g_Z."""
	g = torch.Generator().manual_seed(seed)
	B, T, H = case.B, case.T, case.H
	if case.layer == 2:
		V0 = -70.0 + 110.0 * torch.rand(B, H, generator=g)             # v_rest - 10 .. v_peak + 5
		a0 = 20.0 * torch.rand(B, H, generator=g)
	else:
		V0 = case.theta * (0.4 + 1.2 * torch.rand(B, H, generator=g))
		a0 = case.theta / 3 * torch.rand(B, H, generator=g)
	Z0 = (torch.rand(B, H, generator=g) < 0.3).float()
	gV = torch.randn(B, T, H, generator=g) * 0.5
	gZ = torch.randn(B, T, H, generator=g) * 0.5
	return {k: v.to(DEV) for k, v in dict(V0=V0, a0=a0, Z0=Z0, g_V=gV, g_Z=gZ).items()}


def run_step(case, st, dense, seeds=True, V0_null=False):
	"""Forward (with the fused head) and backward of `case` with state `st` (a dict; None entries are NULL)."""
	V0 = None if V0_null else st["V0"]
	state = (V0, st["a0"], st["Z0"]) if case.layer else (V0, st["Z0"])
	f = F_.run_forward(case.c, case.x, case.W_in, case.W_rec, case.mask, case.beta, case.W_out, case.b_out, traces=True,
		state=state, labels=case.labels)
	kw = dict(g_y=case.g_y) if dense else dict(g_logits=case.sparse_seeds(f), tstar=f["tstar"])
	g = F_.run_backward(case.c, case.x, case.W_rec, case.mask, case.beta, case.W_out, f["V"], f["a"], f["zbits"],
		g_V=st["g_V"] if seeds else None, g_Z=st["g_Z"] if seeds else None, Z0=st["Z0"], Z=f["Z"], W_effT=f["W_effT"], **kw)
	return f, g


def x_dense(case):
	x = case.x
	if F_.bits_width(x) is not None:
		return case.x_raster
	return npy(x)


def oracle_pair(case, st, f, dense, seeds=True, V0_null=False):
	x = x_dense(case)
	ref = oracle.forward(case.cfg, x, npy(case.W_in), npy(case.W_rec), npy(case.mask), npy(case.W_out), npy(case.b_out),
		V0=None if V0_null else npy(st["V0"]), a0=npy(st["a0"]) if case.layer else None, Z0=npy(st["Z0"]))
	g_y = npy(case.g_y) if dense else scatter_seeds(case.sparse_seeds(f), f["tstar"], case.T)
	gref = oracle.backward(case.cfg, x, npy(case.W_rec), npy(case.mask), npy(case.W_out), npy(f["V"]), npy(f["a"]),
		npy(f["Z"]), g_y, Z0=npy(st["Z0"]), g_Vs=npy(st["g_V"]) if seeds else None, g_Zs=npy(st["g_Z"]) if seeds else None)
	return ref, gref


def check_weights(case, g, gref, gI_tol, w_tol):
	assert rel_err(npy(g["gI"]()), gref["gI"]) <= gI_tol, rel_err(npy(g["gI"]()), gref["gI"])
	for k in ("dW_in", "dW_out", "db") + (("dW_rec",) if case.rec else ()):
		assert rel_err(npy(g[k]), gref[k]) <= w_tol, (k, rel_err(npy(g[k]), gref[k]))
		assert elementwise_err(npy(g[k]), gref[k]) <= 1e-3, (k, elementwise_err(npy(g[k]), gref[k]))
	if case.rec:
		assert np.abs(gref["dW_rec"]).max() > 0
		assert np.all(np.diag(npy(g["dW_rec"])) == 0.0)


def outputs(f, g):
	out = {k: f[k] for k in ("y", "V", "a", "Z", "zbits", "logits", "tstar", "loss", "g_logits") if f.get(k) is not None}
	out.update({k: g[k] for k in ("dW_in", "dW_rec", "dW_out", "db") if g[k] is not None})
	out["gI"] = g["gI"]().clone()
	return out


def check_zero_is_null(case, st, dense, seeds):
	"""All-zero state / seed tensors give the bits of NULL ones (for Izhikevich, V0 = v_rest is what NULL means)."""
	zero = {k: torch.zeros_like(v) for k, v in st.items()}
	if case.layer == 2:
		zero["V0"] = torch.full_like(st["V0"], case.vr)
	null = dict(V0=None, a0=None, Z0=None, g_V=None, g_Z=None)
	a = outputs(*run_step(case, zero, dense, seeds))
	b = outputs(*run_step(case, null, dense, seeds))
	for k in a:
		assert torch.equal(a[k], b[k]), k


# family: (B, N, H, layer types, rec, tc, env, fwd kernel, bwd kernel, bit-exact forward)
FAMILIES = {
	"simt_h32": (13, 64, 32, (0, 1), True, False, {"SNNK_LEAN": "0"}, r"k_recur_fwd<32, 1\b", r"k_recur_bwd<32, 1\b", True),
	"simt_h64": (13, 64, 64, (0, 1), True, False, {"SNNK_LEAN": "0"}, r"k_recur_fwd<64, 1\b", r"k_recur_bwd<64, 1\b", True),
	"simt_h128": (13, 64, 128, (0, 1), True, False, {"SNNK_LEAN": "0"}, r"k_recur_fwd<128, 1\b", r"k_recur_bwd<128, 1\b",
		True),
	"simt_r2_fp32": (1025, 64, 128, (1,), True, False, {}, r"k_recur_fwd<128, 2\b", r"k_recur_bwd<128, 2\b", True),
	"simt_r2_tc": (1025, 64, 128, (0,), True, True, {}, r"k_recur_fwd<128, 2\b", r"k_recur_bwd<128, 2\b", False),
	"tc_recur": (64, 64, 128, (0, 1), True, True, {"SNNK_MMA_RECUR": "1"}, r"k_recur_fwd_tc\b", r"k_recur_bwd_tc\b", False),
	"tc_recur_b1024": (1024, 64, 128, (1,), True, True, {}, r"k_recur_fwd_tc\b", r"k_recur_bwd_tc\b", False),
	"nonrec_h32": (48, 64, 32, (1,), False, True, {}, r"k_nonrec_fwd<", r"k_nonrec_bwd<", False),
	"nonrec_h128": (48, 64, 128, (1,), False, True, {}, r"k_nonrec_fwd<", r"k_nonrec_bwd<", False),
	"wide_tc_h256": (21, 64, 256, (0, 1), True, True, {}, r"k_wide_fwd<", r"k_wide_bwd<", False),
	"wide_tc_h512": (21, 64, 512, (1,), True, True, {}, r"k_wide_fwd<", r"k_wide_bwd<", False),
	"wide_gen_h256": (11, 64, 256, (0, 1), True, False, {}, r"k_recur_fwd_gen<", r"k_recur_bwd_gen<", True),
	"wide_gen_nonrec_h384": (11, 64, 384, (1,), False, True, {}, r"k_recur_fwd_gen<", r"k_recur_bwd_gen<", False),
	"izh_h128": (9, 48, 128, (2,), True, False, {}, r"k_recur_fwd<128, 1, [^<>]+, 2>", r"k_recur_bwd<", True),
	"izh_h256": (9, 48, 256, (2,), True, False, {}, r"k_recur_fwd_gen<", r"k_recur_bwd_gen<", True),
	# tensor-core GEMMs on a bit-packed raster: k_wgrad_bits (the lean kernels do the recurrence)
	"bits": (40, 64, 128, (1,), True, True, {}, r"k_recur_fwd_lean<", r"k_wgrad_bits<", False),
	# input not tf32-exact: K4 falls back to k_wgrad_simt on the device, whose partials include Z0 already
	"tc_fallback": (40, 60, 128, (1,), True, True, {}, r"k_recur_fwd_lean<", r"k_wgrad_simt<", False),
}


def make_case(family, T, layer, seed):
	B, N, H, _, rec, tc, _, _, _, _ = FAMILIES[family]
	if layer == 2:
		return izh_case(B, T, N, H, 10, rec, seed)
	O = 16 if family == "simt_r2_tc" else 10
	case = Case(B, T, N, H, O, layer, rec, phi=seed % 2, tc=tc, density=0.2, seed=seed, wscale=1 / 8 if H > 128 else 1.0)
	if family == "bits":
		case.x_raster = npy(case.x)
		case.x = pack(case.x)
	if family == "tc_fallback":
		case.x = torch.rand(B, T, N, generator=torch.Generator().manual_seed(seed)).to(DEV) * 0.4    # not {0,1}
	return case


@pytest.mark.parametrize("T", [1, 2])
@pytest.mark.parametrize("family", list(FAMILIES))
def test_state_and_seeds_vs_oracle(family, T, monkeypatch):
	B, N, H, layers, rec, tc, env, kf, kb, exact = FAMILIES[family]
	for k, v in env.items():
		monkeypatch.setenv(k, v)
	if "SNNK_MMA_RECUR" not in env:
		monkeypatch.delenv("SNNK_MMA_RECUR", raising=False)
	for layer in layers:
		seed = 7000 + 100 * T + 10 * layer + H // 32
		case = make_case(family, T, layer, seed)
		st = make_state(case, seed + 1)
		for dense in (True, False):
			(f, g), names = launched(lambda: run_step(case, st, dense))
			assert ran(names, kf) and ran(names, kb), (family, [n for n in names if "snnk::" in n])
			if family == "tc_fallback":
				assert ran(names, r"k_wgrad_tc<")
			ref, gref = oracle_pair(case, st, f, dense)
			if exact:
				check_forward_exact(case, f, ref)
			else:
				check_forward_forks(case, f, ref, max_fork_frac=0.05)
			check_weights(case, g, gref, 1e-5, 1e-5 if exact else 1e-4)
		check_zero_is_null(case, st, dense=False, seeds=True)
		if layer == 2:      # NULL V0 is v_rest
			(f, g) = run_step(case, st, True, V0_null=True)
			ref, gref = oracle_pair(case, st, f, True, V0_null=True)
			for k in ("V", "a", "Z", "y"):          # from v_rest, two steps may not reach a spike
				assert np.array_equal(npy(f[k]), ref[k]), k
			check_weights(case, g, gref, 1e-5, 1e-5)


@pytest.mark.parametrize("T", [1, 2])
@pytest.mark.parametrize("mode", ["tc", "dedup"])
def test_lean_kernels_with_state_vs_oracle(mode, T, monkeypatch):
	"""H = 128 tensor-core, state given: the lean forward reads V0 / a0 / Z0 in its prologue; with sparse seeds and no
	g_V / g_Z the lean sweep runs (Z0 in its spike words), with g_V / g_Z the general SIMT sweep; dedup adds the frame-run
	table (K4: compact x GEMM + Z-only GEMM)."""
	monkeypatch.delenv("SNNK_MMA_RECUR", raising=False)
	monkeypatch.delenv("SNNK_LEAN", raising=False)
	for layer in (0, 1):
		seed = 7500 + 10 * T + layer
		case = Case(96, T, 64, 128, 10, layer, True, phi=layer, tc=True, dedup=mode == "dedup", seed=seed)
		st = make_state(case, seed + 1)
		for seeds in (False, True):
			(f, g), names = launched(lambda: run_step(case, st, False, seeds=seeds))
			assert ran(names, r"k_recur_fwd_lean<")
			assert ran(names, r"k_recur_bwd_lean<") == (not seeds) and ran(names, r"k_recur_bwd<128, 1\b") == seeds
			if mode == "dedup":
				assert F_.get_runs(case.x) is not None and ran(names, r"k_wgrad_tc<")
			ref, gref = oracle_pair(case, st, f, False, seeds=seeds)
			check_forward_forks(case, f, ref, max_fork_frac=0.05)
			check_weights(case, g, gref, 1e-5, 1e-4)
			check_zero_is_null(case, st, dense=False, seeds=seeds)


@pytest.mark.parametrize("T", [1, 2])
@pytest.mark.parametrize("mode", ["fp32", "tc", "dedup"])
def test_fused_training_kernel_with_state_vs_oracle(mode, T, monkeypatch):
	"""k_train_lean (snnk_forward_nll_sweep) with an initial state, then snnk_backward with SNNK_F_SWEEP_DONE and Z0:
	the fused sweep reads Z0 for step 0, the weight-gradient GEMM after it must add the Z0 term of dW_rec."""
	monkeypatch.delenv("SNNK_MMA_RECUR", raising=False)
	monkeypatch.delenv("SNNK_LEAN", raising=False)
	for layer in (0, 1):
		seed = 7600 + 10 * T + layer
		case = Case(96, T, 64, 128, 10, layer, True, phi=1 - layer, tc=mode != "fp32", dedup=mode == "dedup", seed=seed)
		st = make_state(case, seed + 1)
		state = (st["V0"], st["a0"], st["Z0"]) if layer else (st["V0"], st["Z0"])
		scale = torch.ones((1,), device=DEV)

		def step(state=state, Z0=st["Z0"]):
			f = F_.run_forward(case.c, case.x, case.W_in, case.W_rec, case.mask, case.beta, case.W_out, case.b_out,
				traces=False, state=state, labels=case.labels, sweep_scale=scale)
			g = F_.run_backward(case.c, case.x, case.W_rec, case.mask, case.beta, case.W_out, None, None, f["zbits"],
				g_logits=f["g_logits"], tstar=f["tstar"], Z0=Z0, Z=f["Z"], sweep_ws=f["sweep_ws"])
			return f, g
		(f, g), names = launched(step)
		assert ran(names, r"k_train_lean<") and not ran(names, r"k_recur_bwd")
		# the traces of the same forward (lean kernel, same arithmetic) for the oracle's sweep
		ft, _ = run_step(case, st, False)
		for k in ("Z", "zbits", "logits", "tstar", "loss", "g_logits"):
			assert torch.equal(f[k], ft[k]), k
		ref, gref = oracle_pair(case, st, ft, False, seeds=False)
		if mode == "fp32":
			check_forward_exact(case, ft, ref)
		else:
			check_forward_forks(case, ft, ref, max_fork_frac=0.05)
		check_weights(case, g, gref, 1e-5, 1e-5 if mode == "fp32" else 1e-4)
		# zeros == NULL
		z = {k: torch.zeros_like(v) for k, v in st.items()}
		a = step((z["V0"], z["a0"], z["Z0"]) if layer else (z["V0"], z["Z0"]), z["Z0"])
		b = step(None, None)
		oa, ob = outputs(*a), outputs(*b)
		for k in oa:
			if k not in ("V", "a"):
				assert torch.equal(oa[k], ob[k]), k


# ---- stacked layers against the oracle applied layer by layer ---------------------------------------------------------
STACKED = {
	# name: (N, widths, layer type, rec, tensor_core, B, T, backward kernel of the lower layer)
	"tc_recur": (64, [128, 128], LayerType.ALIF, True, True, 1024, 6, r"k_recur_bwd_tc\b"),
	"wide_tc": (64, [256, 128], LayerType.ALIF, True, True, 24, 8, r"k_wide_bwd<"),
	"wide_gen": (64, [256, 64], LayerType.LIF, True, False, 24, 8, r"k_recur_bwd_gen<"),
	"nonrec": (64, [128, 64], LayerType.ALIF, False, True, 48, 10, r"k_nonrec_bwd<"),
	"simt_r2": (64, [128, 128], LayerType.ALIF, True, False, 1025, 4, r"k_recur_bwd<128, 2\b"),
	"izh": (48, [128, 64], LayerType.Izhikevich, True, False, 12, 30, r"k_recur_bwd<128, 1\b"),
	"padded": (100, [100, 200], LayerType.ALIF, True, False, 24, 8, r"k_recur_bwd<128, 1\b"),
}


def layer_cfg(B, T, N, layer, kappa, O):
	if hasattr(layer, "v_peak"):
		return OracleCfg(B, T, N, layer.output_size, O, layer_type=2, surrogate=0, recurrent=int(layer.use_recurrent_connection),
			gamma=float(layer.gamma), kappa=kappa, dt=float(layer.dt), iz_C=float(layer.C), iz_vr=float(layer.v_rest),
			iz_vth=float(layer.v_th), iz_k=float(layer.k), iz_a=float(layer.a), iz_b=float(layer.b), iz_c=float(layer.c),
			iz_d=float(layer.d), iz_vpeak=float(layer.v_peak))
	alif = hasattr(layer, "beta")
	return OracleCfg(B, T, N, layer.output_size, O, layer_type=int(alif), surrogate=0,
		recurrent=int(layer.use_recurrent_connection), alpha=float(layer.alpha), rho=float(getattr(layer, "rho", 0.0)),
		theta=float(layer.threshold), gamma=float(layer.gamma), kappa=kappa, beta=float(layer.beta) if alif else 0.0)


@pytest.mark.parametrize("name", list(STACKED))
def test_stacked_layers_vs_chained_oracle(name, monkeypatch):
	"""SNN(N, O, [h1, h2]): forward of layer 1, its raster into layer 2, head, backward of layer 2, gX = gI_2 W_in2^T in
	float64, backward of layer 1 with g_Z = gX, a zero readout and g_y = 0 (inner layers run with kappa = 0)."""
	monkeypatch.delenv("SNNK_MMA_RECUR", raising=False)
	monkeypatch.delenv("SNNK_LEAN", raising=False)
	N, widths, lt, rec, tc, B, T, kern = STACKED[name]
	O = 10
	torch.manual_seed(len(name))
	kw = dict(learn_beta=False) if lt == LayerType.ALIF else dict(dt=1.0) if lt == LayerType.Izhikevich else {}
	net = SNN(N, O, widths, use_recurrent_connection=rec, int_time_steps=T, spike_func=SpikeFuncType.FastSigmoid,
		hidden_layer_type=lt, device=DEV, tensor_core=tc, **kw)
	L1, L2, R = net.layers["input"], net.layers["hidden_0"], net.layers["readout"]
	with torch.no_grad():
		if lt == LayerType.Izhikevich:
			L1.forward_weights.mul_(25.0).add_(20.0)
			L2.forward_weights.mul_(25.0).add_(60.0)      # fewer input spikes than layer 1 gets
		else:
			L1.forward_weights.mul_(3.0)
			L2.forward_weights.mul_(3.0)
	g = torch.Generator().manual_seed(11)
	x = (torch.rand(B, T, N, generator=g) < 0.2).float()
	labels = torch.randint(0, O, (B,), generator=g)
	net.train()

	def step():
		net.zero_grad()
		loss = net.batch_loss(x, labels)
		loss.backward()
		return loss
	loss, names = launched(step)
	assert ran(names, kern), [n for n in names if "snnk::" in n]
	with torch.no_grad():
		y, hs = net(x.to(DEV))
	# the oracle takes widths that are multiples of 16: [100, 200] runs zero-padded to [112, 208], as the glue pads them
	h1, h2 = widths
	p1, p2 = -h1 % 16, -h2 % 16
	pad = lambda a, *w: None if a is None else np.pad(npy(a), [(0, k) for k in w])  # noqa: E731
	Win1, Win2, Wout = pad(L1.forward_weights, 0, p1), pad(L2.forward_weights, 0, p2), pad(R.forward_weights, p2, 0)
	(Wr1, M1), (Wr2, M2) = ((pad(L.recurrent_weights, p, p), pad(L.rec_mask, p, p)) if rec else (None, None)
		for L, p in ((L1, p1), (L2, p2)))
	tr = lambda t, p: None if t is None else np.pad(t, [(0, 0), (0, 0), (0, p)])  # noqa: E731
	Z1g, Z2g = npy(hs["input"][-1]), npy(hs["hidden_0"][-1])
	st1 = [tr(npy(t), p1) for t in hs["input"]]
	st2 = [tr(npy(t), p2) for t in hs["hidden_0"]]
	zero_out, zero_b = np.zeros((h1 + p1, 1), np.float32), np.zeros(1, np.float32)
	cfg1 = layer_cfg(B, T, N, L1, 0.0, 1)
	cfg2 = layer_cfg(B, T, h1, L2, float(R.kappa), O)
	cfg1.H, cfg2.H = h1 + p1, h2 + p2
	xn = npy(x)
	f1 = oracle.forward(cfg1, xn, Win1, Wr1, M1, zero_out, zero_b)
	f2 = oracle.forward(cfg2, Z1g, Win2, Wr2, M2, Wout, npy(R.bias_weights))
	f1["Z"], f2["Z"] = f1["Z"][..., :h1], f2["Z"][..., :h2]
	# rasters: bit-identical in fp32; tensor-core projections may fork at near-ties
	for Zg, fr, cfg in ((Z1g, f1, cfg1), (Z2g, f2, cfg2)):
		same = ~(Zg != fr["Z"]).any(axis=(1, 2))
		if tc:
			assert same.mean() >= 0.95
		else:
			assert same.all()
	assert 0.001 < Z1g.mean() < 0.999 and 0.001 < Z2g.mean() < 0.999
	h = oracle.head(npy(y), labels.numpy())
	assert abs(loss.item() - h["loss"]) <= 1e-5 * abs(h["loss"])
	# backward, layer by layer, over the GPU's own traces
	V2, a2 = st2[0], (st2[1] if len(st2) == 3 else None)
	b2 = oracle.backward(cfg2, Z1g, Wr2, M2, Wout, V2, a2, st2[-1], h["g_y"])
	gX = (b2["gI"].astype(np.float64) @ Win2.astype(np.float64).T).astype(np.float32)
	V1, a1 = st1[0], (st1[1] if len(st1) == 3 else None)
	b1 = oracle.backward(cfg1, xn, Wr1, M1, zero_out, V1, a1, st1[-1], np.zeros((B, T, 1), np.float32), g_Zs=tr(gX, p1))
	want = {"layers.input.forward_weights": b1["dW_in"][:, :h1], "layers.hidden_0.forward_weights": b2["dW_in"][:, :h2],
		"layers.readout.forward_weights": b2["dW_out"][:h2], "layers.readout.bias_weights": b2["db"]}
	if rec:
		want["layers.input.recurrent_weights"] = b1["dW_rec"][:h1, :h1]
		want["layers.hidden_0.recurrent_weights"] = b2["dW_rec"][:h2, :h2]
	for k, p in net.named_parameters():
		if k not in want:
			assert p.grad is None or float(p.grad.abs().max()) == 0.0, k
			continue
		assert np.abs(want[k]).max() > 0, k
		assert rel_err(npy(p.grad), want[k]) <= 1e-4, (k, rel_err(npy(p.grad), want[k]))
		assert elementwise_err(npy(p.grad), want[k]) <= 1e-3, (k, elementwise_err(npy(p.grad), want[k]))


def test_stacked_training_steps_graphed_and_eager():
	"""Stacked [128, 128] tensor-core net at B = 256: four _exec_batch steps graphed and eager, losses and parameters
	bit-identical; the graphed top layer trains in k_train_lean and its gI feeds snnk_input_grad below."""
	from snnimageclassification_b200 import FusedAdam
	N, T, B, O = 64, 12, 256, 10

	def make(graphs):
		torch.manual_seed(5)
		net = SNN(N, O, [128, 128], use_recurrent_connection=True, int_time_steps=T, spike_func=SpikeFuncType.FastSigmoid,
			hidden_layer_type=LayerType.ALIF, device=DEV, learn_beta=False, tensor_core=True, cuda_graphs=graphs)
		with torch.no_grad():
			net.layers["input"].forward_weights.mul_(3.0)
			net.layers["hidden_0"].forward_weights.mul_(3.0)
		net.train()
		return net, FusedAdam(net.parameters(), lr=1e-3, weight_decay=1e-5)
	(eager, oe), (graphed, og) = make(False), make(True)
	g = torch.Generator().manual_seed(3)
	crit = torch.nn.NLLLoss()
	for it in range(4):
		x = (torch.rand(B, T, N, generator=g) < 0.2).float()
		y = torch.randint(0, O, (B,), generator=g)
		if it == 2:
			le, names = launched(lambda: eager._exec_batch(x, y, crit, oe))
			assert ran(names, r"k_input_grad") and ran(names, r"k_recur_bwd_lean<")
			lg, names = launched(lambda: graphed._exec_batch(x, y, crit, og))
			assert ran(names, r"k_input_grad") and ran(names, r"k_train_lean<"), [n for n in names if "snnk::" in n]
		else:
			le = eager._exec_batch(x, y, crit, oe)
			lg = graphed._exec_batch(x, y, crit, og)
		assert lg == le, (it, lg, le)
		for (k, pe), pg in zip(eager.named_parameters(), graphed.parameters()):
			assert torch.equal(pe, pg), (it, k)


# ---- snnk_input_grad against float64 ------------------------------------------------------------------------------------
@pytest.mark.parametrize("K", [32, 64, 128, 256, 2048])
@pytest.mark.parametrize("Nn", [1, 20, 100, 127, 128, 784])
def test_input_grad_vs_float64(K, Nn):
	"""gX = gI W_in^T over B*T = 1025*3 rows (several 128-row tiles and a partial one), with gI spread over magnitudes;
	gX sits between guard bands."""
	from snnimageclassification_b200 import _cabi
	import ctypes
	B, T = 1025, 3
	g = torch.Generator().manual_seed(K * 1000 + Nn)
	gI = torch.randn(B, T, K, generator=g) * torch.exp(torch.randn(B, T, 1, generator=g) * 4.0)
	W = torch.randn(Nn, K, generator=g)
	c = F_.LayerConsts(1, 0, True, ALPHA, RHO, 0.03, 0.3, KAPPA)
	desc = F_.make_desc(c, B, T, Nn, K, 1, True)
	out = Guarded((B, T, Nn))
	gId, Wd = gI.to(DEV), W.to(DEV)
	# the library's own launch count: torch.profiler loses the activity of such one-kernel windows late in a long
	# session (an empty kernel list), which says nothing about the kernel
	with _cabi.kernel_profile() as prof:
		_cabi.check(_cabi.lib().snnk_input_grad(ctypes.byref(desc), _cabi.ptr(gId), _cabi.ptr(Wd), _cabi.ptr(out.t),
			_cabi.stream_ptr()), "snnk_input_grad")
		torch.cuda.synchronize()
	assert [(k.split()[0], n) for k, (_, n) in prof.result.items()] == [("k_input_grad", 1)], prof.result
	out.check("gX")
	ref = (gI.double().reshape(-1, K) @ W.double().T).reshape(B, T, Nn).numpy()
	got = npy(out.t)
	assert rel_err(got, ref) <= 1e-5
	assert elementwise_err(got, ref) <= 1e-3
	assert torch.equal(out.t, F_.run_input_grad(c, gId, Wd))
