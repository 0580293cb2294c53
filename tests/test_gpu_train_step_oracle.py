"""The fused training kernel (recur_lean.cuh, k_train_lean) against the C oracle, at the bench batch and at the edges of
its selection.

Every captured training step of the headline geometry (recurrent LIF / ALIF, H = 128, O <= 12, one row per CTA,
built-in surrogate) runs the forward recurrence, the head and the BPTT sweep of a row in one CTA, and so does the step
bench.py times.  test_gpu_fused_sweep.py compares that kernel with the project's own lean kernels at B <= 37; here it
is compared with an independent reference (oracle/snn_oracle.c: the same operation order, built with
-ffp-contract=off), output by output, where it runs:

  * at B = 256 (two CTAs per SM: where the cross-proxy hand-overs of a shared staging area could race), at exactly two
    CTAs on every SM, in a second wave and over several waves up to the largest batch the kernel takes;
  * at the longest sequence it takes (T = 122) and at T = 1, 2; for a single row; for a run table in which samples of
    two runs (the second one step long) sit next to samples with a run at nearly every step;
  * with labels the head treats specially (ignore_index, out of range);
  * in the captured end-to-end step over a stream of different batches (the two alternating step graphs).

Bars: the twin (forward with traces + the regular sweep, same inputs) bit for bit; in fp32 mode the forward bit for bit
against the oracle, in tensor-core mode (I_in rounds differently) the fork-aware bar of test_gpu_configs.py; the head
within 1e-5; gI bit for bit against the oracle's sweep over the twin's traces in BOTH modes (the sweep restates the
oracle's arithmetic and the tf32 planes are an exact hi / lo split); weight gradients against the oracle's double
accumulation within 1e-5.
"""
import dataclasses
import os
from concurrent.futures import ThreadPoolExecutor

import numpy as np
import pytest
import torch

import oracle
from oracle import OracleCfg
from _util import elementwise_err, rel_err, unexplained_forks

pytestmark = pytest.mark.gpu

from snnimageclassification_b200 import SNN, FusedAdam, LayerType, SpikeFuncType, ToSpikes  # noqa: E402
from snnimageclassification_b200.modules import functional as F_  # noqa: E402

from test_gpu_fused_sweep import _kernels, _ran  # noqa: E402

DEV = torch.device("cuda:0")
N, H = 784, 128
FUSED, SWEEP = r"k_train_lean<", r"k_recur_bwd_lean<"
# lean_fwd_smem_bytes<128>(T, O) = 39 952 + 592 T bytes (any O <= 16) against the 110 KB (112 640 B) cap of make_plan:
# T = 122 -> 112 176 B is the longest sequence the fused kernel takes, T = 123 -> 112 768 B is not
T_MAX = 122


def npy(t):
	return None if t is None else t.detach().cpu().numpy()


def _net(layer, spike, O, T, tc, **kw):
	torch.manual_seed(0)
	alif = layer == "ALIF"
	return SNN(N, O, H, use_recurrent_connection=True, int_time_steps=T, device=DEV, tensor_core=tc,
		spike_func=SpikeFuncType.FastSigmoid if spike == "fs" else SpikeFuncType.Phi,
		hidden_layer_type=LayerType.ALIF if alif else LayerType.LIF, **({"learn_beta": True} if alif else {}), **kw)


def _images(B, ink, g):
	"""MNIST-shaped (ink 0.19) / Fashion-MNIST-shaped (ink 0.5) synthetic images: k/255 levels."""
	return (torch.randint(1, 256, (B, N), generator=g).float() / 255.0) * (torch.rand(B, N, generator=g) < ink)


def _runs_per_sample(x):
	"""Number of runs of equal consecutive frames of every sample of a (B, T, N) raster (test_gpu_runs.py restates the
	whole table the same way)."""
	changed = (x[:, 1:] != x[:, :-1]).any(axis=2)
	return 1 + changed.sum(axis=1)


def _input(kind, B, T, g):
	"""(raster on the device, host images or None)."""
	if kind == "dense":      # a binary raster without a run table: the dense kernels
		return F_.mark_binary((torch.rand(B, T, N, generator=g) < 0.2).float().to(DEV)), None
	if kind == "runs":       # the bench encoder (tau 0.02, periodic) with its run table: the frame-dedup kernels
		img = _images(B, 0.19, g)
		x = ToSpikes(T, use_periods=True).encode_batch(img.to(DEV))
	else:
		# "extremes": blank images next to four dense ones.  A blank image's pixels all fire at the last step only, so
		# its row is one run of T - 1 silent frames and a run of length 1 that closes the row.  A dense image's shortest
		# period is ~4.5 steps at tau = 20: its first four frames are silent, and from then on every frame differs
		# (runs of length 1 throughout)
		assert kind == "extremes"
		img = torch.zeros(B, N)
		dense = torch.arange(3, B, B // 4)[:4]
		img[dense] = torch.rand(len(dense), N, generator=g)
		x = ToSpikes(T, tau=20.0, use_periods=True).encode_batch(img.to(DEV))
		n_runs = _runs_per_sample(npy(x))
		blank = np.ones(B, bool)
		blank[dense.numpy()] = False
		assert (n_runs[blank] <= 2).all() and (n_runs[dense.numpy()] >= T - 3).all(), n_runs[dense.numpy()]
	runs = F_.get_runs(x)
	assert runs is not None and int(runs[1]) == 1, "the run table must describe every run (the frame-dedup path)"
	return x, img


def _step(c, x, labels, ws, scale, fused):
	"""One training step's kernels, as numpy: the fused entry (run_forward(sweep_scale) + the rest of the backward), or
	its twin (forward with traces + the regular sweep).  None where the fused entry does not take the geometry."""
	W_in, W_rec, M, beta, W_out, b_out = ws
	if fused:
		f = F_.run_forward(c, x, *ws, traces=False, labels=labels, sweep_scale=scale)
		if f is None:
			return None
		g = F_.run_backward(c, x, W_rec, M, beta, W_out, None, None, f["zbits"], g_logits=f["g_logits"], tstar=f["tstar"],
			Z=f["Z"], g_scale=scale, sweep_ws=f["sweep_ws"])
	else:
		f = F_.run_forward(c, x, *ws, traces=True, labels=labels)
		g = F_.run_backward(c, x, W_rec, M, beta, W_out, f["V"], f["a"], f["zbits"], g_logits=f["g_logits"],
			tstar=f["tstar"], Z=f["Z"], g_scale=scale, W_effT=f["W_effT"])
	out = {k: npy(f[k]) for k in ("Z", "zbits", "y", "logits", "tstar", "loss", "logp", "g_logits", "V", "a")}
	out.update({k: npy(g[k]) for k in ("dW_in", "dW_rec", "dW_out", "db")}, gI=npy(g["gI"]()))
	return out


def _setup(layer, spike, tc, kind, B, T, O, seed=None):
	net = _net(layer, spike, O, T, tc)
	c = net._consts()
	ws = tuple(F_._c(w) for w in net._weights())
	g = torch.Generator().manual_seed(B * 1000 + T if seed is None else seed)
	x, img = _input(kind, B, T, g)
	labels = torch.randint(0, O, (B,), generator=g)
	return c, ws, x, img, labels


def _oracle_cfg(c, ws, B, T, O):
	beta = ws[3]
	return OracleCfg(B, T, N, H, O, layer_type=c.layer_type, surrogate=c.surrogate, recurrent=1, alpha=c.alpha,
		rho=c.rho, theta=c.theta, gamma=c.gamma, kappa=c.kappa, beta=float(beta) if beta is not None else 0.0)


def _oracle_forward(cfg, x, w):
	"""oracle.forward over row chunks in threads (rows are independent; the C call releases the GIL)."""
	chunks = [ix for ix in np.array_split(np.arange(cfg.B), min(cfg.B, os.cpu_count() or 1)) if len(ix)]

	def one(ix):
		return oracle.forward(dataclasses.replace(cfg, B=len(ix)), x[ix], w["W_in"], w["W_rec"], w["mask"], w["W_out"], w["b"])
	with ThreadPoolExecutor(len(chunks)) as ex:
		parts = list(ex.map(one, chunks))
	return {k: np.concatenate([p[k] for p in parts]) for k in parts[0]}


def _where(a, b):
	"""First differing (b, t, i) of two (B, T, H) arrays, how many rows differ and the two values there."""
	d = a != b
	rows = np.nonzero(d.any(axis=(1, 2)))[0]
	idx = tuple(int(v) for v in np.argwhere(d)[0])
	return f"first difference at (b, t, i) = {idx}: {a[idx]!r} vs {b[idx]!r}; {len(rows)} rows differ: {rows[:12].tolist()}"


def _rows(B):
	"""Rows the oracle's forward check evaluates: all of them, or for B >= 512 a spread subset holding the first rows,
	the last rows (the last wave of CTAs) and rows in between (rows are independent)."""
	if B < 512:
		return np.arange(B)
	return np.unique(np.concatenate([np.arange(4), np.linspace(0, B - 1, 24).astype(int), np.arange(B - 8, B)]))


# layer, surrogate, tensor cores, input, B, T, O, seed scale: each line names the edge it covers
CASES = {
	"bench_step_b256": ("ALIF", "fs", True, "runs", 256, 100, 10, 1.0),               # the bench step: two CTAs per SM
	"two_ctas_per_sm_b296_fp32": ("ALIF", "fs", False, "dense", 296, 100, 10, 1.0),  # exactly two CTAs on every SM
	"second_wave_b297_fp32": ("LIF", "phi", False, "dense", 297, 37, 12, 0.75),      # one CTA in a second wave
	"largest_tc_batch_b1023": ("ALIF", "phi", True, "runs", 1023, 23, 10, 1.0),     # B = 1024 takes the MMA recurrence
	# B = 1025 takes two rows per CTA.  (Two classes: with one, log_softmax is 0 and the loss has no gradient.)
	"largest_fp32_batch_b1024": ("LIF", "fs", False, "dense", 1024, 9, 2, 0.75),
	"longest_sequence_t122": ("ALIF", "fs", True, "dense", 256, T_MAX, 12, 1.0),    # largest shared memory
	"single_row_b1": ("ALIF", "fs", True, "runs", 1, 100, 10, 0.75),                # ticket and loss from one row
	"one_step_t1_fp32": ("ALIF", "fs", False, "dense", 5, 1, 10, 1.0),
	"two_steps_t2": ("LIF", "phi", True, "dense", 3, 2, 7, 0.75),
	"run_table_extremes_b64": ("ALIF", "fs", True, "extremes", 64, 100, 10, 1.0),   # 2-run and ~T-run samples
}


@pytest.mark.parametrize("case", list(CASES))
def test_fused_step_vs_oracle(case):
	layer, spike, tc, kind, B, T, O, s = CASES[case]
	c, ws, x, _, labels = _setup(layer, spike, tc, kind, B, T, O)
	alif = layer == "ALIF"
	scale = torch.full((1,), s, device=DEV)
	box = {}
	names = _kernels(lambda: box.update(fu=_step(c, x, labels.to(DEV), ws, scale, fused=True)))
	assert _ran(names, FUSED) and not _ran(names, SWEEP), names
	fu = box["fu"]

	# 1. the twin on the same inputs: bit for bit
	tw = _step(c, x, labels.to(DEV), ws, scale, fused=False)
	for k in ("Z", "zbits", "y", "logits", "tstar", "loss", "logp", "g_logits", "gI", "dW_in", "dW_rec", "dW_out", "db"):
		assert np.array_equal(fu[k], tw[k]), f"{k}: the fused kernel differs from forward + regular sweep"

	# 2. forward vs the oracle
	xh = npy(x)
	cfg = _oracle_cfg(c, ws, B, T, O)
	w = dict(zip(("W_in", "W_rec", "mask", "beta", "W_out", "b"), (npy(t) for t in ws)))
	sel = _rows(B)
	f = _oracle_forward(dataclasses.replace(cfg, B=len(sel)), xh[sel], w)
	Z = fu["Z"][sel]
	assert 0.001 < f["Z"].mean() < 0.9, f"spike rate {f['Z'].mean():.4f}: the raster checks would say little"
	if not tc:      # fp32 GEMMs: the whole forward is the oracle's arithmetic
		assert np.array_equal(Z, f["Z"]), _where(Z, f["Z"])
		assert np.array_equal(fu["y"][sel], f["y"]), "y differs from the oracle"
		assert np.array_equal(tw["V"][sel], f["V"]), _where(tw["V"][sel], f["V"])
		if alif:
			assert np.array_equal(tw["a"][sel], f["a"]), _where(tw["a"][sel], f["a"])
		h = oracle.head(f["y"], None)
		assert np.array_equal(fu["logits"][sel], h["logits"]) and np.array_equal(fu["tstar"][sel], h["tstar"])
	else:           # tensor-core projection: I_in rounds differently, so a spike ON the threshold may flip
		thr = cfg.theta + (np.float32(cfg.beta) * f["a"] if alif else 0.0)
		forked, unexplained = unexplained_forks(Z, f["Z"], f["V"], thr)
		assert unexplained == 0, f"{unexplained} of {forked} forked samples differ first at a spike that is no near-tie"
		assert forked <= max(1, int(0.05 * len(sel))), f"{forked} of {len(sel)} samples forked"
		ok = ~(Z != f["Z"]).any(axis=(1, 2))
		assert rel_err(fu["y"][sel][ok], f["y"][ok]) <= 1e-5
		assert rel_err(tw["V"][sel][ok], f["V"][ok]) <= 1e-5

	# 3. head vs the oracle on the GPU's own y
	h = oracle.head(fu["y"], labels.numpy())
	assert np.array_equal(fu["logits"], h["logits"]) and np.array_equal(fu["tstar"], h["tstar"])
	assert abs(float(fu["loss"]) - h["loss"]) <= 1e-5 * abs(h["loss"]), (float(fu["loss"]), h["loss"])
	assert rel_err(fu["logp"], h["logp"]) <= 1e-5
	bi, oi = np.arange(B)[:, None], np.arange(O)[None, :]
	assert rel_err(fu["g_logits"], h["g_y"][bi, h["tstar"], oi]) <= 1e-5

	# 4. gI vs the oracle's sweep over the twin's traces, seeded as the kernel seeds: __fmul_rn(g_logits, scale)
	g_y = np.zeros((B, T, O), np.float32)
	g_y[bi, fu["tstar"], oi] = fu["g_logits"] * np.float32(s)
	gr = oracle.backward(cfg, xh, w["W_rec"], w["mask"], w["W_out"], tw["V"], tw["a"] if alif else np.zeros_like(tw["V"]),
		tw["Z"], g_y)
	assert np.abs(gr["gI"]).max() > 0
	assert np.array_equal(fu["gI"], gr["gI"]), "gI: " + _where(fu["gI"], gr["gI"])

	# 5. weight gradients vs the oracle's double accumulation
	assert np.all(np.diag(fu["dW_rec"]) == 0.0)
	for k in ("dW_in", "dW_rec", "dW_out", "db"):
		assert rel_err(fu[k], gr[k]) <= 1e-5, (k, rel_err(fu[k], gr[k]))
		assert elementwise_err(fu[k], gr[k], 1e-3) <= 1e-3, (k, elementwise_err(fu[k], gr[k], 1e-3))


# ---- selection at the limits -----------------------------------------------------------------------------------------
@pytest.mark.parametrize("T,fused", [(T_MAX, True), (T_MAX + 1, False)])
def test_longest_sequence_selection_and_captured_step(T, fused):
	"""The fused entry takes T = 122 and refuses T = 123 (SNNK_ERR_UNSUPPORTED); on both sides the captured step runs the
	kernel the selection names and takes the same three steps as the eager path, bit for bit."""
	B, O = 64, 10
	c, ws, x, _, labels = _setup("ALIF", "fs", True, "runs", B, T, O)
	y = labels.to(DEV)
	scale = torch.ones(1, device=DEV)
	if fused:
		box = {}
		names = _kernels(lambda: box.update(out=F_.run_forward(c, x, *ws, traces=False, labels=y, sweep_scale=scale)))
		assert box["out"] is not None and _ran(names, FUSED), names
	else:
		assert F_.run_forward(c, x, *ws, traces=False, labels=y, sweep_scale=scale) is None
	crit = torch.nn.NLLLoss()
	ref, net = _net("ALIF", "fs", O, T, True), _net("ALIF", "fs", O, T, True)
	opt_ref = FusedAdam(ref.parameters(), lr=1e-3, weight_decay=1e-5)
	opt = FusedAdam(net.parameters(), lr=1e-3, weight_decay=1e-5)
	ref.train(); net.train()
	step = net.graphed_train_step(x, y, crit, opt, static_inputs=True)
	names = _kernels(step)
	assert _ran(names, FUSED) == fused and _ran(names, SWEEP) != fused, names
	for k in range(3):
		if k > 0:
			step()
		loss_ref = ref.batch_loss(x, y, crit)
		opt_ref.zero_grad()
		loss_ref.backward()
		opt_ref.step()
		assert float(step.loss) == float(loss_ref), (k, float(step.loss), float(loss_ref))
		for (name, p), q in zip(ref.named_parameters(), net.parameters()):
			assert torch.equal(p, q), f"step {k}: {name} differs"


@pytest.mark.parametrize("B,tc,fused", [(1023, True, True), (1024, True, False), (1024, False, True), (1025, False, False)])
def test_batch_limits_selection(B, tc, fused):
	"""The largest batches the fused kernel takes: 1023 with tensor cores (B >= 1024 takes the MMA recurrence) and 1024
	in fp32 mode (B = 1025 takes two rows per CTA).  Beyond them the fused entry returns None before launching."""
	T, O = 9, 10
	c, ws, x, _, labels = _setup("ALIF", "fs", tc, "dense", B, T, O)
	args = (c, x, *ws)
	kw = dict(traces=False, labels=labels.to(DEV), sweep_scale=torch.ones(1, device=DEV))
	if fused:
		box = {}
		names = _kernels(lambda: box.update(out=F_.run_forward(*args, **kw)))
		assert box["out"] is not None and _ran(names, FUSED), names
	else:
		assert F_.run_forward(*args, **kw) is None


# ---- labels the head treats specially --------------------------------------------------------------------------------
def _same(a, b, name):
	a, b = np.asarray(a), np.asarray(b)
	assert np.array_equal(np.isnan(a), np.isnan(b)), f"{name}: NaN patterns differ"
	assert np.array_equal(np.nan_to_num(a), np.nan_to_num(b)), f"{name} differs"


@pytest.mark.parametrize("variant", ["every_third_ignored", "one_out_of_range", "all_ignored"])
def test_fused_step_with_special_labels(variant):
	"""ignore_index rows (excluded from the mean, zero gradient) and an out-of-range label (NaN loss and row gradient,
	as documented in include/snnk.h) on the fused path: everything bit for bit as forward_nll + the regular backward;
	twice, so that a ticket word left non-zero by the first launch would show in the second."""
	B, T, O = 256, 40, 10
	c, ws, x, img, labels = _setup("ALIF", "fs", True, "runs", B, T, O)
	if variant == "every_third_ignored":
		labels[::3] = -100
	elif variant == "one_out_of_range":
		labels[77] = O + 3
	else:
		labels[:] = -100
	y = labels.to(DEV)
	scale = torch.ones(1, device=DEV)
	ref = _step(c, x, y, ws, scale, fused=False)
	keys = ("loss", "logp", "g_logits", "gI", "dW_in", "dW_rec", "dW_out", "db")
	for rep in range(2):
		box = {}
		names = _kernels(lambda: box.update(fu=_step(c, x, y, ws, scale, fused=True)))
		assert _ran(names, FUSED), names
		assert int(F_._head_scratch(DEV, B)[B]) == 0, "the head's ticket word was left non-zero"
		for k in keys:
			_same(box["fu"][k], ref[k], f"call {rep}: {k}")
	fu = box["fu"]
	ign = (labels == -100).numpy()
	assert (fu["g_logits"][ign] == 0).all(), "ignored rows have a non-zero dL/dlogits"
	if variant == "all_ignored":
		for k in ("gI", "dW_in", "dW_rec", "dW_out", "db"):
			assert not np.any(fu[k]), f"{k}: rows without a valid label contributed"
	elif variant == "every_third_ignored":
		# the valid rows alone: same number of valid rows, so the same seeds, and the same gradients -- the ignored rows
		# contributed nothing (up to the order of the batch reductions)
		keep = torch.from_numpy(~ign)
		xv = ToSpikes(T, use_periods=True).encode_batch(img[keep].to(DEV))
		sub = _step(c, xv, y[keep.to(DEV)], ws, scale, fused=True)
		assert np.array_equal(sub["logp"], fu["logp"][~ign]) and np.array_equal(sub["g_logits"], fu["g_logits"][~ign])
		assert abs(float(sub["loss"]) - float(fu["loss"])) <= 1e-6 * abs(float(fu["loss"]))
		for k in ("dW_in", "dW_rec", "dW_out", "db"):
			assert rel_err(fu[k], sub[k]) <= 1e-5, (k, rel_err(fu[k], sub[k]))
	else:
		assert np.isnan(fu["loss"]).all() and np.isnan(fu["g_logits"][77]).all()
		assert not np.isnan(np.delete(fu["g_logits"], 77, axis=0)).any()


# ---- the captured end-to-end step over a stream of different batches ----------------------------------------------------
def test_captured_step_over_a_stream_of_batches():
	"""The bench / end-to-end configuration fed pinned host images: six calls rotating through three different batches
	(MNIST-like ink, Fashion-like ink, half blank images: three different run tables; one batch with ignored rows).
	The captured path (two alternating step graphs, each with its own encoder buffers and run table) takes the same
	steps as the eager path: loss and every parameter bit for bit after every call."""
	B, T, O = 256, 100, 10
	g = torch.Generator().manual_seed(23)
	img0, img1, img2 = _images(B, 0.19, g), _images(B, 0.5, g), _images(B, 0.19, g)
	img2[::2] = 0.0
	labs = [torch.randint(0, O, (B,), generator=g) for _ in range(3)]
	labs[1][::7] = -100
	n_runs = [int(F_.get_runs(ToSpikes(T, use_periods=True).encode_batch(im.to(DEV)))[0]) for im in (img0, img1, img2)]
	assert n_runs[2] < n_runs[0], n_runs
	batches = [(im.pin_memory(), lab) for im, lab in zip((img0, img1, img2), labs)]
	crit = torch.nn.NLLLoss()
	nets, opts = [], []
	for graphs in (False, True):
		net = _net("ALIF", "fs", O, T, True, input_encoder=ToSpikes(T, use_periods=True), cuda_graphs=graphs)
		net.train()
		nets.append(net)
		opts.append(FusedAdam(net.parameters(), lr=1e-3, weight_decay=1e-5))
	(eager, graphed), (opt_e, opt_g) = nets, opts
	for k in range(6):
		xb, lab = batches[k % 3]
		loss_e = eager._exec_batch(xb, lab, crit, opt_e)
		if k == 3:
			box = []
			names = _kernels(lambda: box.append(graphed._exec_batch(xb, lab, crit, opt_g)))
			assert graphed._last_graphed_step is not None, "call 4 did not replay a captured step"
			assert _ran(names, FUSED) and not _ran(names, SWEEP), names
			loss_g = box[0]
		else:
			loss_g = graphed._exec_batch(xb, lab, crit, opt_g)
		assert loss_g == loss_e, (k, loss_g, loss_e)
		for (name, p), q in zip(eager.named_parameters(), graphed.parameters()):
			assert torch.equal(p, q), f"call {k}: {name} differs"
